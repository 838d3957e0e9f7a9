"""GPU (>= 2 devices): the C-ABI collective dfm_allgather_results with a REAL ncclComm_t created through ctypes
(ncclGetUniqueId / ncclCommInitRank from the NCCL library torch bundles) -- what INTEGRATION.md tells a Julia
maintainer to call (NCCL.jl hands over the same handle).  Two processes, one per GPU; rank r contributes the records
of its dfm_shard_range shard and every rank must end up with all records in replication order."""
import ctypes as C
import glob
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_nccl():
    import torch
    cands = glob.glob(os.path.join(os.path.dirname(os.path.dirname(torch.__file__)), "nvidia", "nccl", "lib", "libnccl.so*"))
    cands += ["libnccl.so.2", "libnccl.so"]
    for c in cands:
        try:
            return C.CDLL(c, mode=C.RTLD_GLOBAL)
        except OSError:
            continue
    return None


class _UniqueId(C.Structure):
    _fields_ = [("internal", C.c_byte * 128)]


def _worker(rank, world, tmp, n_rep, d):
    sys.path.insert(0, ROOT)
    import torch
    from dynamic_factor_models_b200 import Library
    torch.cuda.set_device(rank)
    nccl = _find_nccl()
    uid = _UniqueId()
    path = os.path.join(tmp, "uid.bin")
    if rank == 0:
        assert nccl.ncclGetUniqueId(C.byref(uid)) == 0
        with open(path + ".tmp", "wb") as f:
            f.write(bytes(uid.internal))
        os.rename(path + ".tmp", path)
    else:
        import time
        for _ in range(600):
            if os.path.exists(path):
                break
            time.sleep(0.05)
        raw = open(path, "rb").read()
        C.memmove(C.byref(uid), raw, 128)
    comm = C.c_void_p()
    nccl.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, _UniqueId, C.c_int]
    assert nccl.ncclCommInitRank(C.byref(comm), world, uid, rank) == 0
    lib = Library(device=rank)
    b, e = lib.shard_range(n_rep, rank, world)
    assert e - b == n_rep // world
    local = torch.arange(b * d, e * d, dtype=torch.float64, device=f"cuda:{rank}") * 0.5 + 1.0     # record i = known function of id
    recv = torch.full((n_rep * d,), float("nan"), dtype=torch.float64, device=f"cuda:{rank}")
    lib.lib.dfm_allgather_results.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong]
    lib.check(lib.lib.dfm_allgather_results(lib.h, comm, C.c_void_p(local.data_ptr()), C.c_void_p(recv.data_ptr()), (e - b) * d),
              "dfm_allgather_results")
    lib.sync()
    np.save(os.path.join(tmp, f"recv{rank}.npy"), recv.cpu().numpy())
    nccl.ncclCommDestroy.argtypes = [C.c_void_p]
    nccl.ncclCommDestroy(comm)
    lib.close()


def test_allgather_results_with_real_nccl_comm(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    if _find_nccl() is None:
        pytest.skip("libnccl not found")
    import torch.multiprocessing as mp
    world, n_rep, d = 2, 10, 7
    mp.spawn(_worker, args=(world, str(tmp_path), n_rep, d), nprocs=world, join=True)
    want = np.arange(n_rep * d, dtype=float) * 0.5 + 1.0
    for rank in range(world):
        got = np.load(tmp_path / f"recv{rank}.npy")
        np.testing.assert_array_equal(got, want)
