#!/usr/bin/env python
"""bench.py -- EM iterations/sec of the B200 DFM hot path (BASELINE.json metric).

Unit of work: one EM iteration (Kalman filter + RTS smoother E-step, M-step) on one C2-shaped panel
(N=200, r=8, T=500, FP64).  A "step" = EM_ITERS iterations over this rank's shard of independent
Monte-Carlo panels (BASELINE config C5 sharded: 10 000 / 8 = 1250 panels per GPU, weak scaling),
followed by the path's single collective: one NCCL all-gather of the per-replication statistics.

  value  : panel-EM-iterations / s, inputs resident in HBM, device-timed (CUDA events), max over ranks
  e2e    : same through the C ABI with pinned HOST buffers (H2D of panel + initial parameters and
           D2H of factors + parameters inside the timed region)
  roofline: dominant kernel's algorithmic bytes (2*T*N*8 per panel-iteration, SURVEY.md 8d) / its
           CUDA-event duration, against MEASURED_PEAKS.json
  cpu_baseline / --impl reference: the oracle's C port of the same EM (OpenMP over panels) on the
           host cores -- the reference itself is Julia and has no Kalman/EM code (SURVEY.md 0).

python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the timed path computed in its last step (rank 0) as DIR/<name>.npy, float64, so that
two builds can be compared output for output: the inputs are the same from run to run for the same arguments.
bench_outputs/ in the repository is ignored by git for this use.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NS, R_, T_, P_ = 200, 8, 500, 1
METRIC = "EM iters/sec (N=200,r=8,T=500)"
UNIT = "panel-EM-iterations/s"


SEED = 20260922            # dynamic_factor_models_b200.replicate.SEED == oracle.dgp.SEED (frozen, SURVEY.md 8d)


def make_panels_host(B, rep0):
    """CPU arm only: the numpy restatement (oracle/dgp.py) of the DEVICE generator's Philox stream -- the same
    replication ids give the same panels (to libm rounding) as dfm_simulate_panels.  (B, T, N) float64."""
    from oracle.dgp import simulate_panel_device_stream
    return np.stack([simulate_panel_device_stream(NS, R_, T_, rep=rep0 + b, seed=SEED)[0] for b in range(B)])


class ClockSampler:
    def __init__(self, dev):
        self.dev, self.rows, self.proc = dev, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True); self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) >= 7 and r[3 + j].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def host_cores():
    """Host CPU allowance of THIS process: logical CPUs, scheduler affinity, cgroup CPU quota, physical cores.
    `threads` = what the CPU arm uses: one OpenMP thread per physical core inside the affinity mask, capped by the
    cgroup quota (os.cpu_count() ignores both, which oversubscribed the 1-GPU lease in round 1)."""
    info = {"logical": os.cpu_count()}
    try:
        aff = sorted(os.sched_getaffinity(0))
    except AttributeError:
        aff = list(range(os.cpu_count() or 1))
    info["affinity"] = len(aff)
    quota = None
    try:                                                   # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except (OSError, ValueError):
        try:                                               # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    info["cgroup_quota"] = quota
    phys = set()
    for c in aff:
        try:
            base = f"/sys/devices/system/cpu/cpu{c}/topology/"
            phys.add((open(base + "physical_package_id").read().strip(), open(base + "core_id").read().strip()))
        except OSError:
            phys.add(("?", str(c)))
    info["physical"] = len(phys)
    n = min(len(aff), len(phys))
    if quota:
        n = max(1, min(n, int(quota)))
    info["threads"] = n
    return info


def _omp_env():
    """Bind the OpenMP threads of the oracle C port (read by libgomp when the library is loaded)."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_WAIT_POLICY", "active")


def cpu_em(Xs, init, iters, nthreads=0):
    """Oracle C port on host cores: (seconds, panel-iterations)."""
    _omp_env()
    from oracle.c import kem
    t0 = time.perf_counter()
    out = kem.em_kalman_batch(Xs, init[0], init[1], init[2], init[3], p=P_, max_iter=iters, tol=0.0, nthreads=nthreads, want_F=True)
    dt = time.perf_counter() - t0
    assert (out["status"] == 0).all()
    return dt, Xs.shape[0] * iters, out


def host_init(Xs):
    from oracle import dfm_ref as Rf, kalman_em as K
    ini = [K.init_from_factors(Xs[b], Rf.pca_score(Xs[b], R_), P_) for b in range(Xs.shape[0])]
    return tuple(np.stack([i[j] for i in ini]) for j in range(4))


DUMP_LIMIT = 60 * 2 ** 20        # array bytes written by --dump-outputs (under 64 MB with the .npy headers)


def dump_outputs(path, per_rep, ids, shared=None):
    """Write `shared` and `per_rep` (replication axis first; replication ids `ids`) as <path>/<name>.npy in float64, and
    the ids as replication_id.npy.  If the total would exceed DUMP_LIMIT, a fixed seeded sample of replications is kept."""
    shared = {n: np.asarray(a, np.float64) for n, a in (shared or {}).items()}
    per_rep = {n: np.asarray(a, np.float64) for n, a in per_rep.items()}
    ids = np.asarray(ids, np.float64)
    room = DUMP_LIMIT - sum(a.nbytes for a in shared.values())
    each = 8 + sum(a.nbytes for a in per_rep.values()) // len(ids)
    keep = np.arange(len(ids))
    if each * len(ids) > room:
        keep = np.sort(np.random.default_rng(0).choice(len(ids), room // each, replace=False))
    os.makedirs(path, exist_ok=True)
    for n, a in {**shared, **{n: a[keep] for n, a in per_rep.items()}, "replication_id": ids[keep]}.items():
        np.save(os.path.join(path, n + ".npy"), a)


def em_outputs(out, B, N, r, k, T, iters_cap, it, st):
    """Column-major EM outputs of B panels (host arrays keyed as EmOut) -> caller-shaped arrays; log-likelihood entries
    past each panel's iteration count are NaN (never written)."""
    ll = out["loglik"].reshape(B, iters_cap)
    return {"F": out["F"].reshape(B, r, T).transpose(0, 2, 1), "Lam": out["Lam"].reshape(B, r, N).transpose(0, 2, 1),
            "R": out["R"].reshape(B, N), "A": out["A"].reshape(B, k, r).transpose(0, 2, 1), "Q": out["Q"].reshape(B, r, r).transpose(0, 2, 1),
            "loglik": np.where(np.arange(iters_cap) < it[:, None], ll, np.nan), "iters": it, "status": st}


CPU_SAMPLE_PANELS = 256          # the bounded CPU sample: the first 256 panels of the workload x em_iters iterations


def cpu_sample(iters, steps=1, warmup=1, Xs=None, init=None):
    """The CPU arm, used identically by `--impl reference` and by the product arm's `cpu_baseline`: the oracle's C port
    (OpenMP over panels, threads bound one per physical core of this process's allowance) on the first
    CPU_SAMPLE_PANELS panels of the C2-shaped workload, `iters` EM iterations per step.  Also times one thread."""
    hc = host_cores()
    n = hc["threads"]
    if Xs is None:
        Xs = make_panels_host(CPU_SAMPLE_PANELS, 0)
        init = host_init(Xs)
    for _ in range(warmup):
        cpu_em(Xs[:2 * n], tuple(a[:2 * n] for a in init), 2, nthreads=n)
    t = 0.0; units = 0; out = None
    for _ in range(steps):
        dt, u, out = cpu_em(Xs, init, iters, nthreads=n)
        t += dt; units += u
    dt1, u1, _ = cpu_em(Xs[:2], tuple(a[:2] for a in init), iters, nthreads=1)
    return {"value": units / t, "unit": UNIT, "cores": n, "kind": "port", "host": hc,
            "single_thread_value": u1 / dt1,
            "sample": f"{Xs.shape[0]} panels x {iters} EM iterations per step, oracle C port (gcc -O3, OpenMP over panels, "
                      f"{n} threads bound to physical cores), {t / steps:.1f} s/step"}, t, out


def run_reference(args):
    """--impl reference: the CPU arm.  The reference is Julia (not installable here: no julia, no
    network) and contains no Kalman/EM code, so the oracle's C port of the same EM is timed on the host cores this
    process may use, on a bounded sample of the same workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    iters = args.em_iters
    cpu, t, out = cpu_sample(iters, steps=args.steps, warmup=max(1, min(args.warmup, 2)))
    if args.dump_outputs:
        ll = out["loglik"]
        dump_outputs(args.dump_outputs, {**{n: out[n] for n in ("F", "Lam", "R", "A", "Q", "iters", "status")},
                                         "loglik": np.where(np.arange(ll.shape[1]) < out["iters"][:, None], ll, np.nan)},
                     np.arange(len(ll)))
    v = cpu["value"]
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": f"C2-shaped panels N={NS} r={R_} T={T_}, Kalman-EM, bounded CPU sample", "em_iters": iters},
                      "cpu_baseline": cpu,
                      "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def _peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    if os.path.exists(peaks_path):
        try:
            pk = json.load(open(peaks_path)); peak = float(pk.get("hbm_gbs", peak)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return peak, peak_src


def _dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        sys.stdout.flush(); saved_fd = os.dup(1); os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier(); torch.cuda.synchronize()
        sys.stdout.flush(); os.dup2(saved_fd, 1); os.close(saved_fd)
    return torch, dist, world, rank, local, dev


def _timed(torch, dist, world, dev, fn, nsteps):
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(nsteps):
        fn()
    torch.cuda.synchronize()
    tt = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return float(tt[0])


def run_c4(args):
    """Config C4: bootstrap confidence bands of the factor-VAR impulse responses of the hom_fac_1 model (T = 222, N = 139
    estimation series, r = 8, VAR(4), 5.7 % missing).  A step = one full bootstrap of `--panels` replications per GPU:
    device resampler (dfm_bootstrap_panels) -> standardise + PCA + masked fused ALS (dfm_estimate_factor) -> factor VAR
    (dfm_estimate_var) -> IRF (dfm_irf) -> one all-gather of the per-replication records -> percentile bands
    (dfm_percentiles).  `value` keeps everything device-resident; `e2e` is replicate.bootstrap_irf (host arrays)."""
    torch, dist, world, rank, local, dev = _dist_setup()
    import dynamic_factor_models_b200 as D
    from dynamic_factor_models_b200 import Library, replicate
    from dynamic_factor_models_b200._lib import MEM_DEVICE
    lib = Library(path=os.environ.get("DFM_BENCH_LIB"), device=local)
    z = np.load(os.path.join(ROOT, "tests", "golden", "hom_fac_1_panels.npz"))
    r, p, L, H, burn = 8, 4, 4, 24, 50
    m = D.DFMModel(z["all_bpdata"], z["all_inclcode"], 20, 40, 3, 224, 0, r, 1e-8, L, p)
    D.estimate(m, lib=lib)                                         # the fitted C1 model (estimate!(::NonParametric), :530-543)
    B = args.panels if args.panels != 1250 else 1000 // world      # C4 = 1000 replications, sharded
    K_, W_ = args.steps, args.warmup
    i0, i1 = m.initperiod, m.lastperiod
    incl = m.inclcode == 1
    v = m.factor_var_model
    F0 = m.factor[i0 - 1:i1]; Tw = F0.shape[0]; ns = int(incl.sum()); k = r * p
    resid = v.resid[i0 - 1:i1][p:]
    cm = lambda a: torch.from_numpy(np.ascontiguousarray(np.asarray(a, float).T)).to(dev)      # column-major device copy
    dins = [cm(F0), cm(resid), cm(v.betahat), cm(m.lambda_[incl]), cm(m.uar_coef[incl]),
            torch.from_numpy(np.ascontiguousarray(m.uar_ser[incl])).to(dev), cm(m.data[i0 - 1:i1][:, incl])]
    f0v = dins[0].view(1, r, Tw)
    f64 = lambda n: torch.empty(n, dtype=torch.float64, device=dev)
    dX, dF, dM, dQ, dG, dirf = f64(B * ns * Tw), f64(B * Tw * r), f64(B * k * k), f64(B * r * k), f64(B * k * r), f64(B * r * H * r)
    gathered = f64(world * B * r * H * r) if world > 1 else dirf
    qs = list(replicate.BAND_PERCENTILES); dband = f64(len(qs) * r * H * r)
    sweeps = [0]

    def step_device():
        lib.bootstrap_panels_raw(Tw, ns, r, p, L, resid.shape[0], burn, B, SEED, rank * B, [t.data_ptr() for t in dins], dX.data_ptr())
        st = lib.estimate_factor_raw(dX.data_ptr(), Tw, ns, r, B, MEM_DEVICE, F=dF.data_ptr(), nt_min=m.nt_min_factor_estimation, tol=m.tol)
        sweeps[0] = sum(s_["iters"] for s_ in st)
        lib.sync()
        Fv = dF.view(B, r, Tw)
        sg = torch.sign((Fv * f0v).sum(2)); sg[sg == 0] = 1.0
        Fv.mul_(sg[:, :, None])                                    # factor signs aligned with the original estimate
        torch.cuda.synchronize()
        lib.estimate_var_raw(dF.data_ptr(), Tw, r, p, True, B, MEM_DEVICE, M=dM.data_ptr(), Q=dQ.data_ptr(), G=dG.data_ptr())
        lib.irf_raw(dM.data_ptr(), dQ.data_ptr(), dG.data_ptr(), k, r, H, list(range(r)), B, MEM_DEVICE, dirf.data_ptr())
        lib.sync()
        if world > 1:
            dist.all_gather_into_tensor(gathered, dirf)            # the path's single collective
        lib.percentiles_raw(gathered.data_ptr(), world * B, r * H * r, qs, dband.data_ptr())
        lib.sync()

    for _ in range(W_):
        step_device()
    clocks = ClockSampler(local); clocks.start()
    l0 = lib.launches
    ms = _timed(torch, dist, world, dev, step_device, K_)
    launches = lib.launches - l0
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:                            # records [variable, horizon, shock], as replicate.bootstrap_irf
        dump_outputs(args.dump_outputs, {"irf": dirf.cpu().numpy().reshape(B, r, H, r).transpose(0, 3, 2, 1)}, rank * B + np.arange(B),
                     shared={"bands": dband.cpu().numpy().reshape(len(qs), r, H, r).transpose(0, 3, 2, 1), "percentiles": qs})
    value = world * B * K_ / (ms * 1e-3)
    nfail = int(torch.isnan(dirf.view(B, -1)).any(1).sum().item())

    def step_e2e():
        replicate.bootstrap_irf(lib, m, world * B, H=H, rank=rank, world=world, seed=SEED)

    step_e2e(); step_e2e()                                        # (first calls on a fresh box fault in ~0.7 GB of host pages)
    Ke = 2
    ms_e = _timed(torch, dist, world, dev, step_e2e, Ke)
    nsall = m.ns
    h2d = 8 * B * (Tw * ns + Tw * r + k * k + 2 * r * k)           # panels of the estimation series, factors, M, Q, G
    d2h = 8 * B * (Tw * nsall + Tw * r + ns * r + 2 * ns + (1 + k) * r + Tw * r + r * r + k * k + 2 * r * k + r * H * r)

    # ---- roofline of the dominant kernel (masked fused ALS): X is read twice per sweep (Lambda-step and F-step)
    lib.profile(True); step_device(); prof = lib.profile_report(); lib.profile(False)
    tot = sum(v_[0] for v_ in prof.values()) or 1.0
    dom = max(prof, key=lambda n: prof[n][0])
    als_k = next((n for n in prof if "als_masked" in n), dom)
    peak, peak_src = _peak()
    d_ms, d_cnt = prof[als_k]
    alg = 2.0 * Tw * ns * 8 * sweeps[0]
    roof = {"bound": "hbm", "kernel": als_k, "achieved": alg / (d_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": alg / (d_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
            "kernel_share_of_step": d_ms / tot, "dominant_kernel_of_step": dom, "avg_launch_ms": d_ms / d_cnt, "algorithmic_bytes_per_launch": alg,
            "note": "2*T*N*8 bytes per ALS sweep and panel (SURVEY 8d); the 296 resident panels (73 MB) are re-read from L2, so the "
                    "kernel is latency / issue bound, not HBM bound",
            "kernel_ms": {n: round(v_[0], 3) for n, v_ in sorted(prof.items(), key=lambda kv: -kv[1][0])}}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import dfm_ref as Rf
        nb = 2
        Xb = replicate.bootstrap_panels(m, range(nb), SEED, lib=lib)
        t0 = time.perf_counter()
        for b in range(nb):
            full = np.full_like(z["all_bpdata"], np.nan); full[i0 - 1:i1] = Xb[b]
            mo = Rf.DFMModel(full, z["all_inclcode"], 20, 40, 3, 224, 0, r, 1e-8, L, p)
            Rf.estimate_factor(mo, computeR2=False); Rf.estimate_var(mo.factor_var_model)
            Rf.impulse_response(mo.factor_var_model, list(range(r)), H)
        dt = time.perf_counter() - t0
        cpu = {"value": nb / dt, "unit": "bootstrap replications/s", "cores": 1, "kind": "port",
               "sample": f"{nb} replications re-estimated by oracle/dfm_ref.py (numpy/scipy restatement of estimate_factor!, estimate_var!, "
                         f"impulse_response), {dt:.1f} s"}
    if rank == 0:
        print(json.dumps({"metric": "bootstrap replications/sec (C4: hom_fac_1 model, r=8, VAR(4), IRF H=24)", "value": value,
                          "unit": "bootstrap replications/s", "n_gpus": world, "steps": K_, "warmup": W_, "ms_per_step": ms / K_,
                          "higher_is_better": True, "scaling": "strong" if args.panels == 1250 else "weak", "vs_baseline": None, "dtype": "f64",
                          "data": "residual bootstrap of the hom_fac_1 panel (device resampler)",
                          "config": {"workload": f"C4: {world * B} bootstrap replications of the Stock-Watson panel (T={Tw}, N={ns} estimation "
                                                 f"series, r={r}, VAR({p}), 5.7 % missing): resample -> ALS -> VAR -> IRF(H={H}) -> bands",
                                     "replications_per_gpu": B, "als_sweeps_per_step": sweeps[0], "failed_replications": nfail,
                                     "l2": "panels are regenerated every step; 296 resident panels = 73 MB < L2 (stated, not flushed)"},
                          "e2e": {"value": world * B * Ke / (ms_e * 1e-3), "unit": "bootstrap replications/s", "h2d_bytes_per_step": h2d,
                                  "d2h_bytes_per_step": d2h, "ms_per_step": ms_e / Ke},
                          "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
                          "als": {"value": sweeps[0] * world / (prof[als_k][0] * 1e-3), "unit": "panel-ALS-sweeps/s (masked fused kernel)"}}))
    if world > 1:
        dist.destroy_process_group()
    lib.close()


def run_single_panel(args):
    """Configs C2-single (N=200, r=8, T=500: fused kernel, one CTA, latency bound) and C3 (N=2000, r=20, T=2000: general
    multi-kernel path): ONE panel, Kalman-EM; replicas only across GPUs (SURVEY.md 8e: a single panel does not shard).
    c2-single runs to convergence (relative log-likelihood change 1e-7); c3 runs a fixed 10 iterations."""
    torch, dist, world, rank, local, dev = _dist_setup()
    from dynamic_factor_models_b200 import Library
    from dynamic_factor_models_b200._lib import MEM_DEVICE, MEM_HOST
    import ctypes as C
    lib = Library(path=os.environ.get("DFM_BENCH_LIB"), device=local)
    c3 = args.config == "c3"
    N, r, T, p = (2000, 20, 2000, 1) if c3 else (NS, R_, T_, P_)
    mi, tol = (10, 0.0) if c3 else (500, 1e-7)
    K_, W_ = args.steps, args.warmup
    k = r * p
    f64 = lambda n: torch.empty(n, dtype=torch.float64, device=dev)
    dX, dF0 = f64(T * N), f64(T * r)
    lib.simulate_panels_raw(rank, 1, N, r, T, SEED, dX.data_ptr())
    lib.estimate_factor_raw(dX.data_ptr(), T, N, r, 1, MEM_DEVICE, F=dF0.data_ptr(), max_iter=1)          # PCA + one ALS sweep
    dL0, dR0, dA0, dQ0 = f64(N * r), f64(N), f64(r * k), f64(r * r)
    lib.check(lib.lib.dfm_em_init_from_factors(lib.h, C.c_void_p(dX.data_ptr()), C.c_void_p(dF0.data_ptr()), T, N, r, p, 1, MEM_DEVICE,
                                               C.c_void_p(dL0.data_ptr()), C.c_void_p(dR0.data_ptr()), C.c_void_p(dA0.data_ptr()),
                                               C.c_void_p(dQ0.data_ptr())), "em_init")
    lib.sync()
    dout = {n: f64(sz) for n, sz in dict(Lam=N * r, R=N, A=r * k, Q=r * r, F=T * r, loglik=mi).items()}
    dit = torch.empty(1, dtype=torch.int32, device=dev); dst = torch.empty(1, dtype=torch.int32, device=dev)
    init_d = dict(Lam=dL0.data_ptr(), R=dR0.data_ptr(), A=dA0.data_ptr(), Q=dQ0.data_ptr(), P0=0)
    out_d = dict(Lam=dout["Lam"].data_ptr(), R=dout["R"].data_ptr(), A=dout["A"].data_ptr(), Q=dout["Q"].data_ptr(), P0=0,
                 F=dout["F"].data_ptr(), PF=0, loglik=dout["loglik"].data_ptr(), iters=dit.data_ptr(), status=dst.data_ptr())

    def step_device():
        lib.em_kalman_raw(dX.data_ptr(), T, N, r, p, 1, mi, tol, init_d, out_d, MEM_DEVICE, args.path)
        lib.sync()

    for _ in range(W_):
        step_device()
    clocks = ClockSampler(local); clocks.start()
    l0 = lib.launches
    ms = _timed(torch, dist, world, dev, step_device, K_)
    launches = lib.launches - l0
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, em_outputs({n: t.cpu().numpy() for n, t in dout.items()}, 1, N, r, k, T, mi,
                                                   dit.cpu().numpy(), dst.cpu().numpy()), [rank])
    iters = int(dit.item())
    value = world * iters * K_ / (ms * 1e-3)
    hX = dX.cpu().pin_memory()
    hin = {n: t.cpu().pin_memory() for n, t in dict(Lam=dL0, R=dR0, A=dA0, Q=dQ0).items()}
    hout = {n: torch.empty(t.numel(), dtype=torch.float64).pin_memory() for n, t in dout.items()}
    hit = torch.empty(1, dtype=torch.int32).pin_memory(); hst = torch.empty(1, dtype=torch.int32).pin_memory()
    init_h = dict(Lam=hin["Lam"].data_ptr(), R=hin["R"].data_ptr(), A=hin["A"].data_ptr(), Q=hin["Q"].data_ptr(), P0=0)
    out_h = dict(Lam=hout["Lam"].data_ptr(), R=hout["R"].data_ptr(), A=hout["A"].data_ptr(), Q=hout["Q"].data_ptr(), P0=0,
                 F=hout["F"].data_ptr(), PF=0, loglik=hout["loglik"].data_ptr(), iters=hit.data_ptr(), status=hst.data_ptr())

    def step_e2e():
        lib.em_kalman_raw(hX.data_ptr(), T, N, r, p, 1, mi, tol, init_h, out_h, MEM_HOST, args.path)

    step_e2e()
    Ke = max(2, min(K_, 3))
    ms_e = _timed(torch, dist, world, dev, step_e2e, Ke)
    lib.profile(True); step_device(); prof = lib.profile_report(); lib.profile(False)
    tot = sum(v_[0] for v_ in prof.values()) or 1.0
    dom = max(prof, key=lambda n: prof[n][0])
    peak, peak_src = _peak()
    alg = 2.0 * T * N * 8 * iters
    roof = {"bound": "hbm", "kernel": dom, "achieved": alg / (tot * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (tot * 1e-3) / 1e9 / peak,
            "traffic": None, "peak_source": peak_src, "kernel_share_of_step": prof[dom][0] / tot,
            "algorithmic_bytes_per_step": alg,
            "note": ("one panel: the T-step Kalman / smoother recursions are a serial dependency chain -- latency bound, the HBM fraction "
                     "is reported for completeness (SURVEY.md 8d: do not quote an HBM fraction for B = 1)"),
            "kernel_ms": {n: round(v_[0], 3) for n, v_ in sorted(prof.items(), key=lambda kv: -kv[1][0])}}
    us_per_iter = ms * 1e3 / (K_ * iters)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and not c3:
        from oracle.c import kem
        Xh = np.ascontiguousarray(hX.numpy().reshape(1, N, T).transpose(0, 2, 1))
        Lh = lambda t, rows, cols: np.ascontiguousarray(t.cpu().numpy().reshape(1, cols, rows).transpose(0, 2, 1))
        ini = (Lh(dL0, N, r), dR0.cpu().numpy().reshape(1, N), Lh(dA0, r, k), Lh(dQ0, r, r))
        _omp_env()
        t0 = time.perf_counter()
        o = kem.em_kalman_batch(Xh, *ini, p=p, max_iter=mi, tol=tol, nthreads=1)
        dt = time.perf_counter() - t0
        cpu = {"value": int(o["iters"][0]) / dt, "unit": "EM iterations/s", "cores": 1, "kind": "port",
               "sample": f"the same panel to the same convergence rule, oracle C port, 1 thread, {int(o['iters'][0])} iterations in {dt:.2f} s"}
    if rank == 0:
        name = "C3 (N=2000, r=20, T=2000)" if c3 else "C2 (N=200, r=8, T=500), EM to convergence"
        print(json.dumps({"metric": f"EM iters/sec, single panel {name}", "value": value, "unit": "EM iterations/s", "n_gpus": world,
                          "steps": K_, "warmup": W_, "ms_per_step": ms / K_, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f64", "data": "synthetic (device-generated frozen DGP, SURVEY.md 8d)",
                          "config": {"workload": f"one panel N={N} r={r} T={T} p={p}; " + ("10 EM iterations" if c3 else f"EM to convergence (rel. loglik change {tol}): {iters} iterations"),
                                     "parallelism": f"replicas x{world} (a single panel does not shard)", "iterations": iters,
                                     "status_ok": bool((dst == 0).all().item()), "l2": "panel fits L2 (stated; latency-bound configuration)"},
                          "critical_path": {"us_per_em_iteration": us_per_iter, "us_per_time_step": us_per_iter / T,
                                            "note": "E-step + M-step of one iteration / T periods"},
                          "e2e": {"value": world * int(hit.item()) * Ke / (ms_e * 1e-3), "unit": "EM iterations/s",
                                  "h2d_bytes_per_step": 8 * (T * N + N * r + N + r * k + r * r), "d2h_bytes_per_step": 8 * (T * r + N * r + N + r * k + r * r + mi) + 8,
                                  "ms_per_step": ms_e / Ke},
                          "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu}))
    if world > 1:
        dist.destroy_process_group()
    lib.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--panels", type=int, default=1250, help="panels per GPU (C5 shard = 10000/8)")
    ap.add_argument("--em-iters", type=int, default=50, help="EM iterations per step (SURVEY 8d: fixed 50)")
    ap.add_argument("--path", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--config", default="c5", choices=["c5", "c4", "c3", "c2-single"],
                    help="c5 (default, the headline metric): Monte-Carlo shard of C2-shaped panels; c4: bootstrap IRF bands of the "
                         "hom_fac_1 model; c3: one large panel N=2000 r=20 T=2000; c2-single: one C2 panel, EM to convergence")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if args.config != "c5":
        return {"c4": run_c4, "c3": run_single_panel, "c2-single": run_single_panel}[args.config](args)

    import torch
    import torch.distributed as dist
    from dynamic_factor_models_b200 import Library
    from dynamic_factor_models_b200._lib import MEM_DEVICE, MEM_HOST

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL may print a version banner on stdout: keep stdout clean for the single JSON line
        sys.stdout.flush(); saved_fd = os.dup(1); os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush(); os.dup2(saved_fd, 1); os.close(saved_fd)
    lib = Library(path=os.environ.get("DFM_BENCH_LIB"), device=local)      # DFM_BENCH_LIB: dev-only A/B of kernel variants

    B, iters, K_, W_ = args.panels, args.em_iters, args.steps, args.warmup
    k = R_ * P_; np_ = R_ * (R_ + 1) // 2
    # ---- inputs: this rank's replication shard (ids rank*B .. rank*B+B-1: identical whatever the GPU count), generated
    # on the device (dfm_simulate_panels: counter-based Philox keyed by the replication id)
    dX = torch.empty(B * T_ * NS, dtype=torch.float64, device=dev)
    t_gen = time.perf_counter()
    lib.simulate_panels_raw(rank * B, B, NS, R_, T_, SEED, dX.data_ptr())
    lib.sync(); t_gen = time.perf_counter() - t_gen
    X_cm = dX.cpu()                                                # column-major panels on the host (e2e leg, CPU baseline)
    # initial parameters on the device: one ALS sweep from PCA (reference path) -> init_from_factors
    dF0 = torch.empty(B * T_ * R_, dtype=torch.float64, device=dev)
    lib.estimate_factor_raw(dX.data_ptr(), T_, NS, R_, B, MEM_DEVICE, F=dF0.data_ptr(), max_iter=1)
    dLam0 = torch.empty(B * NS * R_, dtype=torch.float64, device=dev); dR0 = torch.empty(B * NS, dtype=torch.float64, device=dev)
    dA0 = torch.empty(B * R_ * k, dtype=torch.float64, device=dev); dQ0 = torch.empty(B * R_ * R_, dtype=torch.float64, device=dev)
    import ctypes as C
    lib.check(lib.lib.dfm_em_init_from_factors(lib.h, C.c_void_p(dX.data_ptr()), C.c_void_p(dF0.data_ptr()), T_, NS, R_, P_, B, MEM_DEVICE,
                                               C.c_void_p(dLam0.data_ptr()), C.c_void_p(dR0.data_ptr()), C.c_void_p(dA0.data_ptr()),
                                               C.c_void_p(dQ0.data_ptr())), "em_init")
    lib.sync()
    dout = {n: torch.empty(sz, dtype=torch.float64, device=dev) for n, sz in
            dict(Lam=B * NS * R_, R=B * NS, A=B * R_ * k, Q=B * R_ * R_, F=B * T_ * R_, loglik=B * iters).items()}
    dit = torch.empty(B, dtype=torch.int32, device=dev); dst = torch.empty(B, dtype=torch.int32, device=dev)
    init_d = dict(Lam=dLam0.data_ptr(), R=dR0.data_ptr(), A=dA0.data_ptr(), Q=dQ0.data_ptr(), P0=0)
    out_d = dict(Lam=dout["Lam"].data_ptr(), R=dout["R"].data_ptr(), A=dout["A"].data_ptr(), Q=dout["Q"].data_ptr(), P0=0,
                 F=dout["F"].data_ptr(), PF=0, loglik=dout["loglik"].data_ptr(), iters=dit.data_ptr(), status=dst.data_ptr())
    rec = torch.empty(B, 2, dtype=torch.float64, device=dev)       # per-replication record: final loglik, iterations
    gathered = torch.empty(world * B, 2, dtype=torch.float64, device=dev) if world > 1 else None

    def step_device():
        lib.em_kalman_raw(dX.data_ptr(), T_, NS, R_, P_, B, iters, 0.0, init_d, out_d, MEM_DEVICE, args.path)
        lib.sync()
        rec[:, 0] = dout["loglik"].view(B, iters)[:, -1]; rec[:, 1] = dit.to(torch.float64)
        if world > 1:
            dist.all_gather_into_tensor(gathered, rec)             # the path's single collective (NCCL / NVLink)

    def timed(fn, nsteps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter(); e0.record()
        for _ in range(nsteps):
            fn()
        e1.record(); torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        ms = max(ms, 0.0)
        tt = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt[0]), float(tt[1])

    for _ in range(W_):
        step_device()
    clocks = ClockSampler(local); clocks.start()
    l0 = lib.launches
    ms_dev, ms_wall = timed(step_device, K_)
    launches = lib.launches - l0
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:                            # later legs overwrite these buffers
        dump_outputs(args.dump_outputs, em_outputs({n: t.cpu().numpy() for n, t in dout.items()}, B, NS, R_, k, T_, iters,
                                                   dit.cpu().numpy(), dst.cpu().numpy()), rank * B + np.arange(B))
    ms = max(ms_dev, 0.0)
    # library work is on its own stream: the step ends with lib.sync(), so torch-stream events bracket
    # host-synchronised steps; use the larger of event / wall clock (they agree to < 1%)
    ms = max(ms, ms_wall) if ms < 0.5 * ms_wall else ms
    units = world * B * iters * K_
    value = units / (ms * 1e-3)
    status_ok = bool((dst == 0).all().item())

    # ---- e2e through the C ABI with pinned host buffers
    hX = X_cm.pin_memory()
    hin = {n: t.cpu().pin_memory() for n, t in dict(Lam=dLam0, R=dR0, A=dA0, Q=dQ0).items()}
    hout = {n: torch.empty(t.numel(), dtype=torch.float64).pin_memory() for n, t in dout.items()}
    hit = torch.empty(B, dtype=torch.int32).pin_memory(); hst = torch.empty(B, dtype=torch.int32).pin_memory()
    init_h = dict(Lam=hin["Lam"].data_ptr(), R=hin["R"].data_ptr(), A=hin["A"].data_ptr(), Q=hin["Q"].data_ptr(), P0=0)
    out_h = dict(Lam=hout["Lam"].data_ptr(), R=hout["R"].data_ptr(), A=hout["A"].data_ptr(), Q=hout["Q"].data_ptr(), P0=0,
                 F=hout["F"].data_ptr(), PF=0, loglik=hout["loglik"].data_ptr(), iters=hit.data_ptr(), status=hst.data_ptr())
    h2d = 8 * (hX.numel() + sum(t.numel() for t in hin.values()))
    d2h = 8 * sum(t.numel() for t in hout.values()) + 8 * B

    def step_e2e():
        lib.em_kalman_raw(hX.data_ptr(), T_, NS, R_, P_, B, iters, 0.0, init_h, out_h, MEM_HOST, args.path)
        if world > 1:
            rec[:, 0] = hout["loglik"].view(B, iters)[:, -1].to(dev); rec[:, 1] = hit.to(dev).to(torch.float64)
            dist.all_gather_into_tensor(gathered, rec)

    step_e2e()
    Ke = max(2, min(K_, 3))
    _, ms_e2e = timed(step_e2e, Ke)
    e2e_value = world * B * iters * Ke / (ms_e2e * 1e-3)

    # ---- roofline: per-kernel CUDA-event timing of one profiled step (outside the timed region)
    lib.profile(True)
    lib.em_kalman_raw(dX.data_ptr(), T_, NS, R_, P_, B, iters, 0.0, init_d, out_d, MEM_DEVICE, args.path)
    lib.sync()
    prof = lib.profile_report(); lib.profile(False)
    tot = sum(v[0] for v in prof.values()) or 1.0
    dom = max(prof, key=lambda n: prof[n][0]) if prof else None
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    if os.path.exists(peaks_path):
        try:
            pk = json.load(open(peaks_path)); peak = float(pk.get("hbm_gbs", peak)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    roof = None
    if dom:
        d_ms, d_cnt = prof[dom]
        units_per_launch = B * iters / d_cnt                       # panel-iterations one launch of the dominant kernel processes
        alg_bytes = 2.0 * T_ * NS * 8 * units_per_launch           # SURVEY 8d: 2*T*N*8 bytes per panel-iteration
        ach = alg_bytes / (d_ms / d_cnt * 1e-3) / 1e9
        traffic = None; traffic_src = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp) and "fused2" in dom:
            tj = json.load(open(tp)); traffic = tj["dram_bytes_per_panel_iteration"] * units_per_launch; traffic_src = tj["source"]
        roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": peak_src, "kernel_share_of_step": d_ms / tot, "avg_launch_ms": d_ms / d_cnt,
                "algorithmic_bytes_per_launch": alg_bytes,
                "kernel_ms": {n: round(v[0], 3) for n, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}

    # ---- ALS sweep = the reference's own "EM" (estimate_factor!, dfm_functions.ipynb:352-370), reported as a
    # separate line (SURVEY 8d); outside the timed region of the headline metric
    als = None
    if rank == 0 and world == 1:
        sweeps = 10
        dF1 = torch.empty_like(dF0)
        lib.estimate_factor_raw(dX.data_ptr(), T_, NS, R_, B, MEM_DEVICE, F=dF1.data_ptr(), F_init=dF0.data_ptr(), max_iter=2, tol=0.0)
        l0a = lib.launches; t0 = time.perf_counter()
        lib.estimate_factor_raw(dX.data_ptr(), T_, NS, R_, B, MEM_DEVICE, F=dF1.data_ptr(), F_init=dF0.data_ptr(), max_iter=sweeps, tol=0.0)
        lib.sync(); dt = time.perf_counter() - t0
        als = {"value": B * sweeps / dt, "unit": "panel-ALS-sweeps/s", "sweeps": sweeps, "panels": B, "launches": lib.launches - l0a,
               "algorithmic_GBps": 2.0 * T_ * NS * 8 * B * sweeps / dt / 1e9,
               "note": "includes standardisation; starts from given factors (F_init)"}
        if not args.no_cpu:
            from oracle import dfm_ref as Rf
            m_ = Rf.DFMModel(np.ascontiguousarray(X_cm[:T_ * NS].numpy().reshape(NS, T_).T), np.ones(NS, int), 20, 40, 1, T_, 0, R_, 0.0, 4, 1)
            t0 = time.perf_counter(); Rf.estimate_factor(m_, max_iter=3, computeR2=False); dtc = time.perf_counter() - t0
            als["cpu_restated_reference"] = {"value": 3 / dtc, "unit": "panel-ALS-sweeps/s", "cores": 1, "kind": "port",
                                             "sample": "1 panel x 3 sweeps, oracle/dfm_ref.py (numpy/scipy pivoted-QR loops mirroring the reference's control flow; includes one PCA/SVD)"}

    # ---- CPU baseline (rank 0, N=1 only): the same bounded sample as `--impl reference`, started from the device-made
    # initial parameters so that the factors can be compared
    cpu = None; rmse = None
    if rank == 0 and world == 1 and not args.no_cpu:
        Bs = min(B, CPU_SAMPLE_PANELS)
        Lh = lambda t, rows, cols: np.ascontiguousarray(t[:Bs * rows * cols].cpu().numpy().reshape(Bs, cols, rows).transpose(0, 2, 1))
        init = (Lh(dLam0, NS, R_), dR0[:Bs * NS].cpu().numpy().reshape(Bs, NS), Lh(dA0, R_, k), Lh(dQ0, R_, R_))
        Xh = np.ascontiguousarray(X_cm[:Bs * T_ * NS].numpy().reshape(Bs, NS, T_).transpose(0, 2, 1))     # (Bs, T, N)
        cpu, _, out = cpu_sample(iters, steps=1, warmup=1, Xs=Xh, init=init)
        Fg = dout["F"][:Bs * T_ * R_].cpu().numpy().reshape(Bs, R_, T_).transpose(0, 2, 1)
        rmse = float(np.sqrt(np.mean((Fg - out["F"]) ** 2)))

    # ---- "EM to convergence as a user runs it": PCA -> ALS sweep -> initial parameters -> EM until the relative change of
    # the log-likelihood is below 1e-6 (outside the timed region of the headline metric; device resident)
    conv = None
    if rank == 0 and world == 1:
        mi_c = 200
        dll_c = torch.empty(B * mi_c, dtype=torch.float64, device=dev)
        out_c = dict(out_d); out_c["loglik"] = dll_c.data_ptr()
        def init_once():
            lib.estimate_factor_raw(dX.data_ptr(), T_, NS, R_, B, MEM_DEVICE, F=dF0.data_ptr(), max_iter=1)
            lib.check(lib.lib.dfm_em_init_from_factors(lib.h, C.c_void_p(dX.data_ptr()), C.c_void_p(dF0.data_ptr()), T_, NS, R_, P_, B, MEM_DEVICE,
                                                       C.c_void_p(dLam0.data_ptr()), C.c_void_p(dR0.data_ptr()), C.c_void_p(dA0.data_ptr()),
                                                       C.c_void_p(dQ0.data_ptr())), "em_init")
            lib.sync()
        init_once()
        t0 = time.perf_counter(); init_once(); t_init = time.perf_counter() - t0
        t0 = time.perf_counter()
        lib.em_kalman_raw(dX.data_ptr(), T_, NS, R_, P_, B, mi_c, 1e-6, init_d, out_c, MEM_DEVICE, args.path)
        lib.sync(); t_em = time.perf_counter() - t0
        its = dit.to(torch.float64)
        conv = {"init_ms": t_init * 1e3, "em_ms": t_em * 1e3, "panels": B, "tol": 1e-6, "max_iter": mi_c,
                "em_iterations_mean": float(its.mean().item()), "em_iterations_max": int(its.max().item()),
                "panels_per_s": B / (t_init + t_em), "all_status_ok": bool((dst == 0).all().item()),
                "note": "init = standardise + PCA (tensor-core Gram, subspace iteration) + one ALS sweep + initial parameters; wall clock incl. launches"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K_, "warmup": W_,
                "ms_per_step": ms / K_, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic (device-generated frozen DGP, SURVEY.md 8d)",
                "config": {"workload": f"C5 shard of C2-shaped Monte-Carlo panels: {B} panels/GPU, N={NS} r={R_} T={T_} p={P_}, "
                                       f"{iters} EM iterations (Kalman filter + RTS smoother + M-step) per step, then one all-gather",
                           "panels_per_gpu": B, "em_iters_per_step": iters, "parallelism": f"replications x{world}",
                           "l2": f"inputs {B * T_ * NS * 8 / 1e6:.0f} MB/GPU > 126 MB L2 (no flush needed)",
                           "path": args.path, "all_status_ok": status_ok},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / Ke},
                "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
                "factor_rmse_vs_oracle": rmse, "als": als, "e2e_to_convergence": conv, "timing": {"cuda_event_ms": ms_dev, "wall_ms": ms_wall},
                "generator": {"where": "device (dfm_simulate_panels, Philox4x32-10 keyed by replication id)", "panels": B,
                              "seconds": t_gen}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    lib.close()


if __name__ == "__main__":
    main()
