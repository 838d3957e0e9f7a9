"""Product-side panel ingestion (dynamic_factor_models_b200/ingest.py, SURVEY 8(f)2) against the committed output of
the ingestion oracle (tests/golden/hom_fac_1_panels.npz = oracle/readin.py on the reference's workbook).  The workbook
is rebuilt as an .xlsx from every cell of its Monthly and Quarterly sheets, stored in tests/golden/hom_fac_1_sheets.tsv.xz
(tests/golden/make_golden.py)."""
import os
import sys

import numpy as np
import pytest

from dynamic_factor_models_b200 import ingest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def xlsx(tmp_path_factory):
    sys.path.insert(0, GOLDEN)
    import make_golden
    path = str(tmp_path_factory.mktemp("workbook") / "hom_fac_1.xlsx")
    make_golden.write_xlsx(path, make_golden.load_sheets(os.path.join(GOLDEN, "hom_fac_1_sheets.tsv.xz")))
    return path


@pytest.mark.parametrize("datatype,key", [("All", "all"), ("Real", "real")])
def test_readin_data_matches_oracle_fixture(xlsx, panels, datatype, key):
    p = ingest.readin_data(xlsx, datatype)
    gold = panels[f"{key}_bpdata"]
    assert p.bpdata.shape == gold.shape
    assert (np.isnan(p.bpdata) == np.isnan(gold)).all()
    np.testing.assert_allclose(p.bpdata, gold, rtol=1e-11, atol=1e-13)      # biweight sums are associated differently
    np.testing.assert_array_equal(p.inclcode, panels[f"{key}_inclcode"])
    assert p.bpnamevec == [str(n) for n in panels[f"{key}_names"]]
    assert p.calds == [tuple(int(v) for v in r) for r in panels["calds"]]
    assert p.row(1959, 3) == 3 and p.row(2014, 4) == 224                   # Stock_Watson.ipynb:1266-1267


def test_survey_panel_facts(xlsx):
    """SURVEY.md section 8: 224 x 207, N = 139 estimation series, 94.3 % observed, 94 balanced columns."""
    p = ingest.readin_data(xlsx, "All")
    est = p.bpdata[2:224][:, p.inclcode == 1]
    assert p.bpdata.shape == (224, 207) and est.shape == (222, 139)
    assert abs(1 - np.isnan(est).mean() - 0.943) < 5e-4
    assert int((~np.isnan(est).any(0)).sum()) == 94


def test_transform_and_biweight_small():
    x = np.array([1.0, 2.0, 4.0, 8.0, np.nan, 32.0])
    np.testing.assert_allclose(ingest.transform_series(x, 5)[1:4], np.log(2) * np.ones(3))
    assert np.isnan(ingest.transform_series(x, 6)[:2]).all()
    X = np.column_stack([np.arange(10.0), np.r_[np.nan, np.ones(9)]])
    tr = ingest.biweight_trend(X, 4.0)
    assert np.isnan(tr[0, 1]) and np.allclose(tr[1:, 1], 1.0)              # local mean of a constant is the constant
    assert np.allclose(tr[4:6, 0], X[4:6, 0])                              # symmetric window around an interior point of a line


def test_workbook_to_table2B_through_product_code(xlsx, notebook_tables):
    """Workbook -> product ingestion -> estimate_factor! through the kernel source (host emulation build) ->
    golden Table 2B row r = 8 (trace R2 0.501, BN-ICp2 -0.223; Stock_Watson.ipynb:619-628)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "emu"))
    import build_emu
    import dynamic_factor_models_b200 as D
    lib = D.Library(build_emu.build())
    try:
        p = ingest.readin_data(xlsx, "All")
        m = D.DFMModel(p.bpdata, p.inclcode, 20, 40, p.row(1959, 3), p.row(2014, 4), 0, 8, 1e-8, 4, 4)
        D.estimate_factor(m, lib=lib)
        gold = np.array(notebook_tables["table2B"])[7]                  # nfac, traceR2, margR2, BN-ICp2, AH-ER
        assert abs((1 - m.fes.ssr / m.fes.tss) - gold[1]) < 6e-4
        assert abs(D.bai_ng_criterion(m) - gold[3]) < 6e-4
    finally:
        lib.close()
