"""tests/scan_ref.py (the reference window loop restated over the oracle) against the golden traces of the UNMODIFIED
reference (tests/golden/*/trace.npz, whose folds came from the same oracle through the RNA shim).  Fed the shuffles the
reference drew, scan_ref must reproduce every recorded field: energies and structures exactly, ED and ensemble dG within
1e-6 relative.  This anchors the restatement the GPU route matrix (tests/test_gpu_scan_routes.py) compares with."""
import os

import numpy as np
import pytest

from scan_ref import OracleCache, scan_ref
from test_host_pipeline import load_case

CASES = ["mono_w40", "hc_w40", "shape_w40", "t25_w40", "step7_w40", "di_w40", "q10_n130_w120", "c1_w120_r100"]
# Q10: the reference skips the fold of a 120-nt all-N window and prints MFE 0, z "#DIV/0", p 0, ED 0 and 120 dots for it.
# Those three -- mfe_dcal, ed, pair_tbl -- are the fields it records for such a window; its shuffles, energy_list,
# centroid and ensemble energy do not exist and are not compared.
ALLN_FIELDS = ("mfe_dcal", "ed", "pair_tbl")


def _inputs(case):
    args = case["args"]
    kw = {}
    if "-t" in args:
        kw["temperature"] = float(args[args.index("-t") + 1])
    if "--constraints" in args:
        kw["hc"] = open(os.path.join(case["dir"], "constraints.dbn")).readlines()[2]
    if "--react" in args:
        from scanfold_b200.cli import read_reactivities
        kw["react"] = read_reactivities(os.path.join(case["dir"], "react.shape"))
    return kw


@pytest.mark.parametrize("name", CASES)
def test_scan_ref_reproduces_golden_trace(oracle, name):
    case = load_case(name)
    t = case["trace"]
    seq, W, step, r, nwin = case["seq"], case["W"], case["step"], case["r"], case["n_windows"]
    n = nwin + 1
    alln = t["alln"] if "alln" in t.files else np.zeros(n, dtype=bool)
    shuf = t["shuffles"].copy()
    for k in np.nonzero(alln)[0]:                  # nothing was drawn for a skipped window: an all-N fragment shuffles to itself
        shuf[k] = ord("N")
    ref = scan_ref(seq, W, step, r, shuf, cache=OracleCache(), **_inputs(case))
    assert ref.n == n == len(t["mfe_dcal"])
    ok = ~alln
    for f in ("mfe_dcal", "native_unconstrained_dcal", "shuffle_dcal", "pair_tbl", "centroid_tbl"):
        got, exp = getattr(ref, f), t[f]
        bad = np.nonzero((got[ok] != exp[ok]).reshape(ok.sum(), -1).any(axis=1))[0]
        assert len(bad) == 0, (name, f, np.nonzero(ok)[0][bad[:5]].tolist())
    for f in ("ed", "ensemble_dG"):
        got, exp = getattr(ref, f), t[f]
        bad = np.nonzero(np.abs(got[ok] - exp[ok]) > 1e-6 * np.maximum(1.0, np.abs(exp[ok])))[0]
        assert len(bad) == 0, (name, f, np.nonzero(ok)[0][bad[:5]].tolist())
    if alln.any():
        for f in ALLN_FIELDS:
            assert np.array_equal(getattr(ref, f)[alln], t[f][alln]), (name, f)
    if name == "shape_w40":                         # the final slot's pf() saw the soft constraints: not a copy (Q5 + Q6)
        assert ref.ed[n - 1] != ref.ed[n - 2] and ref.mfe_dcal[n - 1] == ref.mfe_dcal[n - 2]
    if name == "q10_n130_w120":
        assert alln.sum() > 0
