"""The scan plan's kernel routes against the reference window loop restated over the oracle (tests/scan_ref.py).

sfb_scan_plan_run picks, per chunk, which kernel folds each part of the work: energy-only mfe3 / mfe2 / mfe.cu / mfe4 or
the general path (enforced pairs, span), pf2 or pf.cu, the background temperature for the shuffles and energy_list[0]
and the model temperature for the native fold and the PF, and one of three variants for the final-window slot (Q5: a
copy of the last regular window, a PF re-run with its soft constraints, a rescaled retry).  With parity shuffles every
field of engine.scan is deterministic and must equal scan_ref: integers and structures bit-exact, ED and ensemble dG
within 1e-6 relative (max(1, |x|)).  Every case also runs a shard that starts inside the record and ends with the final
slot, which must equal the same rows of the full scan.

The second half sweeps fold_batch / pf_batch over the widths where the kernels' own geometry changes (below the
hairpin minimum, pf.cu's 256-thread diagonal stride, mfe4's 32-wide block pitch, MAX_W) with batches of n_sm*k + 1
folds, and checks the device shuffles of windows too short to rearrange."""
import os
import random

import numpy as np
import pytest

from scan_ref import FIELDS, OracleCache, react_slice_stack, scan_ref
from test_gpu_engine import _nested_constraint, _rand_hc
from test_gpu_pairprob import check_rows
from util import db_from_pt, rand_seqs

pytestmark = pytest.mark.gpu

R = 2
INT_FIELDS = ("mfe_dcal", "native_unconstrained_dcal", "shuffle_dcal", "pair_tbl", "centroid_tbl")
# width -> the route it selects (native MFE + PF without constraints)
WIDTHS = {8: "mfe.cu + pf.cu", 12: "mfe.cu + pf2", 64: "mfe3 4 warps + pf2", 120: "mfe3 12 warps + pf2",
          121: "mfe3 + pf.cu", 201: "mfe3, multiloop matrix in L2", 300: "mfe3 + pf.cu", 301: "mfe4",
          321: "mfe4 pitch edge", 513: "mfe4 + pf.cu stride edge", 1024: "MAX_W"}
KINDS = ("none", "flags", "brackets", "react", "span", "tbg", "t45")
LONG_KINDS = ("none", "brackets", "react", "span", "tbg")     # above 300 nt: flags and T=45 take no new route


@pytest.fixture(scope="module")
def cache(oracle):
    c = OracleCache()
    yield c
    oracle.set_temperature(37.0)


def np_parity(seq, W, step, r, seed, first_window=0, n_windows=None, final_window=True):
    """seeded mono-nucleotide shuffles [n, r, W] (ASCII) of a shard, the final slot's drawn from seq[L-W:L]"""
    L = len(seq)
    total = (L - W) // step + 1
    n_windows = total - first_window if n_windows is None else n_windows
    n = n_windows + (1 if final_window else 0)
    s = np.frombuffer(seq.encode(), dtype=np.uint8)
    starts = (first_window + np.arange(n)) * step
    if final_window:
        starts[-1] = L - W
    frags = s[starts[:, None] + np.arange(W)[None, :]]                        # [n, W]
    perm = np.argsort(np.random.default_rng(seed).random((n, r, W)), axis=2)
    return np.take_along_axis(np.broadcast_to(frags[:, None, :], (n, r, W)), perm, axis=2).copy()


def rand_react(rng, L):
    react = np.concatenate([[-999.0], np.clip(rng.exponential(0.4, L), 0, 4)])
    react[rng.random(L + 1) < 0.1] = -999.0                                   # missing values
    return react


def kind_kwargs(kind, seq, W, seed):
    L = len(seq)
    rng = random.Random(seed)
    if kind == "none":
        return {}
    if kind == "flags":
        return {"hc": _rand_hc(rng, L, False)}
    if kind == "brackets":
        # nested enforced pairs across the record (window slices cut some of them: unbalanced lines), a stray ')' at the
        # start and an unmatched '(' at the end
        return {"hc": ")" + _nested_constraint(rng, L - 2, max(4, L // 6)) + "("}
    if kind == "react":
        return {"react": rand_react(np.random.default_rng(seed), L)}
    if kind == "span":
        return {"max_span": W // 3}
    if kind == "tbg":
        return {"temperature": 25.0, "background_temperature": 45.0}
    if kind == "t45":
        return {"temperature": 45.0}
    raise ValueError(kind)


def assert_same(got, ref, label, rows=None):
    """engine.scan result vs scan_ref (or another scan): integers exact, ED / dG within 1e-6 * max(1, |x|)"""
    sl = slice(None) if rows is None else rows
    for f in INT_FIELDS:
        a, b = getattr(got, f)[sl], getattr(ref, f)
        bad = np.nonzero((a != b).reshape(len(b), -1).any(axis=1))[0]
        assert len(bad) == 0, (label, f, bad[:6].tolist(), a[bad[:2]].tolist(), b[bad[:2]].tolist())
    for f in ("ed", "ensemble_dG"):
        a, b = getattr(got, f)[sl], getattr(ref, f)
        bad = np.nonzero(~(np.abs(a - b) <= 1e-6 * np.maximum(1.0, np.abs(b))))[0]
        assert len(bad) == 0, (label, f, bad[:6].tolist(), a[bad[:2]].tolist(), b[bad[:2]].tolist())


def geometry(W):
    """(n regular windows, step) with (L - W) % step != 0, so the final slot differs from the last regular window"""
    n_reg = 6 if W <= 300 else 3
    step = W // 4 + 1
    return n_reg, step, W + step * (n_reg - 1) + step // 2 + 1


def run_case(engine, cache, seq, W, step, kw, seed, label, pairprob=None):
    par = np_parity(seq, W, step, R, seed)
    full = engine.scan(seq, W, step, R, parity_shuffles=par, pairprob=pairprob, **kw)
    ref = scan_ref(seq, W, step, R, par, cache=cache, **kw)
    assert full.n == ref.n
    assert_same(full, ref, label)
    nwin = full.n - 1
    f0 = max(1, nwin // 2)                                      # a shard that ends with the last window + final slot
    part = engine.scan(seq, W, step, R, parity_shuffles=par[f0:], first_window=f0, n_windows=nwin - f0, **kw)
    for f in FIELDS:
        assert np.array_equal(getattr(part, f), getattr(full, f)[f0:]), (label, "shard", f)
    return full, ref


def route_cases():
    for W in WIDTHS:
        for kind in (KINDS if W <= 300 else LONG_KINDS):
            yield pytest.param(W, kind, id="W%d-%s" % (W, kind))


@pytest.mark.parametrize("W,kind", list(route_cases()))
def test_scan_route_matches_reference_loop(engine, cache, W, kind):
    n_reg, step, L = geometry(W)
    seq = rand_seqs(60000 + 13 * W + KINDS.index(kind), 1, L, gc_rich=False)[0]
    assert (L - W) % step != 0 and (L - W) // step + 1 == n_reg
    kw = kind_kwargs(kind, seq, W, W * 31 + KINDS.index(kind))
    full, _ = run_case(engine, cache, seq, W, step, kw, seed=W, label=(W, kind, WIDTHS[W]))
    if kind in ("none", "flags", "brackets", "span", "t45") and "react" not in kw:   # Q5 without sc: the final slot is a copy
        for f in ("mfe_dcal", "pair_tbl", "centroid_tbl", "ed", "ensemble_dG"):
            assert np.array_equal(getattr(full, f)[n_reg], getattr(full, f)[n_reg - 1]), (W, kind, f)


@pytest.mark.parametrize("kind", ["none", "react"])
def test_scan_step_greater_than_window(engine, cache, kind):
    W, step = 40, 55
    seq = rand_seqs(61001, 1, W + 4 * step + 17)[0]
    kw = kind_kwargs(kind, seq, W, 5)
    run_case(engine, cache, seq, W, step, kw, seed=7, label=("step>W", kind))


@pytest.mark.parametrize("n_windows", [65536, 65537])
@pytest.mark.parametrize("react", [False, True], ids=["plain", "react"])
def test_final_slot_riding_a_full_chunk(engine, cache, n_windows, react):
    """W = 40, r = 1: 65,536 windows per chunk.  65,536 regular windows put the final slot on the full first chunk
    (cn = chunk + 1, the plan's capacity); 65,537 leave one regular window and the final slot for a second chunk.  With
    reactivities the final slot's PF with soft constraints runs inside the large chunk."""
    W, r = 40, 1
    L = n_windows + W - 1
    rng = np.random.default_rng(n_windows)
    seq = "".join("ACGU"[k] for k in rng.integers(0, 4, L))
    kw = {"react": rand_react(rng, L)} if react else {}
    par = np_parity(seq, W, 1, r, seed=3)
    full = engine.scan(seq, W, 1, r, parity_shuffles=par, want_pf=True, **kw)
    assert full.n == n_windows + 1
    lo = n_windows - 8               # the last eight regular windows (65,535 and 65,536 among them) and the final slot
    ref = scan_ref(seq, W, 1, r, par[lo:], first_window=lo, cache=cache, **kw)
    assert_same(full, ref, ("chunk", n_windows, react), rows=slice(lo, None))
    part = engine.scan(seq, W, 1, r, parity_shuffles=par[lo:], first_window=lo, n_windows=8, **kw)
    for f in FIELDS:
        assert np.array_equal(getattr(part, f), getattr(full, f)[lo:]), (n_windows, react, f)
    head = scan_ref(seq, W, 1, r, par[:3], n_windows=3, final_window=False, cache=cache, **kw)
    assert_same(full, head, ("chunk head", n_windows, react), rows=slice(0, 3))


@pytest.mark.parametrize("react", [True, False], ids=["react-retry", "copy"])
def test_final_slot_rescaled_retry(engine, cache, oracle, react):
    """The last regular window and the final slot are GC repeats whose Z leaves the fp64 range under the default scale.
    With reactivities the final slot is the last regular window's PF WITH its soft constraints, computed again with a
    per-window scale (the final_slot && react branch of the retry); without, it is a copy of that window's rescaled PF."""
    W, step = 400, 100
    seq = rand_seqs(4242, 1, 207)[0] + "GGGGGCCCCC" * 40
    L = len(seq)
    nwin = (L - W) // step + 1
    last = (nwin - 1) * step
    kw = {"react": rand_react(np.random.default_rng(9), L)} if react else {}
    sc = react_slice_stack(kw["react"], last, W, 0.8, -0.2) if react else None
    with pytest.raises(RuntimeError):           # the branch under test is reached: out of range at the default scale
        oracle.pf(seq[last:last + W], sc_stack=sc, pf_scale=0)
    full, ref = run_case(engine, cache, seq, W, step, kw, seed=11, label=("retry", react))
    o = oracle.pf(seq[last:last + W], sc_stack=sc)                              # rescaled as the oracle does it
    assert np.isfinite(full.ed[nwin]) and np.isfinite(full.ensemble_dG[nwin])
    assert abs(full.ensemble_dG[nwin] - o["dG"]) <= 1e-6 * max(1.0, abs(o["dG"]))
    assert abs(full.ed[nwin] - o["ed"]) <= 1e-6 * max(1.0, abs(o["ed"]))
    assert db_from_pt(full.centroid_tbl[nwin]) == o["centroid"]
    if react:
        assert full.ed[nwin] != full.ed[nwin - 1]
    else:
        assert full.ed[nwin] == full.ed[nwin - 1] and full.ensemble_dG[nwin] == full.ensemble_dG[nwin - 1]


@pytest.mark.parametrize("W", [12, 121, 301])
@pytest.mark.parametrize("kind", ["brackets", "span", "tbg"])
def test_pairprob_table_on_routes(engine, cache, oracle, W, kind):
    """The pair-probability table sums the same PF the scan reports, on the routes above: it equals the restatement over
    the oracle's per-window pair probabilities (hard constraints, span and the model temperature apply)."""
    n_reg, step, L = geometry(W)
    seq = rand_seqs(62000 + W + KINDS.index(kind), 1, L)[0]
    kw = kind_kwargs(kind, seq, W, W + KINDS.index(kind))
    t = engine.PairProbTable(L, W, step, 0, n_reg)
    try:
        run_case(engine, cache, seq, W, step, kw, seed=W + 1, label=("pairprob", W, kind), pairprob=t)
        check_rows(t, seq, W, step, 0, n_reg, 0, (n_reg - 1) * step + W, hc=kw.get("hc"), max_span=kw.get("max_span", 0),
                   temperature=kw.get("temperature", 37.0))
    finally:
        t.close()
        oracle.set_temperature(37.0)


# ---------------------------------------------------------------------------------------------------------------------
# kernel width sweep

def n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def sweep_seqs(W, n, seed):
    seqs = rand_seqs(seed, n - 3, W, gc_rich=True)
    return seqs + [("GGGGGCCCCC" * W)[:W], "A" * W, ("ACGUN" * W)[:W]]


@pytest.mark.parametrize("W", [1, 2, 3, 4, 6, 7, 15, 319, 320, 321, 1023])
def test_mfe_width_sweep(engine, oracle, W):
    """energies (every fold, against the oracle's batch path) and structures (head and tail of the batch, every fold
    below 16 nt) of fold_batch with n_sm*k + 1 folds"""
    n = 2 * n_sm() + 1 if W <= 15 else (n_sm() + 1 if W <= 321 else 5)
    seqs = sweep_seqs(W, n, 63000 + W)
    e, pt = engine.fold_batch(seqs, structure=True)
    e2, _ = engine.fold_batch(seqs, structure=False)
    assert np.array_equal(e, e2), W
    a = np.frombuffer("".join(seqs).encode(), dtype=np.uint8).reshape(n, W)
    eo = oracle.fold_batch(a, n_threads=os.cpu_count() or 1, fast=True) if W > 15 else [oracle.mfe(s)[0] for s in seqs]
    bad = np.nonzero(e != eo)[0]
    assert len(bad) == 0, (W, bad[:5].tolist())
    check = range(n) if W <= 15 else list(range(4)) + list(range(n - 5, n))
    for k in check:
        assert db_from_pt(pt[k]) == oracle.mfe(seqs[k])[1], (W, k)


@pytest.mark.parametrize("W", [1, 2, 3, 4, 5, 9, 255, 256, 257, 511, 512, 513, 601, 767, 1024])
def test_pf_width_sweep(engine, oracle, W):
    """dG / ED (1e-6 relative), centroid (exact) and base-pair probabilities (1e-9 absolute) of pf_batch(want_bpp=True)
    with n_sm*k + 1 folds where cheap; every fold below 10 nt, head and tail of the batch above"""
    n = 2 * n_sm() + 1 if W <= 9 else (n_sm() + 1 if W <= 257 else (9 if W <= 513 else 3))
    seqs = sweep_seqs(W, n, 64000 + W)
    res = engine.pf_batch(seqs, want_bpp=True)
    check = range(n) if W <= 9 else (list(range(3)) + list(range(n - 3, n)) if n > 6 else range(n))
    if W >= 767:
        check = [0, n - 1]
    for k in check:
        o = oracle.pf(seqs[k], want_bpp=True)
        assert abs(res["dG"][k] - o["dG"]) <= 1e-6 * max(1.0, abs(o["dG"])), (W, k)
        assert abs(res["ed"][k] - o["ed"]) <= 1e-6 * max(1.0, abs(o["ed"])), (W, k)
        assert db_from_pt(res["centroid"][k]) == o["centroid"], (W, k)
        assert np.abs(np.triu(res["bpp"][k], 1) - np.triu(o["bpp"], 1)).max() <= 1e-9, (W, k)


@pytest.mark.parametrize("stype", ["mono", "di"])
def test_shuffles_of_windows_below_three_nt(engine, stype):
    """windows of 1-3 nt: a shuffle keeps the composition; where no other arrangement exists it is the window itself
    (every 1-nt window; 2-nt homopolymers for mono; every di shuffle up to 3 nt, which keeps both end nucleotides and the
    dinucleotides)"""
    seq = "ACGUUGCAAAGGGCUCCUAGUAC"
    r = 16
    for W in (1, 2, 3):
        plan = engine.ScanPlan(seq, W, 1, r, shuffle_type=stype, seed=W, keep_shuffles=True)
        try:
            res = plan.run().fetch()
        finally:
            plan.close()
        nwin = len(seq) - W + 1
        for w in range(nwin + 1):
            frag = seq[w:w + W] if w < nwin else seq[-W:]
            for k in range(r):
                sh = bytes(res.shuffles[w, k]).decode()
                assert sorted(sh) == sorted(frag), (stype, W, w, sh)
                if W == 1 or stype == "di" or len(set(frag)) == 1:
                    assert sh == frag, (stype, W, w, sh)
                if stype == "di" and W == 3:
                    assert sh[0] == frag[0] and sh[-1] == frag[-1]
                    assert sorted([sh[0:2], sh[1:3]]) == sorted([frag[0:2], frag[1:3]])
