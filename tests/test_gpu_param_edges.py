"""Every MFE / PF kernel against the CPU oracle under energy tables at the edges of the table space (tests/param_tables.py):
random, coarse (ties), INF-holed, one-class-dominant, stack-scaled (int16 redo) and declined tables, across the widths
where the dispatch changes kernel, with flag-only hard constraints, Deigan pseudo-energies and other temperatures; and
partition functions whose Z leaves the fp64 range under the default scale.

Dispatch (api.cu FoldWork, launch_mfe3, pf2_supports): W < 16 mfe.cu; 16-64 / 65-120 / 121-200 / 201-300 mfe3 <64> /
<120> / <200> / <300>; >= 301 mfe4 when the tables fit its packed fields, else mfe.cu; int16 overflow: mfe.cu redo.
PF: pf2 for 10-120 nt with flag-only constraints, pf.cu otherwise and for the rescaled retry."""
import contextlib
import math
import os
import random

import numpy as np
import pytest

import param_tables as PT
from test_gpu_engine import _nested_constraint, _rand_hc
from util import db_from_pt, rand_seqs

pytestmark = pytest.mark.gpu

MFE_WIDTHS = (12, 16, 64, 65, 120, 121, 200, 201, 300, 301, 450)
FAMILIES = {"uniform": lambda: PT.uniform(1), "coarse": lambda: PT.coarse(2), "inf": lambda: PT.inf(3),
            "declined_ninio": lambda: PT.declined("ninio"), "declined_mismatch": lambda: PT.declined("mismatch")}
FAMILIES.update({"favour_" + c: (lambda c=c: PT.favour(c)) for c in PT.FAVOUR_CLASSES})
SFB_E_PARAMS = -2


@contextlib.contextmanager
def loaded(engine, oracle, t, tmp_path, name="t"):
    par = t.write(tmp_path / (name + ".par"))
    try:
        engine.init(0, par)
        oracle.load_params(par)
        yield par
    finally:
        engine.init(0, None)
        oracle.load_params(oracle.DEFAULT_PAR)
        oracle.set_temperature(37.0)
        engine.set_engines(mfe=3, pf=2)


def _oracle_energies(oracle, seqs, temperature=37.0):
    a = np.frombuffer("".join(seqs).encode(), dtype=np.uint8).reshape(len(seqs), len(seqs[0]))
    return oracle.fold_batch(a, n_threads=os.cpu_count(), fast=True, temperature=temperature)


def _seqs(t, W, seed):
    n = 40 if W <= 121 else (10 if W <= 300 else 3)
    out = rand_seqs(seed + W, n, W, gc_rich=True)
    if W <= 300:
        out += PT.plant_special(t, random.Random(seed + W), W, 1 if W > 121 else 3)[:24 if W <= 121 else 6]
    return out + [("GGGGAAAACCCC" * W)[:W], ("GC" * W)[:W], "A" * W]


def _check_mfe(engine, oracle, seqs, kw, okw_of, label, n_sample=3, temperature=37.0):
    """energies of every fold equal the oracle and the int32 kernel; structures equal the int32 kernel for every fold
    and the oracle for a sample"""
    e, pt = engine.fold_batch(seqs, structure=True, temperature=temperature, **kw)
    try:
        engine.set_engines(mfe=1)
        e1, pt1 = engine.fold_batch(seqs, structure=True, temperature=temperature, **kw)
    finally:
        engine.set_engines(mfe=3)
    bad = np.nonzero(e != e1)[0]
    assert len(bad) == 0, (label, [(int(k), seqs[k], int(e[k]), int(e1[k])) for k in bad[:3]])
    bad = np.nonzero((pt != pt1).any(axis=1))[0]
    assert len(bad) == 0, (label, [seqs[k] for k in bad[:3]])
    if not kw:
        eo = _oracle_energies(oracle, seqs, temperature)
        bad = np.nonzero(e != eo)[0]
        assert len(bad) == 0, (label, [(int(k), seqs[k], int(e[k]), int(eo[k])) for k in bad[:3]])
    for k in list(range(n_sample)) + [len(seqs) - 4]:
        eo, so = oracle.mfe(seqs[k], temperature=temperature, **okw_of(k))
        assert e[k] == eo and db_from_pt(pt[k]) == so, (label, k, seqs[k])


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_mfe_kernels_under_table_families(engine, oracle, tmp_path, family):
    t = FAMILIES[family]()
    with loaded(engine, oracle, t, tmp_path):
        for W in MFE_WIDTHS:
            seqs = _seqs(t, W, 500)
            _check_mfe(engine, oracle, seqs, {}, lambda k: {}, (family, W, "plain"))
        rng = random.Random(7)
        for W in (12, 64, 120, 200, 300, 450):     # one width per kernel: random flag-only constraint lines
            seqs = _seqs(t, W, 600)
            hcs = [_rand_hc(rng, W, False) for _ in seqs]
            _check_mfe(engine, oracle, seqs, {"hc": hcs}, lambda k: {"hc": hcs[k]}, (family, W, "hc"))
        for W in (64, 120, 200, 300):              # Deigan pseudo-energies on mfe3, +-4000 kept and +-4001 flagged
            seqs = _seqs(t, W, 700)
            sc = np.random.default_rng(W).integers(-150, 150, size=(len(seqs), W + 1)).astype(np.int32)
            sc[:, 0] = 0
            sc[0, 5], sc[1, W // 2], sc[2, 7], sc[len(seqs) - 4, 9] = 4000, -4000, 4001, -4001
            _check_mfe(engine, oracle, seqs, {"sc": sc}, lambda k: {"sc_stack": sc[k]}, (family, W, "sc"))


def _check_pf(engine, oracle, seqs, label, temperature=37.0, bpp=True):
    res = engine.pf_batch(seqs, want_bpp=bpp, temperature=temperature)
    for k, s in enumerate(seqs):
        o = oracle.pf(s, want_bpp=bpp, temperature=temperature)
        assert abs(res["dG"][k] - o["dG"]) <= 1e-6 * max(1.0, abs(o["dG"])), (label, k, s)
        assert abs(res["ed"][k] - o["ed"]) <= 1e-6 * max(1.0, abs(o["ed"])), (label, k, s)
        if bpp:
            assert np.abs(res["bpp"][k] - o["bpp"]).max() < 1e-9, (label, k)
        assert db_from_pt(res["centroid"][k]) == o["centroid"], (label, k, s)
    return res


@pytest.mark.parametrize("family", ["uniform", "coarse", "inf", "favour_special", "favour_mlintern", "favour_interior"])
def test_pf_kernels_under_table_families(engine, oracle, tmp_path, family):
    t = FAMILIES[family]()
    with loaded(engine, oracle, t, tmp_path):
        for W in (9, 10, 120, 121, 200, 300):
            n = 6 if W <= 121 else (2 if W <= 200 else 1)
            seqs = (rand_seqs(800 + W, n, W, gc_rich=True) + PT.plant_special(t, random.Random(W), W, 1)[:2])[:n + 2]
            r2 = _check_pf(engine, oracle, seqs, (family, W), bpp=W <= 200)
            if 10 <= W <= 120:
                engine.set_engines(pf=1)
                r1 = engine.pf_batch(seqs)
                engine.set_engines(pf=2)
                for key in ("dG", "ed"):
                    assert np.allclose(r1[key], r2[key], rtol=1e-9, atol=1e-9), (family, W, key)
                assert np.array_equal(r1["centroid"], r2["centroid"])


@pytest.mark.parametrize("T", [10.0, 60.0])
def test_random_enthalpies_at_other_temperatures(engine, oracle, tmp_path, T):
    """uniform tables with random enthalpies: every block rescaled to T, one width per MFE and PF kernel"""
    t = PT.uniform(5)
    with loaded(engine, oracle, t, tmp_path):
        for W in (12, 40, 100, 150, 250, 350):
            seqs = _seqs(t, W, 900)[:12 if W <= 121 else 4]
            _check_mfe(engine, oracle, seqs, {}, lambda k: {}, (T, W), n_sample=2, temperature=T)
        for W in (9, 100, 150):
            _check_pf(engine, oracle, rand_seqs(950 + W, 4, W, gc_rich=True), (T, W), temperature=T, bpp=False)


@pytest.mark.parametrize("family", ["uniform", "coarse", "declined_mismatch"])
def test_fold_long_under_table_families(engine, oracle, tmp_path, family):
    t = FAMILIES[family]()
    with loaded(engine, oracle, t, tmp_path):
        for n in (700, 2000):
            rng = random.Random(n)
            seq = rand_seqs(4242 + n, 1, n)[0]
            hc = _nested_constraint(rng, n, 40)
            if family == "declined_mismatch":   # the blocked kernel declines the table: a clean error, no wrong answer
                with pytest.raises(engine.EngineError) as ei:
                    engine.fold_long(seq, hc=hc)
                assert ei.value.code == SFB_E_PARAMS
                continue
            e, pt = engine.fold_long(seq, hc=hc)
            eo, so = oracle.mfe(seq, hc=hc)
            assert e == eo and db_from_pt(pt) == so, (family, n)


@pytest.mark.parametrize("k,W,mixed", [(2, 120, True), (3, 120, False), (4, 64, True), (3, 200, False)])
def test_int16_redo_with_constraints_and_natives(engine, oracle, tmp_path, k, W, mixed):
    """stack x k: folds below -12000 dcal leave the int16 kernels and are folded again in int32 -- with flag-only hard
    constraints, Deigan pseudo-energies, T = 25 and structures, in batches where all or some folds are flagged"""
    t = PT.stack_scaled(k)
    with loaded(engine, oracle, t, tmp_path):
        seqs = rand_seqs(31 * k + W, 40, W, gc_rich=True)
        eo = _oracle_energies(oracle, seqs)
        frac = float(np.mean(eo < -12000))
        assert (0.2 <= frac <= 0.8) if mixed else frac == 1.0, frac
        rng = random.Random(k)
        hcs = [_rand_hc(rng, W, False) for _ in seqs]
        sc = np.random.default_rng(k).integers(-100, 100, size=(len(seqs), W + 1)).astype(np.int32)
        sc[:, 0] = 0
        _check_mfe(engine, oracle, seqs, {}, lambda q: {}, (k, W, "plain"))
        _check_mfe(engine, oracle, seqs, {"hc": hcs}, lambda q: {"hc": hcs[q]}, (k, W, "hc"))
        _check_mfe(engine, oracle, seqs, {"sc": sc}, lambda q: {"sc_stack": sc[q]}, (k, W, "sc"))
        _check_mfe(engine, oracle, seqs, {"hc": hcs, "sc": sc}, lambda q: {"hc": hcs[q], "sc_stack": sc[q]},
                   (k, W, "hc+sc", 25), temperature=25.0)


@pytest.mark.parametrize("k", [2, 3])
def test_int16_redo_in_a_scan(engine, oracle, tmp_path, k):
    """engine.scan at W = 120 under stack x k with parity shuffles, a flag-only constraint line and reactivities: the
    native fold (hc + sc), its unconstrained energy and every shuffle energy of every window equal the oracle, flagged
    windows and unflagged ones alike; the PF of the constrained window stays within 1e-6 (stack x 3 overflows the default
    scale at 120 nt: the rescaled retry)"""
    W, step, r = 120, 9, 3
    rng = random.Random(40 + k)
    seq = "".join(rng.choice("GGCCAU" if (p // 60) % 2 else "ACGU") for p in range(W + 8 * step))
    nwin = (len(seq) - W) // step + 1
    shuf = np.zeros((nwin + 1, r, W), dtype=np.uint8)
    for w in range(nwin + 1):
        start = w * step if w < nwin else len(seq) - W
        for q in range(r):
            shuf[w, q] = np.frombuffer("".join(rng.sample(seq[start:start + W], W)).encode(), dtype=np.uint8)
    hc = "".join(rng.choice("......x<>") for _ in seq)
    L = len(seq)
    react = np.concatenate([[-999.0], np.clip(np.random.default_rng(k).exponential(0.4, L), 0, 4)])
    with loaded(engine, oracle, PT.stack_scaled(k), tmp_path):
        res = engine.scan(seq, W, step, r, parity_shuffles=shuf, hc=hc, react=react, shape_m=0.8, shape_b=-0.2)
        es = oracle.deigan(react, 0.8, -0.2)
        flagged = 0
        for w in range(nwin):
            frag, shc = seq[w * step:w * step + W], hc[w * step:w * step + W]
            scw = np.zeros(W + 1, dtype=np.int32)
            for p in range(1, W):                       # Q7: +1 shift, as test_scan_shape_mode
                g = w * step + 1 + p
                scw[p] = es[g] if g <= L else 0
            eo, so = oracle.mfe(frag, hc=shc, sc_stack=scw)
            assert res.mfe_dcal[w] == eo and db_from_pt(res.pair_tbl[w]) == so, (k, w)
            eu = oracle.mfe(frag, structure=False)[0]
            flagged += eu < -12000
            assert res.native_unconstrained_dcal[w] == eu, (k, w)
            for q in range(r):
                assert res.shuffle_dcal[w, q] == oracle.mfe(bytes(shuf[w, q]).decode(), structure=False)[0], (k, w, q)
            o = oracle.pf(frag, hc=shc)
            assert abs(res.ed[w] - o["ed"]) <= 1e-6 * max(1, abs(o["ed"])), (k, w)
            assert db_from_pt(res.centroid_tbl[w]) == o["centroid"], (k, w)
        assert 0 < flagged < nwin if k == 2 else flagged == nwin, flagged


def test_pf_out_of_fp64_range_is_rescaled(engine, oracle, tmp_path):
    """Z above the fp64 range under the default scale (GC repeats of 400-600 nt at 37 C, 300 nt at 10 C, and at 120 nt on
    the shared-memory kernel under stack x 3): finite dG / ED / centroid equal to the oracle's rescaled PF, in batches
    mixed with ordinary windows, which stay as they were; and the same through a scan plan"""
    for n, T in ((400, 37.0), (450, 37.0), (600, 37.0), (300, 10.0)):
        big = ("GGCGCC" * 100)[:n] if n == 600 else ("GGGGGCCCCC" * n)[:n]
        seqs = [rand_seqs(n, 1, n)[0], big]
        res = _check_pf(engine, oracle, seqs, (n, T), temperature=T, bpp=n <= 400)
        alone = engine.pf_batch(seqs[:1], temperature=T)
        assert alone["dG"][0] == res["dG"][0] and alone["ed"][0] == res["ed"][0]
    oracle.set_temperature(37.0)
    seq = rand_seqs(17, 1, 200)[0] + "GGGGGCCCCC" * 40 + rand_seqs(18, 1, 200)[0]
    W, step = 400, 100
    res = engine.scan(seq, W, step, 2, seed=5)
    nwin = (len(seq) - W) // step + 1
    assert res.n == nwin + 1
    for w in range(nwin + 1):
        start = w * step if w < nwin else len(seq) - W
        o = oracle.pf(seq[start:start + W] if w < nwin else seq[(nwin - 1) * step:(nwin - 1) * step + W])
        assert math.isfinite(res.ed[w]) and abs(res.ed[w] - o["ed"]) <= 1e-6 * max(1, abs(o["ed"])), w
        assert db_from_pt(res.centroid_tbl[w]) == o["centroid"], w
    with loaded(engine, oracle, PT.stack_scaled(3), tmp_path):
        seqs = ["GGGGGCCCCC" * 12, ("GC" * 60), rand_seqs(3, 1, 120)[0]]
        _check_pf(engine, oracle, seqs, "stack3 pf2")
