"""The CPU oracle under energy tables at the edges of the table space (tests/param_tables.py), and the promises of the
table generator itself.  The GPU parity tests (test_gpu_param_edges.py) use the oracle as their reference under the
same tables, so it is checked here first: against exhaustive enumeration, and its tuned batch path against the simple
one."""
import math
import random

import numpy as np
import pytest

import param_tables as PT
from test_oracle import all_structures
from util import rand_seqs

FAMILIES = {"uniform": lambda: PT.uniform(1), "coarse": lambda: PT.coarse(2), "inf": lambda: PT.inf(3),
            "stack_scaled": lambda: PT.stack_scaled(3), "declined_ninio": lambda: PT.declined("ninio"),
            "declined_mismatch": lambda: PT.declined("mismatch")}
FAMILIES.update({"favour_" + c: (lambda c=c: PT.favour(c)) for c in PT.FAVOUR_CLASSES})


@pytest.fixture
def tables(oracle, tmp_path):
    """load(table) -> path; the oracle's own tables and 37 C are restored afterwards"""
    def load(t, name="t.par"):
        path = t.write(tmp_path / name)
        oracle.load_params(path)
        return path
    try:
        yield load
    finally:
        oracle.load_params(oracle.DEFAULT_PAR)
        oracle.set_temperature(37.0)


def _enum_seqs(family, t, rng, n):
    if family == "favour_special":
        return PT.plant_special(t, rng, 16, 1)[:n]
    return ["".join(rng.choice("GGCCAU" if k % 2 else "ACGU") for _ in range(13 + k % 4)) for k in range(n)]


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_oracle_equals_enumeration(oracle, tables, family):
    """MFE = min over all structures, the traced structure evaluates to it, Z and the base-pair probabilities equal the
    Boltzmann sums over all structures (13-16 nt)"""
    t = FAMILIES[family]()
    tables(t)
    rng = random.Random(sum(map(ord, family)))
    kT = (37 + 273.15) * 1.98717 / 1000.0
    for seq in _enum_seqs(family, t, rng, 4):
        structs = all_structures(seq)
        energies = [oracle.eval_structure(seq, s) for s in structs]
        e, db = oracle.mfe(seq)
        assert e == min(energies), (family, seq)
        assert oracle.eval_structure(seq, db) == e, (family, seq, db)
        w = [oracle.eval_weight(seq, s) for s in structs]
        z = sum(w)
        o = oracle.pf(seq, want_bpp=True)
        assert abs(o["dG"] - (-kT * math.log(z))) < 1e-9 * max(1.0, abs(o["dG"])), (family, seq)
        n = len(seq)
        bpp = np.zeros((n, n))
        for s, ws in zip(structs, w):
            stk = []
            for k, ch in enumerate(s):
                if ch == "(":
                    stk.append(k)
                elif ch == ")":
                    bpp[stk.pop(), k] += ws / z
        assert np.abs(bpp - o["bpp"]).max() < 1e-9, (family, seq)


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_fast_batch_path_equals_simple(oracle, tables, family):
    """the tuned batch path (bulk energies of the GPU tests) equals the simple one at 9 / 40 / 120 / 200 nt"""
    t = FAMILIES[family]()
    tables(t)
    for W, n in ((9, 60), (40, 40), (120, 16), (200, 6)):
        seqs = rand_seqs(W + len(family), n, W, gc_rich=True) + PT.plant_special(t, random.Random(W), W, 1)[:6]
        a = np.frombuffer("".join(seqs).encode(), dtype=np.uint8).reshape(len(seqs), W)
        simple = oracle.fold_batch(a, n_threads=4)
        fast = oracle.fold_batch(a, n_threads=4, fast=True)
        assert np.array_equal(simple, fast), (family, W, np.nonzero(simple != fast)[0][:5])


def test_coarse_tables_produce_ties(oracle, tables):
    """coarse tables: many short GC-rich sequences have more than one optimal structure, so traceback order matters"""
    tables(PT.coarse(2))
    rng = random.Random(5)
    ties = 0
    for _ in range(40):
        seq = "".join(rng.choice("GGCCAU") for _ in range(15))
        e, _ = oracle.mfe(seq)
        ties += sum(oracle.eval_structure(seq, s) == e for s in all_structures(seq)) > 1
    assert ties >= 6, ties


@pytest.mark.parametrize("k,W,lo,hi", [(2, 120, 0.1, 0.5), (4, 64, 0.4, 0.8), (3, 120, 0.95, 1.0)])
def test_stack_scaled_crosses_the_int16_bound(oracle, tables, k, W, lo, hi):
    """stack x k puts the stated share of GC-rich folds below -12000 dcal, where the int16 kernels flag for a redo"""
    tables(PT.stack_scaled(k))
    seqs = rand_seqs(100 + k, 150, W, gc_rich=True)
    a = np.frombuffer("".join(seqs).encode(), dtype=np.uint8).reshape(len(seqs), W)
    e = oracle.fold_batch(a, n_threads=8, fast=True)
    frac = float(np.mean(e < -12000))
    assert lo <= frac <= hi, frac


def test_declined_tables_break_the_kernel_conditions():
    """the mirrors of mfe3.cu's split condition (mfe3_upload_tables: 5 * ninio >= max_ninio) and mfe4.cu's 10-bit fit
    (mfe4_upload_tables: fits10) accept the stand-in and every enabled family, and reject the declined variants"""
    std = PT.Table()
    assert PT.mfe3_accepts(std) and PT.mfe4_accepts(std)
    m, mx = PT.declined("ninio").ninio()
    assert 5 * m < mx and not PT.mfe3_accepts(PT.declined("ninio")) and PT.mfe4_accepts(PT.declined("ninio"))
    assert not PT.mfe4_accepts(PT.declined("mismatch")) and PT.mfe3_accepts(PT.declined("mismatch"))
    for s in range(3):
        assert PT.mfe3_accepts(PT.uniform(s)) and PT.mfe3_accepts(PT.coarse(s))
        assert not PT.mfe3_accepts(PT.inf(s))          # INF would wrap in int16: the upload declines the table
    for c in PT.FAVOUR_CLASSES:
        assert PT.mfe3_accepts(PT.favour(c)) and PT.mfe4_accepts(PT.favour(c))


def test_favour_tables_make_their_class_win(oracle, tables):
    """each favoured loop class and size occurs in optimal structures (the class is exercised, not just loaded)"""
    rng = random.Random(8)
    seqs = rand_seqs(81, 30, 120, gc_rich=True)
    tables(PT.favour("hairpin"))
    assert any(max(len(r) for r in s.replace("(", " ").replace(")", " ").split()) > 30 for s in
               (oracle.mfe(x)[1] for x in seqs[:10]))
    tables(PT.favour("special"))
    t = PT.favour("special")
    hits = 0
    for seq in PT.plant_special(t, rng, 40, 3):
        e, db = oracle.mfe(seq)
        hits += e <= -1500
    assert hits > 0.8 * 3 * len(t.special_keys())


@pytest.mark.parametrize("n,T", [(400, 37.0), (450, 37.0), (600, 37.0), (300, 10.0)])
def test_pf_retries_with_a_larger_scale_on_overflow(oracle, n, T):
    """GC-rich sequences whose Z overflows fp64 under the default per-nucleotide scale get finite dG / ED / centroid,
    equal to a PF with exp_params_rescale's scale; the default scale alone really overflows"""
    seq = ("GGCGCC" * 100)[:n] if n == 600 else ("GGGGGCCCCC" * n)[:n]
    with pytest.raises(RuntimeError):
        oracle.pf(seq, temperature=T, pf_scale=0.0)
    e, _ = oracle.mfe(seq, temperature=T)
    kT = (T + 273.15) * 1.98717
    ref = oracle.pf(seq, temperature=T, pf_scale=math.exp(-1.07 * e * 10 / (kT * n)))
    o = oracle.pf(seq, temperature=T)
    assert math.isfinite(o["dG"]) and math.isfinite(o["ed"]) and o["dG"] <= e / 100 + 1e-9
    assert o["dG"] == ref["dG"] and o["ed"] == ref["ed"] and o["centroid"] == ref["centroid"]
    oracle.set_temperature(37.0)


def test_pf_is_scale_invariant(oracle):
    """on ordinary windows the scale changes nothing beyond rounding (<= 1e-12 relative): the overflow retry may use any"""
    for s in rand_seqs(12, 6, 90, gc_rich=True) + ["GGGGAAAACCCC" * 10]:
        a = oracle.pf(s, want_bpp=True)
        for ps in (1.0, 1.7, 3.0):
            b = oracle.pf(s, want_bpp=True, pf_scale=ps)
            assert abs(a["dG"] - b["dG"]) <= 1e-12 * max(1.0, abs(a["dG"]))
            assert abs(a["ed"] - b["ed"]) <= 1e-12 * max(1.0, abs(a["ed"]))
            assert np.abs(a["bpp"] - b["bpp"]).max() <= 1e-12 and a["centroid"] == b["centroid"]


def test_pf_range_at_the_pf2_widths(oracle, tables):
    """the shared-memory PF kernel (<= 120 nt) keeps Z inside fp64 with the default scale for the strongest 120-nt
    folds under the stand-in, uniform, coarse, favour and stack x 2 tables, at 37 C and 10 C.  With stack x 3 it does not
    (MFE below -490 kcal/mol): such windows need the rescaled retry too, which test_gpu_param_edges exercises."""
    worst = [("GGGGGCCCCC" * 12), ("GC" * 60), ("GGCGCC" * 20), "G" * 60 + "C" * 60]
    for name, t in (("uniform", PT.uniform(1)), ("coarse", PT.coarse(2)), ("stack2", PT.stack_scaled(2)),
                    ("special", PT.favour("special")), ("mlintern", PT.favour("mlintern")), ("stack3", PT.stack_scaled(3))):
        tables(t)
        for T in (37.0, 10.0):
            for s in worst:
                try:
                    oracle.pf(s, temperature=T, pf_scale=0.0)
                    finite = True
                except RuntimeError:
                    finite = False
                assert finite == (name != "stack3"), (name, T, s)
