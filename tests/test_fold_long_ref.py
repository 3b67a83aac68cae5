"""The identities tests/test_gpu_fold_long.py relies on: at 3,000 nt the oracle's whole-sequence fold equals the answer
tests/fold_long_ref.py assembles from island folds, in energy and structure."""
import pytest

import fold_long_ref as R

N = 3000


@pytest.mark.parametrize("a,b", [(0, 500), (1250, 1800), (2450, 3000)], ids=["5p", "middle", "3p"])
def test_n_island_equals_whole_fold(oracle, a, b):
    seq, (e, db) = R.n_island(N, a, b, seed=a + 1)
    eo, so = oracle.mfe(seq)
    assert (eo, so) == (e, db)
    assert so.count("(") > 20
    assert set(so[:a] + so[b:]) <= {"."}


ISLANDS = [(0, 420), (1000, 1480), (2480, 3000)]
SPAN = 400


def _check_x_islands(oracle, T, **kw):
    seq, hc, span, (e, db) = R.x_islands(N, ISLANDS, SPAN, T=T, **kw)
    try:
        eo, so = oracle.mfe(seq, hc=hc, max_span=span, temperature=T)
    finally:
        oracle.set_temperature(37.0)
    assert (eo, so) == (e, db)
    pt = R.pair_table(so)
    for i, j in R.helix_pairs(kw.get("enforce", ())):
        assert pt[i] == j + 1, (i, j)
    for k, ch in enumerate(hc):
        if ch == "x":
            assert pt[k] == 0
    return seq, hc, so


@pytest.mark.parametrize("T", [37.0, 25.0])
def test_x_islands_equal_whole_fold(oracle, T):
    """nested and side-by-side enforced helices and 'x' flags inside the islands, one helix closing at the last nucleotide"""
    enforce = [(10, 300, 3), (40, 120, 4), (150, 260, 3), (1100, 1400, 3), (2700, 2999, 3)]
    _check_x_islands(oracle, T, seed=int(T), enforce=enforce)


def test_x_islands_span_edge(oracle):
    """An enforced helix whose outer pair spans exactly max_span nucleotides forms.  A G-C pair spanning max_span + 1
    nucleotides, which would stack onto an enforced helix, stays open."""
    enforce = [(5, 5 + SPAN - 1, 3), (1011, 1011 + SPAN - 2, 4)]
    plant = [(1010, 1010 + SPAN, 1)]
    seq, hc, so = _check_x_islands(oracle, 37.0, seed=3, enforce=enforce, plant=plant)
    pt = R.pair_table(so)
    i, j = enforce[0][:2]
    assert j - i + 1 == SPAN and pt[i] == j + 1
    i, j = plant[0][:2]
    assert j - i + 1 == SPAN + 1 and pt[i] != j + 1 and pt[i + 1] == j
