"""sfb_fold_long (the three whole-sequence folds of --global_refold) from 2,000 nt to SFB_MAX_LONG = 40,000 nt.

Up to 3,000 nt the oracle folds the whole sequence.  Above that its O(n^3) fold is out of reach, and the exact answers
come from tests/fold_long_ref.py: an island of sequence in a run of N, or islands between 'x'-flagged gaps at least as
long as the span limit, folded by the oracle island by island.  The lengths sit where the blocked kernel (mfe4.cu) could
go wrong: one C / FML / split matrix past 2^31 bytes (n >= 23,169), the three past 2^31 elements (n >= 26,753), partner
indices past int16 (n >= 32,768), the exterior kernel's f5 row at 160 KB of shared memory and the matrix row whose byte
offset passes 2^31 (40,000 nt).  A 40,000-nt fold needs 19.2 GB of device memory; a device that cannot give it skips.
"""
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import fold_long_ref as R
from util import db_from_pt, rand_seqs

pytestmark = pytest.mark.gpu


def _nested_constraint(rng, n, n_pairs):
    """a constraint line with nested / side-by-side enforced pairs '(' ')' plus a few 'x' flags"""
    hc = ["."] * n
    free = [(0, n - 1)]
    for _ in range(n_pairs):
        if not free:
            break
        lo, hi = free.pop(rng.randrange(len(free)))
        if hi - lo < 12:
            continue
        i = rng.randrange(lo, lo + (hi - lo) // 3)
        j = rng.randrange(hi - (hi - lo) // 3, hi + 1)
        if j - i < 5:
            continue
        hc[i], hc[j] = "(", ")"
        free += [(lo, i - 1), (i + 1, j - 1), (j + 1, hi)]
    for k in range(n):
        if hc[k] == "." and rng.random() < 0.03:
            hc[k] = "x"
    return "".join(hc)


def _fold(engine, seq, **kw):
    """engine.fold_long; a device that cannot hold the fold's matrices (shared GPU) skips instead of failing"""
    try:
        e, pt = engine.fold_long(seq, **kw)
    except engine.EngineError as err:
        if "out of memory" in str(err):
            pytest.skip("%d-nt fold: device memory not available (%s)" % (len(seq), err))
        raise
    assert pt.dtype == np.int32 and pt.shape == (len(seq),)
    return e, pt


def _table(db):
    return np.asarray(R.pair_table(db), dtype=np.int32)


def _eval(oracle, seq, db, T=37.0):
    """oracle energy of a structure at temperature T (eval_structure uses the oracle's current temperature)"""
    oracle.set_temperature(T)
    try:
        return oracle.eval_structure(seq, db)
    finally:
        oracle.set_temperature(37.0)


# ---- direct oracle parity, 2,001-3,000 nt: the 64-block edge of mfe4 (NP = 2,048 / 2,080) and 3,000 nt

DIRECT_N = (2047, 2048, 2049, 3000)
DIRECT_VARIANTS = ("plain", "hc", "span", "T25")


def _direct_case(n, variant):
    seq = rand_seqs(40000 + n, 1, n)[0]
    kw = {}
    if variant == "hc":
        kw["hc"] = _nested_constraint(random.Random(n), n, 60)
    elif variant == "span":
        kw["max_span"] = 400
    elif variant == "T25":
        kw["temperature"] = 25.0
    return seq, kw


@pytest.fixture(scope="module")
def direct_ref(oracle):
    """oracle folds of every direct case, on all cores (the oracle releases the GIL).  The oracle's temperature is
    global state, so each pool runs the folds of one temperature only."""
    cases = {(n, v): _direct_case(n, v) for n in DIRECT_N for v in DIRECT_VARIANTS}
    out = {}
    try:
        for T in (37.0, 25.0):
            keys = [k for k, (_, kw) in cases.items() if kw.get("temperature", 37.0) == T]
            oracle.set_temperature(T)
            with ThreadPoolExecutor(max(1, min(len(keys), os.cpu_count() or 1))) as ex:
                futs = {k: ex.submit(oracle.mfe, cases[k][0], hc=cases[k][1].get("hc"),
                                     max_span=cases[k][1].get("max_span", 0), temperature=T) for k in keys}
                out.update({k: f.result() for k, f in futs.items()})
    finally:
        oracle.set_temperature(37.0)
    return cases, out


@pytest.mark.parametrize("variant", DIRECT_VARIANTS)
@pytest.mark.parametrize("n", DIRECT_N)
def test_direct_oracle_parity(engine, direct_ref, n, variant):
    cases, ref = direct_ref
    seq, kw = cases[(n, variant)]
    eo, so = ref[(n, variant)]
    e, pt = _fold(engine, seq, **kw)
    assert e == eo, (n, variant)
    assert db_from_pt(pt) == so, (n, variant)
    assert np.array_equal(pt, _table(so)), (n, variant)
    if variant == "hc":
        assert all(pt[k] == 0 for k, ch in enumerate(kw["hc"]) if ch == "x")


# ---- construction 1: one island in N (no constraint line, no span limit) at the size edges

ISLAND = 560


def _island_at(n, where):
    if where == "5p":
        return 0, ISLAND
    if where == "3p":
        return n - ISLAND, n
    if where == "row":            # the row of the C matrix whose byte offset passes 2^31 (NP = pitch of n)
        r = (1 << 31) // (4 * (-(-n // 32) * 32))
        return r - ISLAND // 2, r + ISLAND // 2
    return n // 2 - ISLAND // 2, n // 2 + ISLAND // 2


@pytest.mark.parametrize("n,where", [(23168, "3p"), (23169, "3p"), (26752, "3p"), (26753, "3p"), (29903, "mid"),
                                     (32768, "3p"), (32769, "3p"), (40000, "5p"), (40000, "row"), (40000, "3p")])
def test_n_island_size_edges(engine, n, where):
    """A 3' island is drawn (first of 20 seeds) so that its fold pairs the last nucleotide: from 32,768 nt on the table
    then holds partners past the int16 range, whatever the island's random fold would have done."""
    a, b = _island_at(n, where)
    for seed in range(n + b, n + b + (20 if where == "3p" else 1)):
        seq, (eo, so) = R.n_island(n, a, b, seed=seed)
        if so[n - 1] == ")":
            break
    assert so.count("(") > 20
    if where == "3p":
        assert so[n - 1] == ")"
        assert n < 32768 or _table(so).max() > 32767
    e, pt = _fold(engine, seq)
    assert e == eo, (n, where)
    assert np.array_equal(pt, _table(so)), (n, where, np.nonzero(pt != _table(so))[0][:10])
    assert not pt[:a].any() and not pt[b:].any()


# ---- construction 2: islands between 'x' gaps, enforced pairs, flags, span and temperature at full length

SPAN = 400


def _c2_layout(n, mid):
    """islands at both ends and one around `mid`.  5' island: an enforced helix whose outer pair spans exactly SPAN and
    a nested one.  Middle island: an enforced helix with a G-C pair of span SPAN + 1 planted on top of it (it must stay
    open) and a nested helix.  3' island: an enforced helix closing at the last nucleotide n - 1, and a nested one."""
    m = mid - 220
    islands = [(0, 450), (m, m + 450), (n - 480, n)]
    enforce = [(10, 10 + SPAN - 1, 3), (60, 200, 4),
               (m + 11, m + 11 + SPAN - 2, 4), (m + 100, m + 300, 3),
               (n - 350, n - 1, 3), (n - 300, n - 100, 3)]
    plant = [(m + 10, m + 10 + SPAN, 1)]
    return islands, enforce, plant


C2_CASES = {
    # the 3' island carries no constraint: the line passed to the kernel stops before it and is padded with '.'
    "29903-short-line": (29903, 37.0, True),
    "40000": (40000, 37.0, False),
    "40000-T25": (40000, 25.0, False),
}


@pytest.mark.parametrize("case", list(C2_CASES))
def test_x_islands_full_length(engine, oracle, case):
    n, T, short = C2_CASES[case]
    islands, enforce, plant = _c2_layout(n, (1 << 31) // (4 * n) if n == 40000 else n // 2)
    if short:
        enforce = [h for h in enforce if h[0] < islands[-1][0]]
    x_rate = [0.03, 0.03, 0.0 if short else 0.03]
    seq, hc, span, (eo, so) = R.x_islands(n, islands, SPAN, seed=n + int(T), enforce=enforce, plant=plant, x_rate=x_rate,
                                          T=T)
    line = hc.rstrip(".") if short else hc
    if short:
        assert len(line) == islands[-1][0] and so[len(line):].count("(") > 20
    e, pt = _fold(engine, seq, hc=line, max_span=span, temperature=T)
    assert e == eo, case
    assert db_from_pt(pt) == so, case
    assert np.array_equal(pt, _table(so)), case
    for i, j in R.helix_pairs(enforce):
        assert pt[i] == j + 1 and pt[j] == i + 1, (case, i, j)
    if not short:
        assert pt[n - 1] > 0
    i, j = plant[0][:2]
    assert pt[i] != j + 1, case
    assert _eval(oracle, seq, db_from_pt(pt), T) == e, case


# ---- full length without a known answer: what any correct fold must satisfy

@pytest.mark.parametrize("n", [29903, 40000])
def test_full_length_self_consistency(engine, oracle, n):
    seq, hc, helices = R.enforced_helices(n, seed=n)
    assert len(helices) > 40
    e0, pt0 = _fold(engine, seq)
    e1, pt1 = _fold(engine, seq, hc=hc)
    e2, pt2 = _fold(engine, seq, hc=hc)
    assert e2 == e1 and np.array_equal(pt2, pt1)
    assert e1 >= e0
    for pt in (pt0, pt1):
        paired = np.nonzero(pt)[0]
        assert np.array_equal(pt[pt[paired] - 1], paired + 1)       # a symmetric table
    assert _eval(oracle, seq, db_from_pt(pt0)) == e0
    assert _eval(oracle, seq, db_from_pt(pt1)) == e1
    open_pairs = _check_weak_enforcement(oracle, seq, db_from_pt(pt1), e1, R.helix_pairs(helices))
    # not a property of every correct fold (a weakly enforced pair may stay open), but of these seeded records: a
    # three-pair G-C helix always forms here, so the constrained fold really runs with enforced pairs in it
    assert not open_pairs


# ---- API edges

@pytest.mark.parametrize("n", [300, 301, 320, 321])
def test_batch_and_blocked_route_edge(engine, oracle, n):
    """300 nt is the last length sfb_fold_long hands to the 16-bit batch path, 301 the first on mfe4; 320 / 321 are
    mfe4's pitch edge"""
    seq = rand_seqs(60000 + n, 1, n)[0]
    for hc in (None, _nested_constraint(random.Random(n), n, 12)):
        e, pt = _fold(engine, seq, hc=hc)
        eo, so = oracle.mfe(seq, hc=hc)
        assert e == eo and db_from_pt(pt) == so, (n, hc is not None)


def test_length_limit(engine):
    with pytest.raises(engine.EngineError) as err:
        engine.fold_long("ACGU" * 10000 + "A")
    assert err.value.code == -5     # SFB_E_RANGE


# ---- --global_refold end to end at genome length

def _bracket_pairs(line):
    """the enforced pairs of a constraint line as the engine reads it: '(' ')' matched by a stack, unmatched ignored"""
    stk, pairs = [], []
    for k, ch in enumerate(line):
        if ch == "(":
            stk.append(k)
        elif ch == ")" and stk:
            pairs.append((stk.pop(), k))
    return pairs


def _check_weak_enforcement(oracle, seq, db, e, pairs):
    """'(' ')' pairs are enforced weakly (ViennaRNA's default hc_add_from_db, SURVEY A.5): every pair that conflicts
    with one is forbidden, but the pair itself may stay open.  So each is either in the structure or has both ends
    unpaired, nothing crosses it, and adding an open one (with the open pairs stacked on it) must not lower the
    oracle's energy e of the structure.  -> the open pairs."""
    pt = _table(db)
    open_pairs = []
    for i, j in pairs:
        assert (pt[i], pt[j]) in ((j + 1, i + 1), (0, 0)), (i, j, pt[i], pt[j])
        inner = pt[i + 1:j]
        assert np.all((inner == 0) | ((inner > i + 1) & (inner <= j))), (i, j)   # nothing crosses (i, j)
        if pt[i] == 0:
            open_pairs.append((i, j))
    for run in _open_runs(open_pairs):
        alt = list(db)
        for i, j in run:
            alt[i], alt[j] = "(", ")"
        assert _eval(oracle, seq, "".join(alt)) >= e, run
    return open_pairs


def _open_runs(pairs):
    """enforced pairs left open, grouped into runs of stacked pairs"""
    runs = []
    for i, j in sorted(pairs):
        if runs and runs[-1][-1] == (i - 1, j + 1):
            runs[-1].append((i, j))
        else:
            runs.append([(i, j)])
    return runs


def test_global_refold_genome_length(engine, oracle, tmp_path, monkeypatch):
    """The constraint lines are the Zavg pairs of the scan, enforced weakly (see _check_weak_enforcement): on this
    record some of them stay open."""
    from scanfold_b200 import cli
    n = 29903
    rng = random.Random(29903)
    seq = "".join(rng.choice("ACGU") for _ in range(n))
    (tmp_path / "genome.fa").write_text(">genome\n%s\n" % seq)
    monkeypatch.chdir(tmp_path)
    cli.main(["genome.fa", "-w", "120", "-r", "10", "--global_refold", "--seed", "5"])
    out = tmp_path / "genome"
    lines = (out / "AllDBN-global_refold.txt").read_text().split("\n")
    assert len(lines) == 10 and lines[9] == ""
    constraints = {1: "Zavg_-1_pairs.dbn", 2: "Zavg_-2_pairs.dbn"}
    energy = []
    for rec in range(3):
        head, s, db = lines[3 * rec:3 * rec + 3]
        assert s == seq and len(db) == n
        _table(db)                                           # raises unless balanced
        e = _eval(oracle, seq, db)
        energy.append(e)
        assert str(float(np.float32(e / 100.0))) == head.split("MFE=")[1], head
        if rec not in constraints:
            continue
        assert e >= energy[0]
        line = (out / constraints[rec]).read_text().split("\n")[2]
        pairs = _bracket_pairs(line)
        assert pairs, constraints[rec]
        _check_weak_enforcement(oracle, seq, db, e, pairs)
