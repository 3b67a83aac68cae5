"""Exact whole-sequence MFE references at any length, built from oracle folds of a few hundred nucleotides.

The oracle's whole-sequence fold is O(n^3) (about 6 s at 2,000 nt, 20 s at 3,000 nt), so it cannot check sfb_fold_long
at the lengths it exists for (a 29,903-nt genome, up to SFB_MAX_LONG = 40,000 nt).  Two constructions have a known
answer at any length:

1. n_island: every position is N except one island [a, b).  N pairs with nothing, and with dangles = 2 a flanking N
   gives the same exterior terms in the whole sequence as in the island's own fold.  So the MFE and structure are the
   oracle fold of seq[max(a-1, 0):min(b+1, n)], with every position outside the island unpaired.  No constraint line
   and no span limit: this is the product's default path.
2. x_islands: every position outside the islands is flagged 'x' and every gap between two islands is at least the
   span limit, so no pair can leave its island.  The exterior loop is a sum of per-stem terms, so the MFE is the sum
   of the oracle folds of each island together with one flanking ('x') nucleotide on each side, and the structure is
   their concatenation.  Enforced pairs and 'x' flags inside an island, the span limit and the temperature all apply.

tests/test_fold_long_ref.py checks both identities against the oracle's whole-sequence fold at 3,000 nt.
"""
import random

from oracle import oracle as O


def _rand(rng, n):
    return [rng.choice("ACGU") for _ in range(n)]


def n_island(n, a, b, seed):
    """-> (seq, (energy dcal, dot-bracket)): all N except a random ACGU island [a, b)."""
    assert 0 <= a < b <= n
    rng = random.Random(seed)
    seq = "N" * a + "".join(_rand(rng, b - a)) + "N" * (n - b)
    lo, hi = max(a - 1, 0), min(b + 1, n)
    e, s = O.mfe(seq[lo:hi])
    return seq, (e, "." * lo + s + "." * (n - hi))


def helix_pairs(helices):
    """(i, j, k) helices -> the k stacked pairs (i, j), (i+1, j-1), ..., 0-based"""
    return [(i + t, j - t) for i, j, k in helices for t in range(k)]


def x_islands(n, islands, span, seed, enforce=(), plant=(), x_rate=0.03, T=37.0):
    """-> (seq, constraint line, span, (energy dcal, dot-bracket)).

    islands: sorted [a, b) ranges, gaps between them >= span.  Outside the islands the sequence is random and flagged
    'x'.  enforce: (i, j, k) helices of k stacked G-C / C-G pairs written into the sequence and enforced with '(' ')'
    (0-based, inside one island, nested or side by side).  plant: helices written into the sequence the same way but
    not constrained.  x_rate: share of the remaining island positions flagged 'x', one number or one per island.
    The expected structure must contain every enforced pair of span <= span (asserted: a helix that does not form is a
    mistake in the test's design, not in the kernel)."""
    assert span > 0
    for (a0, b0), (a1, b1) in zip(islands, islands[1:]):
        assert b0 <= a1 and a1 - b0 >= span, "islands closer than the span limit"
    rates = list(x_rate) if isinstance(x_rate, (list, tuple)) else [x_rate] * len(islands)
    rng = random.Random(seed)
    seq = _rand(rng, n)
    hc = ["x"] * n
    for a, b in islands:
        hc[a:b] = ["."] * (b - a)

    def island_of(p):
        return next(k for k, (a, b) in enumerate(islands) if a <= p < b)

    for pairs, mark in ((helix_pairs(plant), False), (helix_pairs(enforce), True)):
        for i, j in pairs:
            assert island_of(i) == island_of(j), (i, j)
            seq[i], seq[j] = rng.choice((("G", "C"), ("C", "G")))
            if mark:
                hc[i], hc[j] = "(", ")"
    fixed = {p for ij in helix_pairs(plant) + helix_pairs(enforce) for p in ij}
    for k, (a, b) in enumerate(islands):
        for p in range(a, b):
            if p not in fixed and rng.random() < rates[k]:
                hc[p] = "x"
    seq, hc = "".join(seq), "".join(hc)
    e_sum, db = 0, ["."] * n
    try:
        for a, b in islands:
            lo, hi = max(a - 1, 0), min(b + 1, n)
            e, s = O.mfe(seq[lo:hi], hc=hc[lo:hi], max_span=span, temperature=T)
            e_sum += e
            db[lo:hi] = s
    finally:
        O.set_temperature(37.0)     # the oracle's temperature is global: later eval_structure callers expect 37 C
    db = "".join(db)
    pt = pair_table(db)
    for i, j in helix_pairs(enforce):
        if j - i + 1 <= span:
            assert pt[i] == j + 1, ("enforced pair does not form", i, j)
    return seq, hc, span, (e_sum, db)


def enforced_helices(n, seed, max_span=120, k=3):
    """-> (seq, constraint line, helices): a random sequence with k-pair G-C helices of span <= max_span written in and
    enforced every few hundred nucleotides over the whole record, like the Zavg pair lines --global_refold folds under.
    There is no known MFE: tests check what must hold for any correct fold."""
    rng = random.Random(seed)
    seq, hc, helices = _rand(rng, n), ["."] * n, []
    p = rng.randrange(0, 300)
    while True:
        span = rng.randrange(20, max_span + 1)
        if p + span > n:
            break
        helices.append((p, p + span - 1, k))
        p += span + rng.randrange(100, 800)
    for i, j in helix_pairs(helices):
        seq[i], seq[j] = rng.choice((("G", "C"), ("C", "G")))
        hc[i], hc[j] = "(", ")"
    return "".join(seq), "".join(hc), helices


def pair_table(db):
    """dot-bracket -> 1-based partner list (0 unpaired), the layout of sfb_fold_long's int32 table"""
    pt, stk = [0] * len(db), []
    for k, ch in enumerate(db):
        if ch == "(":
            stk.append(k)
        elif ch == ")":
            i = stk.pop()
            pt[i], pt[k] = k + 1, i + 1
    assert not stk
    return pt
