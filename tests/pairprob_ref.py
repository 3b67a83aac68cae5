"""Test-side restatement of the window-averaged base-pair probabilities (--pair_probs, sfb_pairprob_*).

restate() is the definition written out with dense matrices and per-window loops: it is the reference the device table
and the CLI files are compared with.  NumpyPairProbTable mirrors the device table's fixed-point integer sums (same
export / merge / reduce interface as engine.PairProbTable) for the multi-rank tests that run without a GPU."""
import numpy as np

UNIT = 2.0 ** 40
CUTOFF = 0.01


def window_bpp(seq, W, step, w, hc=None, max_span=0, temperature=37.0, pf_scale=None):
    """upper-triangular [W, W] pair probabilities of regular window w from the CPU oracle"""
    from oracle import oracle as O
    s0 = w * step
    o = O.pf(seq[s0:s0 + W], hc=hc[s0:s0 + W] if hc is not None else None, max_span=max_span, temperature=temperature,
             want_bpp=True, pf_scale=pf_scale)
    return np.triu(o["bpp"], 1)


def restate(L, W, step, bpps):
    """bpps[w] = [W, W] upper-triangular probabilities of regular window w, for every regular window of the record.
    -> (paired [L], n_i [L] windows holding each nucleotide, P [L, L] (upper triangle), n_ij [L, L])"""
    S = np.zeros((L, L))
    N = np.zeros((L, L), dtype=np.int64)
    ps = np.zeros(L)
    n_i = np.zeros(L, dtype=np.int64)
    for w, B in enumerate(bpps):
        a = w * step
        S[a:a + W, a:a + W] += B
        N[a:a + W, a:a + W] += 1
        ps[a:a + W] += B.sum(axis=0) + B.sum(axis=1)
        n_i[a:a + W] += 1
    P = np.divide(S, N, out=np.zeros_like(S), where=N > 0)
    paired = np.divide(ps, n_i, out=np.zeros_like(ps), where=n_i > 0)
    return paired, n_i, np.triu(P, 1), N


def pair_list(P, cutoff=CUTOFF):
    """1-based (i, j, P) of the pairs with P >= cutoff, sorted by i then j"""
    i, j = np.nonzero(np.triu(P, 1) >= cutoff)
    return i + 1, j + 1, P[i, j]


class NumpyPairProbTable:
    """CPU stand-in of engine.PairProbTable: the same integer cells and the same reduction"""

    def __init__(self, L, W, step, first_window, n_windows):
        self.L, self.W, self.step = L, W, step
        self.nt0, self.n_nt = first_window * step, (n_windows - 1) * step + W
        self.n_windows = (L - W) // step + 1
        self.cells = np.zeros((self.n_nt, W), dtype=np.int64)

    def add_window(self, w, B):
        q = np.rint(np.triu(B, 1) * UNIT).astype(np.int64)
        r0 = w * self.step - self.nt0
        for i in range(self.W):
            self.cells[r0 + i, 1:self.W - i] += q[i, i + 1:]
            self.cells[r0 + i, 0] += q[i, :].sum() + q[:, i].sum()

    def empty_tensors(self, n_rows):
        import torch
        return (torch.zeros(n_rows * self.W, dtype=torch.int64),)

    def export_tensors(self, row0, n_rows):
        import torch
        return (torch.from_numpy(self.cells[row0:row0 + n_rows].reshape(-1).copy()),)

    def merge_tensors(self, row0, n_rows, rows):
        self.cells[row0:row0 + n_rows] += rows.numpy().reshape(n_rows, self.W)

    def reduce(self, row0=0, n_rows=None, cutoff=CUTOFF):
        from scanfold_b200.engine import windows_holding
        n_rows = self.n_nt - row0 if n_rows is None else n_rows
        rows = self.cells[row0:row0 + n_rows]
        i0 = self.nt0 + row0 + np.arange(n_rows)
        n_i = windows_holding(i0, i0, self.W, self.step, self.n_windows)
        paired = np.divide(rows[:, 0] / UNIT, n_i, out=np.zeros(n_rows), where=n_i > 0)
        r, d = np.nonzero(rows[:, 1:])
        d = d + 1
        n_ij = windows_holding(i0[r], i0[r] + d, self.W, self.step, self.n_windows)
        p = rows[r, d] / UNIT / n_ij
        keep = p >= cutoff
        return paired, (i0[r] + 1)[keep].astype(np.int32), (i0[r] + d + 1)[keep].astype(np.int32), p[keep]
