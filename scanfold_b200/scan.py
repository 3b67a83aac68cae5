"""The scan step of ScanFold for one record: every window's native fold, partition function, r shuffled
background folds, z-score and p-value -- the loop ScanFold.py:429-692 plus the final-window block
:694-757 -- as ONE batched call into the CUDA engine instead of 2 process pools per window.

The arithmetic (folds, shuffles, partition function) runs only in libscanfold_b200.so; this module is
the host side above the C-ABI: window bookkeeping, the float32 conversions of the ViennaRNA return
values, and the `statistics`-exact z / p of stats.py.
"""
import numpy as np

from . import engine, stats


class WindowTable:
    """Per-window results of a record (or of one shard of its windows), in window order.

    start1/end1       1-based inclusive coordinates        ScanFold.py:431,436-437
    mfe               round(MFE, 2) as float64             :501/:516/:542
    z, p              rounded z-score / p-value            :554,:560
    ed                round(mean_bp_distance, 2)           :504
    pair_tbl          [n, W] int16 MFE structure (1-based partner in the window, 0 unpaired)
    centroid_tbl      [n, W] int16 centroid structure
    final_*           the extra values the final-window block appends to the wig tracks and to
                      zscore_total (Q5); None on shards that do not hold the last window
    """

    def __init__(self):
        self.W = self.step = self.r = self.first_window = 0
        self.start1 = self.end1 = None
        self.mfe_dcal = self.mfe = self.z = self.p = self.ed = None
        self.native_unconstrained_dcal = self.shuffle_dcal = None
        self.pair_tbl = self.centroid_tbl = None
        self.final = None
        self.alln = None           # [n] bool: windows the reference short-circuits as all-N (Appendix B Q10), or None
        self.ms_total = self.ms_mfe = 0.0
        self.n_launches = 0

    def __len__(self):
        return len(self.start1)

    def structure(self, k):
        return engine.pair_table_to_dotbracket(self.pair_tbl[k])

    def centroid(self, k):
        return engine.pair_table_to_dotbracket(self.centroid_tbl[k])


def n_windows_of(L, W, step):
    """windows at i = 0, step, 2*step, ... <= L - W   (ScanFold.py:429,687)"""
    return (L - W) // step + 1 if L >= W else 0


def all_n_windows(seq, W, step, first_window, n_windows):
    """Windows the reference never folds (ScanFold.py:486-492): the fragment equals a LITERAL string of 120 'N', so the
    test only ever fires for 120-nt windows made of upper-case N (Appendix B Q10).  -> bool [n_windows] or None."""
    if W != 120 or "N" * 120 not in seq:
        return None
    is_n = np.frombuffer(seq.encode(), dtype=np.uint8) == ord("N")
    c = np.concatenate([[0], np.cumsum(is_n)])
    start = (first_window + np.arange(n_windows, dtype=np.int64)) * step
    return (c[start + W] - c[start]) == W


def final_window_all_n(seq, W):
    """the final-window block's own test, `frag == "N" * window_size` (ScanFold.py:719): any window length"""
    return seq[len(seq) - W:] == "N" * W


def round_ed(ed):
    """round(fc.mean_bp_distance(), 2) of ScanFold.py:504, vectorised (Python round on the boundary cases)"""
    ed = np.asarray(ed, dtype=np.float64)
    x = ed * 100.0
    out = np.rint(x) / 100.0
    risky = np.nonzero(np.abs(x - np.floor(x) - 0.5) < 1e-7)[0]
    for k in risky:
        out[k] = round(float(ed[k]), 2)
    return out


def empty_table(W, step, r, first_window=0):
    """a shard without windows (more ranks than windows): zero-length columns of the right dtypes and widths"""
    t = WindowTable()
    t.W, t.r, t.step, t.first_window = W, r, step, first_window
    t.start1 = t.end1 = np.zeros(0, dtype=np.int64)
    t.mfe_dcal = t.native_unconstrained_dcal = np.zeros(0, dtype=np.int32)
    t.mfe = t.z = t.p = t.ed = np.zeros(0, dtype=np.float64)
    t.shuffle_dcal = np.zeros((0, r), dtype=np.int32)
    t.pair_tbl = t.centroid_tbl = np.zeros((0, W), dtype=np.int16)
    return t


def table_from_result(res, first_window, step, n_regular, final_window):
    """ScanResult (raw engine arrays) -> WindowTable (reference-rounded values)"""
    t = WindowTable()
    t.W, t.r, t.step, t.first_window = res.W, res.r, step, first_window
    z, p = stats.zscore_pvalue(res.native_unconstrained_dcal, res.shuffle_dcal)
    mfe = stats.round_energy(res.mfe_dcal)
    ed = round_ed(res.ed)
    n = n_regular
    idx = first_window + np.arange(n, dtype=np.int64)
    t.start1 = idx * step + 1
    t.end1 = idx * step + res.W
    t.mfe_dcal = res.mfe_dcal[:n]
    t.mfe, t.z, t.p, t.ed = mfe[:n], z[:n], p[:n], ed[:n]
    t.native_unconstrained_dcal = res.native_unconstrained_dcal[:n]
    t.shuffle_dcal = res.shuffle_dcal[:n]
    t.pair_tbl = res.pair_tbl[:n]
    t.centroid_tbl = res.centroid_tbl[:n]
    if final_window:
        t.final = {"mfe": float(mfe[n]), "z": float(z[n]), "p": float(p[n]), "ed": float(ed[n])}
    t.ms_total, t.ms_mfe, t.n_launches = res.ms_total, res.ms_mfe, res.n_launches
    return t


def scan_record(seq, W=120, step=1, r=100, shuffle_type="mono", seed=42, parity_shuffles=None, temperature=37.0,
                max_span=0, hc=None, react=None, shape_m=0.8, shape_b=-0.2, first_window=0, n_windows=None,
                final_window=None, want_pf=True, background_temperature=None, pairprob=None):
    """Scan one record (or the window range [first_window, first_window + n_windows) of it).

    seq: RNA string (T already transcribed, ScanFold.py:282).  hc: line 3 of --constraints (one char per
    nt) or None.  react: 1-based reactivity list (index 0 unused, -999 = missing) or None.
    final_window: evaluate the extra final-window set; default = this shard holds the last window.
    pairprob: an engine.PairProbTable whose range holds these windows; every part of the scan adds its windows' pair
    probabilities to it.
    """
    L = len(seq)
    total = n_windows_of(L, W, step)
    if total == 0:
        raise ValueError("record shorter than the window")
    if n_windows is None:
        n_windows = total - first_window
    if final_window is None:
        final_window = first_window + n_windows == total
    kw = dict(shuffle_type=shuffle_type, seed=seed, temperature=temperature, max_span=max_span, hc=hc, react=react,
              shape_m=shape_m, shape_b=shape_b, want_pf=want_pf, background_temperature=background_temperature,
              pairprob=pairprob)
    if n_windows <= PIPELINE_WINDOWS:
        res = engine.scan(seq, W, step, r, parity_shuffles=parity_shuffles, first_window=first_window,
                          n_windows=n_windows, final_window=final_window, **kw)
        return table_from_result(res, first_window, step, n_windows, final_window)
    # Long shards go through the engine in parts of PIPELINE_WINDOWS windows: while the GPU folds part k+1 (the ctypes
    # call releases the GIL) a worker thread turns part k into its table (z / p statistics, rounding).  Philox shuffles are
    # keyed by the absolute window index, so the result does not depend on the split.
    from concurrent.futures import ThreadPoolExecutor
    tables, fut, done = [], None, 0
    with ThreadPoolExecutor(max_workers=1) as pool:
        while done < n_windows:
            n = min(PIPELINE_WINDOWS, n_windows - done)
            fin = bool(final_window) and done + n == n_windows
            par = None if parity_shuffles is None else parity_shuffles[done:done + n + (1 if fin else 0)]
            res = engine.scan(seq, W, step, r, parity_shuffles=par, first_window=first_window + done, n_windows=n,
                              final_window=fin, **kw)
            if fut is not None:
                tables.append(fut.result())
            fut = pool.submit(table_from_result, res, first_window + done, step, n, fin)
            done += n
        tables.append(fut.result())
    return concat_tables(tables)


PIPELINE_WINDOWS = 32768


def concat_tables(tables):
    """window tables of consecutive parts of one shard -> one table"""
    t = WindowTable()
    a = tables[0]
    t.W, t.r, t.step, t.first_window = a.W, a.r, a.step, a.first_window
    for f in ("start1", "end1", "mfe_dcal", "mfe", "z", "p", "ed", "native_unconstrained_dcal", "shuffle_dcal",
              "pair_tbl", "centroid_tbl"):
        setattr(t, f, np.concatenate([getattr(x, f) for x in tables]))
    t.final = tables[-1].final
    t.ms_total = sum(x.ms_total for x in tables)
    t.ms_mfe = sum(x.ms_mfe for x in tables)
    t.n_launches = sum(x.n_launches for x in tables)
    return t
