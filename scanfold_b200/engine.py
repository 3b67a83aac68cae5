"""ctypes binding of libscanfold_b200.so (include/scanfold_b200.h) -- the CUDA fold engine.

This is the only route from Python to the fold arithmetic: if the CUDA library is missing or no GPU is
present every call raises (there is no CPU fallback; the CPU oracle under oracle/ is test infrastructure
and is never imported from this package).

Replaces the ViennaRNA calls of the reference: RNA.fold_compound(...).mfe()/pf()/centroid()/
mean_bp_distance()/hc_add_from_db()/sc_add_SHAPE_deigan() (ScanFold.py:494-544) and the helper
functions scramble()/energies() (ScanFoldFunctions.py:805-851).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SFB_LIB") or os.path.join(_HERE, "libscanfold_b200.so")   # SFB_LIB: debug builds only
INF = 10000000
SHUFFLE_MONO, SHUFFLE_DI = 0, 1

EXPORTS = ["sfb_version", "sfb_init", "sfb_shutdown", "sfb_last_error", "sfb_params_besteffort", "sfb_fold_batch",
           "sfb_fold_long", "sfb_pf_batch", "sfb_deigan", "sfb_scan", "sfb_scan_plan_create", "sfb_scan_plan_keep_shuffles",
           "sfb_scan_plan_run", "sfb_scan_plan_fetch", "sfb_scan_plan_stage_ms", "sfb_scan_plan_destroy", "sfb_accumulate_begin",
           "sfb_accumulate_geometry", "sfb_accumulate_export", "sfb_accumulate_merge", "sfb_accumulate_compact",
           "sfb_accumulate_fetch", "sfb_accumulate_launches", "sfb_accumulate_free", "sfb_microbench", "sfb_set_stream", "sfb_set_engines",
           "sfb_pairprob_begin", "sfb_scan_plan_pairprob", "sfb_pairprob_export", "sfb_pairprob_merge", "sfb_pairprob_compact",
           "sfb_pairprob_fetch", "sfb_pairprob_free"]


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("scanfold_b200 engine error %d: %s" % (code, msg))
        self.code = code


class Model(C.Structure):
    _fields_ = [("temperature", C.c_double), ("max_bp_span", C.c_int32)]


class ScanArgs(C.Structure):
    _fields_ = [("seq", C.c_void_p), ("L", C.c_int32), ("W", C.c_int32), ("step", C.c_int32), ("r", C.c_int32),
                ("shuffle_type", C.c_int32), ("seed", C.c_uint64), ("parity_shuffles", C.c_void_p),
                ("model", Model), ("hc", C.c_void_p), ("react", C.c_void_p), ("shape_m", C.c_double),
                ("shape_b", C.c_double), ("first_window", C.c_int32), ("n_windows", C.c_int32),
                ("final_window", C.c_int32), ("want_pf", C.c_int32), ("background_temperature", C.c_double)]


class ScanOut(C.Structure):
    _fields_ = [("mfe_dcal", C.c_void_p), ("native_unconstrained_dcal", C.c_void_p), ("shuffle_dcal", C.c_void_p),
                ("pair_tbl", C.c_void_p), ("centroid_tbl", C.c_void_p), ("ed", C.c_void_p),
                ("ensemble_dG", C.c_void_p), ("shuffles_out", C.c_void_p)]


class AccumArgs(C.Structure):
    _fields_ = [("L", C.c_int32), ("W", C.c_int32), ("step", C.c_int32), ("first_window", C.c_int32),
                ("n_windows", C.c_int32), ("pair_tbl", C.c_void_p), ("z100", C.c_void_p), ("mfe_dcal", C.c_void_p),
                ("ed100", C.c_void_p)]


_lib = None
_initialised = None


def load_library():
    """dlopen the CUDA library; raises if it has not been built (python -m scanfold_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EngineError(-4, "libscanfold_b200.so is not built (run `python scanfold_b200/build.py`); "
                                  "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.sfb_last_error.restype = C.c_char_p
        L.sfb_init.argtypes = [C.c_int, C.c_char_p]
        L.sfb_fold_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(Model), C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]
        L.sfb_fold_long.argtypes = [C.c_void_p, C.c_int, C.POINTER(Model), C.c_void_p, C.c_void_p, C.c_void_p]
        L.sfb_pf_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(Model), C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sfb_deigan.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p]
        L.sfb_scan.argtypes = [C.POINTER(ScanArgs), C.POINTER(ScanOut)]
        L.sfb_scan_plan_create.argtypes = [C.POINTER(ScanArgs), C.POINTER(C.c_void_p)]
        L.sfb_scan_plan_keep_shuffles.argtypes = [C.c_void_p]
        L.sfb_scan_plan_keep_shuffles.restype = None
        L.sfb_scan_plan_run.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int32)]
        L.sfb_scan_plan_fetch.argtypes = [C.c_void_p, C.POINTER(ScanOut)]
        L.sfb_scan_plan_stage_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.sfb_scan_plan_destroy.argtypes = [C.c_void_p]
        L.sfb_scan_plan_destroy.restype = None
        L.sfb_accumulate_begin.argtypes = [C.POINTER(AccumArgs), C.POINTER(C.c_void_p)]
        L.sfb_accumulate_geometry.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.sfb_accumulate_export.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sfb_accumulate_merge.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sfb_accumulate_compact.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int64)]
        L.sfb_accumulate_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sfb_accumulate_launches.argtypes = [C.c_void_p]
        L.sfb_accumulate_free.argtypes = [C.c_void_p]
        L.sfb_accumulate_free.restype = None
        L.sfb_pairprob_begin.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
        L.sfb_scan_plan_pairprob.argtypes = [C.c_void_p, C.c_void_p]
        L.sfb_pairprob_export.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.sfb_pairprob_merge.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.sfb_pairprob_compact.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int64)]
        L.sfb_pairprob_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sfb_pairprob_free.argtypes = [C.c_void_p]
        L.sfb_pairprob_free.restype = None
        L.sfb_shutdown.restype = None
        L.sfb_set_stream.argtypes = [C.c_void_p]
        L.sfb_set_engines.argtypes = [C.c_int, C.c_int]
        L.sfb_microbench.argtypes = [C.c_int, C.POINTER(C.c_double)]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise EngineError(rc, load_library().sfb_last_error().decode())


def init(device=0, params=None):
    """Load the energy tables and bind this process to one GPU (one context per process)."""
    global _initialised
    L = load_library()
    params = params or os.environ.get("SCANFOLD_PARAMS") or None
    _check(L.sfb_init(int(device), os.fsencode(params) if params else None))
    _initialised = (int(device), params)


def ensure_init(device=None):
    if _initialised is None:
        init(int(os.environ.get("LOCAL_RANK", "0")) if device is None else device)


def shutdown():
    global _initialised
    if _lib is not None:
        _lib.sfb_shutdown()
    _initialised = None


def params_besteffort():
    return bool(load_library().sfb_params_besteffort())


def _as_seq_matrix(seqs):
    """list of equal-length strings / bytes, or a uint8 [n,len] array -> contiguous uint8 matrix"""
    if isinstance(seqs, np.ndarray):
        a = np.ascontiguousarray(seqs, dtype=np.uint8)
        if a.ndim != 2:
            raise ValueError("sequence array must be [n, len]")
        return a
    seqs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    if not seqs:
        return np.zeros((0, 1), dtype=np.uint8)
    n = len(seqs[0])
    if any(len(s) != n for s in seqs):
        raise ValueError("all sequences of a batch must have the same length")
    return np.frombuffer(b"".join(seqs), dtype=np.uint8).reshape(len(seqs), n).copy()


def _model(temperature, max_span):
    return Model(float(temperature), int(max_span or 0))


def pair_table_to_dotbracket(pt):
    """int16 pair table (1-based partner, 0 unpaired) -> dot-bracket string"""
    idx = np.arange(1, len(pt) + 1)
    out = np.full(len(pt), ord("."), dtype=np.uint8)
    out[pt > idx] = ord("(")
    out[(pt > 0) & (pt < idx)] = ord(")")
    return out.tobytes().decode()


def pair_tables_to_dotbrackets(tbl):
    """[n, W] int16 pair tables -> list of n dot-bracket strings (one vectorised pass)"""
    tbl = np.asarray(tbl)
    n, W = tbl.shape
    idx = np.arange(1, W + 1, dtype=tbl.dtype)[None, :]
    out = np.full((n, W), ord("."), dtype=np.uint8)
    out[tbl > idx] = ord("(")
    out[(tbl > 0) & (tbl < idx)] = ord(")")
    text = out.tobytes().decode()
    return [text[k * W:(k + 1) * W] for k in range(n)]


def fold_batch(seqs, hc=None, sc=None, structure=False, temperature=37.0, max_span=0):
    """MFE of equal-length sequences.  -> (int32 energies in dcal, int16 pair tables or None)."""
    ensure_init()
    a = _as_seq_matrix(seqs)
    n, ln = a.shape
    e = np.zeros(n, dtype=np.int32)
    pt = np.zeros((n, ln), dtype=np.int16) if structure else None
    hcm = _as_seq_matrix(hc) if hc is not None else None
    scm = np.ascontiguousarray(sc, dtype=np.int32) if sc is not None else None
    if hcm is not None and hcm.shape != a.shape:
        raise ValueError("hc must match the sequence batch shape")
    if scm is not None and scm.shape != (n, ln + 1):
        raise ValueError("sc must be [n, len+1] (1-based)")
    m = _model(temperature, max_span)
    _check(load_library().sfb_fold_batch(a.ctypes.data, n, ln, C.byref(m), hcm.ctypes.data if hcm is not None else None,
                                         scm.ctypes.data if scm is not None else None, e.ctypes.data,
                                         pt.ctypes.data if structure else None))
    return e, pt


def fold_long(seq, hc=None, temperature=37.0, max_span=0):
    """MFE and structure of one whole sequence (the full-length folds of --global_refold, ScanFold.py:1518-1539) on the
    blocked kernel.  hc: constraint line (shorter lines are padded with '.') or None.  -> (energy dcal, int32 pair table)."""
    ensure_init()
    a = np.frombuffer(seq.encode() if isinstance(seq, str) else bytes(seq), dtype=np.uint8).copy()
    n = len(a)
    h = None
    if hc is not None:
        hb = (hc.encode() if isinstance(hc, str) else bytes(hc))[:n]
        h = np.frombuffer(hb + b"." * (n - len(hb)), dtype=np.uint8).copy()
    e = np.zeros(1, dtype=np.int32)
    pt = np.zeros(n, dtype=np.int32)
    m = _model(temperature, max_span)
    _check(load_library().sfb_fold_long(a.ctypes.data, n, C.byref(m), h.ctypes.data if h is not None else None,
                                        e.ctypes.data, pt.ctypes.data))
    return int(e[0]), pt


def pf_batch(seqs, hc=None, sc=None, want_bpp=False, temperature=37.0, max_span=0):
    """Partition function of equal-length sequences -> dict(dG, ed, centroid (pair tables), bpp)."""
    ensure_init()
    a = _as_seq_matrix(seqs)
    n, ln = a.shape
    dG = np.zeros(n)
    ed = np.zeros(n)
    cen = np.zeros((n, ln), dtype=np.int16)
    bpp = np.zeros((n, ln, ln)) if want_bpp else None
    hcm = _as_seq_matrix(hc) if hc is not None else None
    scm = np.ascontiguousarray(sc, dtype=np.int32) if sc is not None else None
    m = _model(temperature, max_span)
    _check(load_library().sfb_pf_batch(a.ctypes.data, n, ln, C.byref(m), hcm.ctypes.data if hcm is not None else None,
                                       scm.ctypes.data if scm is not None else None, dG.ctypes.data, ed.ctypes.data,
                                       cen.ctypes.data, bpp.ctypes.data if want_bpp else None))
    return {"dG": dG, "ed": ed, "centroid": cen, "bpp": bpp}


def deigan(react1, m, b):
    r = np.ascontiguousarray(react1, dtype=np.float64)
    out = np.zeros(len(r), dtype=np.int32)
    _check(load_library().sfb_deigan(r.ctypes.data, len(r) - 1, float(m), float(b), out.ctypes.data))
    return out


class ScanResult:
    """Per-window arrays of one shard; slot n_windows is the extra final-window set when requested."""
    __slots__ = ("W", "r", "n", "mfe_dcal", "native_unconstrained_dcal", "shuffle_dcal", "pair_tbl", "centroid_tbl",
                 "ed", "ensemble_dG", "shuffles", "ms_total", "ms_mfe", "n_launches")


class ScanPlan:
    """Device-resident scan of one record shard (sfb_scan_plan_*)."""

    def __init__(self, seq, W, step, r, shuffle_type="mono", seed=42, parity_shuffles=None, temperature=37.0,
                 max_span=0, hc=None, react=None, shape_m=0.8, shape_b=-0.2, first_window=0, n_windows=None,
                 final_window=True, want_pf=True, keep_shuffles=False, background_temperature=None, pairprob=None):
        ensure_init()
        self._lib = load_library()
        self._seq = np.frombuffer(seq.encode() if isinstance(seq, str) else bytes(seq), dtype=np.uint8).copy()
        L = len(self._seq)
        total = (L - W) // step + 1 if L >= W else 0
        if n_windows is None:
            n_windows = total - first_window
        self.W, self.r, self.step, self.L = W, r, step, L
        self.n_windows = n_windows
        self.n = n_windows + (1 if final_window else 0)
        self._hc = np.frombuffer(hc.encode() if isinstance(hc, str) else bytes(hc), dtype=np.uint8).copy() \
            if hc is not None else None
        if self._hc is not None and len(self._hc) < L:
            self._hc = np.concatenate([self._hc, np.full(L - len(self._hc), ord("."), dtype=np.uint8)])
        self._react = None
        if react is not None:
            rr = np.full(L + 1, -999.0)
            src = np.asarray(react, dtype=np.float64)[:L + 1]
            rr[:len(src)] = src
            self._react = rr
        self._parity = None
        if parity_shuffles is not None:
            p = np.ascontiguousarray(parity_shuffles, dtype=np.uint8)
            if p.size != self.n * r * W:
                raise ValueError("parity_shuffles must hold (n_windows+final)*r*W bytes")
            self._parity = p
        a = ScanArgs()
        a.seq = self._seq.ctypes.data
        a.L, a.W, a.step, a.r = L, W, step, r
        a.shuffle_type = SHUFFLE_DI if shuffle_type == "di" else SHUFFLE_MONO
        a.seed = int(seed)
        a.parity_shuffles = self._parity.ctypes.data if self._parity is not None else None
        a.model = _model(temperature, max_span)
        a.hc = self._hc.ctypes.data if self._hc is not None else None
        a.react = self._react.ctypes.data if self._react is not None else None
        a.shape_m, a.shape_b = float(shape_m), float(shape_b)
        a.first_window, a.n_windows = int(first_window), int(n_windows)
        a.final_window = 1 if final_window else 0
        a.want_pf = 1 if want_pf else 0
        a.background_temperature = float(background_temperature) if background_temperature else 0.0
        self._args = a
        self._plan = C.c_void_p()
        _check(self._lib.sfb_scan_plan_create(C.byref(a), C.byref(self._plan)))
        self._keep = keep_shuffles
        if keep_shuffles:
            self._lib.sfb_scan_plan_keep_shuffles(self._plan)
        if pairprob is not None:
            self.attach_pairprob(pairprob)
        self.ms_total = self.ms_mfe = 0.0
        self.n_launches = 0

    def attach_pairprob(self, table):
        """every later run() adds the pair probabilities of this plan's regular windows to `table` (a PairProbTable)"""
        _check(self._lib.sfb_scan_plan_pairprob(self._plan, table._h))
        self._pairprob = table      # the table must outlive the plan's runs

    def run(self):
        ms_t, ms_m, nl = C.c_float(), C.c_float(), C.c_int32()
        _check(self._lib.sfb_scan_plan_run(self._plan, C.byref(ms_t), C.byref(ms_m), C.byref(nl)))
        self.ms_total, self.ms_mfe, self.n_launches = ms_t.value, ms_m.value, nl.value
        st = (C.c_float * 4)()
        _check(self._lib.sfb_scan_plan_stage_ms(self._plan, st))
        self.stage_ms = {"shuffle": st[0], "mfe": st[1], "pf": st[2], "other": st[3]}
        return self

    def fetch(self):
        n, W, r = self.n, self.W, self.r
        res = ScanResult()
        res.W, res.r, res.n = W, r, n
        res.mfe_dcal = np.zeros(n, dtype=np.int32)
        res.native_unconstrained_dcal = np.zeros(n, dtype=np.int32)
        res.shuffle_dcal = np.zeros((n, r), dtype=np.int32)
        res.pair_tbl = np.zeros((n, W), dtype=np.int16)
        res.centroid_tbl = np.zeros((n, W), dtype=np.int16)
        res.ed = np.zeros(n)
        res.ensemble_dG = np.zeros(n)
        res.shuffles = np.zeros((n, r, W), dtype=np.uint8) if self._keep else None
        o = ScanOut(res.mfe_dcal.ctypes.data, res.native_unconstrained_dcal.ctypes.data, res.shuffle_dcal.ctypes.data,
                    res.pair_tbl.ctypes.data, res.centroid_tbl.ctypes.data, res.ed.ctypes.data,
                    res.ensemble_dG.ctypes.data, res.shuffles.ctypes.data if self._keep else None)
        _check(self._lib.sfb_scan_plan_fetch(self._plan, C.byref(o)))
        res.ms_total, res.ms_mfe, res.n_launches = self.ms_total, self.ms_mfe, self.n_launches
        return res

    def close(self):
        if self._plan:
            self._lib.sfb_scan_plan_destroy(self._plan)
            self._plan = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scan(seq, W, step, r, **kw):
    """Host-buffer scan of one record shard: upload, run, download (sfb_scan semantics)."""
    plan = ScanPlan(seq, W, step, r, **kw)
    try:
        return plan.run().fetch()
    finally:
        plan.close()


class Accumulator:
    """Device-resident ScanFold-Fold accumulators of one shard of windows (sfb_accumulate_*).

    rows = nucleotides [nt0, nt0 + n_nt) touched by the shard, 0-based; 2W-1 partner-offset columns.
    export()/merge() move halo rows through caller-provided DEVICE buffers (multi-GPU exchange);
    compact() returns the per-nucleotide partner lists as numpy arrays."""

    def __init__(self, L, W, step, first_window, pair_tbl, z100, mfe_dcal, ed100, skip=None):
        ensure_init()
        self._lib = load_library()
        pt = np.ascontiguousarray(pair_tbl, dtype=np.int16)
        if skip is not None and np.any(skip):          # windows that leave no pair records (all-N, Appendix B Q10)
            pt = pt.copy()
            pt[np.asarray(skip, dtype=bool)] = -1
        z = np.ascontiguousarray(z100, dtype=np.int32)
        m = np.ascontiguousarray(mfe_dcal, dtype=np.int32)
        e = np.ascontiguousarray(ed100, dtype=np.int32)
        n = pt.shape[0]
        if not (len(z) == len(m) == len(e) == n):
            raise ValueError("per-window arrays must have one entry per pair-table row")
        a = AccumArgs(L, W, step, first_window, n, pt.ctypes.data, z.ctypes.data, m.ctypes.data, e.ctypes.data)
        self._h = C.c_void_p()
        _check(self._lib.sfb_accumulate_begin(C.byref(a), C.byref(self._h)))
        nt0, n_nt = C.c_int32(), C.c_int32()
        _check(self._lib.sfb_accumulate_geometry(self._h, C.byref(nt0), C.byref(n_nt)))
        self.W, self.step, self.nt0, self.n_nt, self.ncol = W, step, nt0.value, n_nt.value, 2 * W - 1

    def export_rows(self, row0, n_rows, d_count, d_first, d_sums):
        """device pointers (ints) of buffers sized n_rows*(2W-1) int32 / int32 / 6x int64"""
        _check(self._lib.sfb_accumulate_export(self._h, row0, n_rows, d_count, d_first, d_sums))

    def merge_rows(self, row0, n_rows, d_count, d_first, d_sums):
        _check(self._lib.sfb_accumulate_merge(self._h, row0, n_rows, d_count, d_first, d_sums))

    # ---- torch views of the halo rows (multi-GPU exchange over NCCL, scanfold_b200.multigpu)
    def empty_tensors(self, n_rows):
        import torch
        n = n_rows * self.ncol
        return (torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda"),
                torch.empty(6 * n, dtype=torch.int64, device="cuda"))

    def export_tensors(self, row0, n_rows):
        t = self.empty_tensors(n_rows)
        self.export_rows(row0, n_rows, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr())
        return t

    def merge_tensors(self, row0, n_rows, count, first, sums):
        self.merge_rows(row0, n_rows, count.data_ptr(), first.data_ptr(), sums.data_ptr())

    def compact(self, row0=0, n_rows=None):
        """-> (nparts [n_rows], partner, count, first_seen [M], sums [6, M]); entries in column order per nucleotide"""
        if n_rows is None:
            n_rows = self.n_nt - row0
        m = C.c_int64()
        _check(self._lib.sfb_accumulate_compact(self._h, row0, n_rows, C.byref(m)))
        M = m.value
        nparts = np.zeros(max(n_rows, 1), dtype=np.int32)
        partner = np.zeros(max(M, 1), dtype=np.int32)
        count = np.zeros(max(M, 1), dtype=np.int32)
        first = np.zeros(max(M, 1), dtype=np.int32)
        sums = np.zeros((6, max(M, 1)), dtype=np.int64)
        _check(self._lib.sfb_accumulate_fetch(self._h, nparts.ctypes.data, partner.ctypes.data, count.ctypes.data,
                                              first.ctypes.data, sums.ctypes.data))
        return nparts[:n_rows], partner[:M], count[:M], first[:M], sums[:, :M]

    @property
    def n_launches(self):
        return self._lib.sfb_accumulate_launches(self._h)

    def close(self):
        if self._h:
            self._lib.sfb_accumulate_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


PAIR_CUTOFF = 0.01     # pairs listed by --pair_probs (RNAplfold's -c default is 0.01 too)


def windows_holding(i, j, W, step, n_windows):
    """number of regular windows w in [0, n_windows) with w*step <= i and j < w*step + W (0-based, i <= j; arrays work)"""
    i, j = np.asarray(i, dtype=np.int64), np.asarray(j, dtype=np.int64)
    lo = np.where(j - W + 1 <= 0, 0, (j - W + 1 + step - 1) // step)
    hi = np.minimum(i // step, n_windows - 1)
    return np.maximum(hi - lo + 1, 0)


class PairProbTable:
    """Device-resident window-averaged base-pair probabilities of one shard of windows (sfb_pairprob_*).

    rows = nucleotides [nt0, nt0 + n_nt) touched by the shard, 0-based; W int64 columns of exact fixed-point sums
    (column 0: paired, d >= 1: pair (i, i+d)).  Attach it to the scan (scan.scan_record(..., pairprob=table)), move halo
    rows with export_tensors() / merge_tensors() (multigpu.exchange_halo), then reduce() the rows this shard owns."""

    def __init__(self, L, W, step, first_window, n_windows):
        ensure_init()
        self._lib = load_library()
        self._h = C.c_void_p()
        _check(self._lib.sfb_pairprob_begin(int(L), int(W), int(step), int(first_window), int(n_windows), C.byref(self._h)))
        self.L, self.W, self.step = L, W, step
        self.nt0, self.n_nt = first_window * step, (n_windows - 1) * step + W

    def export_rows(self, row0, n_rows, d_rows):
        _check(self._lib.sfb_pairprob_export(self._h, row0, n_rows, d_rows))

    def merge_rows(self, row0, n_rows, d_rows):
        _check(self._lib.sfb_pairprob_merge(self._h, row0, n_rows, d_rows))

    # ---- torch views of the halo rows (multi-GPU exchange over NCCL, scanfold_b200.multigpu)
    def empty_tensors(self, n_rows):
        import torch
        return (torch.empty(n_rows * self.W, dtype=torch.int64, device="cuda"),)

    def export_tensors(self, row0, n_rows):
        t = self.empty_tensors(n_rows)
        self.export_rows(row0, n_rows, t[0].data_ptr())
        return t

    def merge_tensors(self, row0, n_rows, rows):
        self.merge_rows(row0, n_rows, rows.data_ptr())

    def rows(self, row0=0, n_rows=None):
        """the raw int64 sums of rows [row0, row0 + n_rows) as a numpy [n_rows, W] array (tests)"""
        n_rows = self.n_nt - row0 if n_rows is None else n_rows
        t = self.export_tensors(row0, n_rows)[0]
        return t.cpu().numpy().reshape(n_rows, self.W)

    def reduce(self, row0=0, n_rows=None, cutoff=PAIR_CUTOFF):
        """-> (paired [n_rows] float64, i, j [M] int32 1-based, p [M] float64): the pairs with P >= cutoff, by i then j"""
        if n_rows is None:
            n_rows = self.n_nt - row0
        m = C.c_int64()
        _check(self._lib.sfb_pairprob_compact(self._h, row0, n_rows, float(cutoff), C.byref(m)))
        M = m.value
        paired = np.zeros(max(n_rows, 1))
        i, j = np.zeros(max(M, 1), dtype=np.int32), np.zeros(max(M, 1), dtype=np.int32)
        p = np.zeros(max(M, 1))
        _check(self._lib.sfb_pairprob_fetch(self._h, paired.ctypes.data, i.ctypes.data, j.ctypes.data, p.ctypes.data))
        return paired[:n_rows], i[:M], j[:M], p[:M]

    def close(self):
        if self._h:
            self._lib.sfb_pairprob_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def microbench(which):
    """Measured device peak: which=0 int32 add-min ops/s, which=1 32-bit shared-memory loads/s, which=2 fp64 FMA/s."""
    ensure_init()
    v = C.c_double()
    _check(load_library().sfb_microbench(int(which), C.byref(v)))
    return v.value


def set_stream(cuda_stream):
    """Route every launch and copy of the library to `cuda_stream` (int handle, e.g. torch's current stream)."""
    ensure_init()
    _check(load_library().sfb_set_stream(C.c_void_p(int(cuda_stream)) if cuda_stream else None))


def set_engines(mfe=0, pf=0):
    """Kernel generations allowed to run (tests / tuning; results never depend on it): mfe 1 = int32 CTA kernel,
    2 = + int16 warp-team kernel, 3 = + int16 CTA kernel with stencil / range-minimum loops (default);
    pf 1 = global-memory kernel, 2 = + shared-memory kernel (default).  0 leaves a setting unchanged."""
    _check(load_library().sfb_set_engines(int(mfe), int(pf)))
