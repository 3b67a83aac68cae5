"""Test-side restatement of the reference's window loop over the CPU oracle: what engine.scan must return.

scan_ref() follows the reference call for call (ScanFold.py:494-544 per window, :694-757 final-window block,
ScanFoldFunctions.py:774-789 rna_folder) with the quirks of SURVEY Appendix B, and is written from those rules only:
  * the native fold compound carries md.temperature and max_bp_span; with a constraint line it gets the window's slice
    of it (hc_add_from_db), otherwise with reactivities it gets the Deigan terms of the slice react[start:end+1]
    (1-based start = i+1, end = i+W), which ViennaRNA reads 1-based: window position p sees react[i+1+p], position W
    reads past the slice and counts as missing (Q7).  --constraints wins over --react (branch order of :508-519);
  * in the reactivity branch pf() / centroid / ED run before the soft constraints are added (Q6);
  * energy_list = rna_folder(frag): a fresh md with only the background temperature -- no hard or soft constraints, no
    span -- folds the native window (energy_list[0]) and its r shuffles;
  * the final-window block (Q5) calls mfe() and pf() again on the STALE fold compound of the last regular window (so its
    pf() sees that window's soft constraints), while its rna_folder call gets seq[L-W:L] and that fragment's shuffles.
Shuffles are the caller's parity shuffles (engine.scan's parity mode), so every field is deterministic.

Oracle calls are cached per (fragment, arguments); energy-only folds go through oracle.fold_batch(fast=True), one call
per temperature (the oracle's temperature is global state)."""
import os
import types

import numpy as np

FIELDS = ("mfe_dcal", "native_unconstrained_dcal", "shuffle_dcal", "pair_tbl", "centroid_tbl", "ed", "ensemble_dG")


def pt_from_db(db):
    """dot-bracket -> int16 pair table (1-based partner, 0 unpaired), the layout of engine.scan's pair_tbl"""
    pt = np.zeros(len(db), dtype=np.int16)
    stack = []
    for k, ch in enumerate(db):
        if ch == "(":
            stack.append(k)
        elif ch == ")":
            i = stack.pop()
            pt[i], pt[k] = k + 1, i + 1
    return pt


def react_slice_stack(react, i, W, m, b):
    """Deigan stacking terms (1-based, [W+1]) the native fold of the window starting at 0-based i sees (Q7)"""
    from oracle import oracle as O
    src = list(react[i + 1:i + W + 1])          # reactivities[start:end+1] with start = i + 1, end = i + W
    r1 = np.full(W + 1, -999.0)
    for p in range(1, W + 1):
        if p < len(src):
            r1[p] = float(src[p])
    return O.deigan(r1, m, b)


class OracleCache:
    """memoised oracle calls; energy-only folds are collected and run in one fold_batch per temperature"""

    def __init__(self, n_threads=None):
        self.n_threads = n_threads or os.cpu_count() or 1
        self._mfe, self._pf, self._energy = {}, {}, {}

    def mfe(self, frag, hc, sc, span, T):
        from oracle import oracle as O
        key = (frag, hc, None if sc is None else bytes(np.asarray(sc, dtype=np.int32)), span, T)
        if key not in self._mfe:
            self._mfe[key] = O.mfe(frag, hc=hc, sc_stack=sc, max_span=span, temperature=T)
        return self._mfe[key]

    def pf(self, frag, hc, sc, span, T):
        from oracle import oracle as O
        key = (frag, hc, None if sc is None else bytes(np.asarray(sc, dtype=np.int32)), span, T)
        if key not in self._pf:
            self._pf[key] = O.pf(frag, hc=hc, sc_stack=sc, max_span=span, temperature=T)
        return self._pf[key]

    def energies(self, frags, T):
        """energy-only MFE (md with the temperature only) of equal-length fragments"""
        from oracle import oracle as O
        todo = sorted({f for f in frags if (f, T) not in self._energy})
        if todo:
            a = np.frombuffer("".join(todo).encode(), dtype=np.uint8).reshape(len(todo), len(todo[0]))
            e = O.fold_batch(a, n_threads=self.n_threads, fast=True, temperature=T)
            O.set_temperature(37.0)
            self._energy.update({(f, T): int(x) for f, x in zip(todo, e)})
        return [self._energy[(f, T)] for f in frags]


def scan_ref(seq, W, step, r, parity_shuffles, hc=None, react=None, shape_m=0.8, shape_b=-0.2, temperature=37,
             max_span=0, background_temperature=None, first_window=0, n_windows=None, final_window=True, cache=None):
    """The per-window outputs of one shard [first_window, first_window + n_windows) (+ the final-window slot), the same
    fields and dtypes as engine.scan.  parity_shuffles: [(n_windows + final) * r * W] ASCII bytes of this shard's
    shuffles, as engine.scan takes them.  hc: the record's constraint line (shorter lines are padded with '.');
    react: 1-based reactivities of the record (index 0 unused, -999 missing)."""
    cache = cache or OracleCache()
    L = len(seq)
    total = (L - W) // step + 1
    if n_windows is None:
        n_windows = total - first_window
    T = float(temperature)
    T_bg = float(background_temperature) if background_temperature else T
    span = int(max_span or 0)
    n = n_windows + (1 if final_window else 0)
    shuf = np.asarray(parity_shuffles, dtype=np.uint8).reshape(n, r, W)
    if hc is not None:
        hc = hc.rstrip("\n")
    if react is not None:
        react = list(react)

    out = types.SimpleNamespace(W=W, r=r, n=n)
    out.mfe_dcal = np.zeros(n, dtype=np.int32)
    out.native_unconstrained_dcal = np.zeros(n, dtype=np.int32)
    out.shuffle_dcal = np.zeros((n, r), dtype=np.int32)
    out.pair_tbl = np.zeros((n, W), dtype=np.int16)
    out.centroid_tbl = np.zeros((n, W), dtype=np.int16)
    out.ed = np.zeros(n)
    out.ensemble_dG = np.zeros(n)

    def native(i):
        """(mfe, structure, pf dict) of the regular window starting at i, and the pf() a later call on the same
        (now stale) fold compound returns"""
        frag = seq[i:i + W]
        if hc is not None:                                      # ScanFold.py:508-519
            h = hc[i:i + W]
            h = h + "." * (W - len(h))
            e, s = cache.mfe(frag, h, None, span, T)
            p = cache.pf(frag, h, None, span, T)
            return e, s, p, p
        if react is not None:                                   # :522-541, pf() before sc (Q6)
            p = cache.pf(frag, None, None, span, T)
            sc = react_slice_stack(react, i, W, shape_m, shape_b)
            e, s = cache.mfe(frag, None, sc, span, T)
            return e, s, p, cache.pf(frag, None, sc, span, T)
        e, s = cache.mfe(frag, None, None, span, T)              # :496-504
        p = cache.pf(frag, None, None, span, T)
        return e, s, p, p

    bg_frags = []
    for k in range(n):
        fin = final_window and k == n - 1
        w = first_window + k
        if fin:                                                 # Q5: stale fc of the last regular window
            e, s, _, p = native((total - 1) * step)
            frag = seq[L - W:L]
        else:
            e, s, p, _ = native(w * step)
            frag = seq[w * step:w * step + W]
        out.mfe_dcal[k] = e
        out.pair_tbl[k] = pt_from_db(s)
        out.ed[k] = p["ed"]
        out.ensemble_dG[k] = p["dG"]
        out.centroid_tbl[k] = pt_from_db(p["centroid"])
        bg_frags.append(frag)
        bg_frags += [bytes(shuf[k, j]).decode() for j in range(r)]
    e = np.asarray(cache.energies(bg_frags, T_bg), dtype=np.int32).reshape(n, r + 1)
    out.native_unconstrained_dcal[:] = e[:, 0]
    out.shuffle_dcal[:] = e[:, 1:]
    return out

