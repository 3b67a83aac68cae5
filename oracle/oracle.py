"""ctypes binding of the CPU ORACLE (oracle/sf_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module.  The product package scanfold_b200/ never does.  PARITY UNPINNED (see sf_oracle.h).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libsf_oracle.so")
DEFAULT_PAR = os.path.join(_HERE, "..", "scanfold_b200", "params", "rna_turner2004_besteffort.par")
INF = 10000000

_lib = None


def build():
    """Compile the oracle with gcc (oracle/Makefile)."""
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        L.sfo_load_params.argtypes = [C.c_char_p]
        L.sfo_last_error.restype = C.c_char_p
        L.sfo_set_temperature.argtypes = [C.c_double]
        L.sfo_mfe.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_void_p, C.c_int, C.c_char_p]
        L.sfo_eval.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_void_p]
        L.sfo_pf.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_void_p, C.c_int, C.c_double,
                             C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p]
        L.sfo_pf_scaled.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_void_p, C.c_int, C.c_double, C.c_double,
                                    C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p]
        L.sfo_deigan.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p]
        L.sfo_fold_batch.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.sfo_fold_batch_fast.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.sfo_pf_batch.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.sfo_eval_weight.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_double]
        L.sfo_eval_weight.restype = C.c_double
        L.sfo_counters.argtypes = [C.c_void_p, C.c_void_p]
        _lib = L
        load_params(DEFAULT_PAR)
    return _lib


def load_params(path):
    L = _lib if _lib is not None else lib()
    if L.sfo_load_params(os.fsencode(path)) != 0:
        raise RuntimeError("oracle: " + L.sfo_last_error().decode())


def _sc_ptr(sc_stack):
    if sc_stack is None:
        return None, None
    a = np.ascontiguousarray(sc_stack, dtype=np.int32)
    return a, a.ctypes.data


def set_temperature(temperature):
    """md.temperature for every later call (tables rescaled from the 37 C values and the enthalpies)"""
    if lib().sfo_set_temperature(float(temperature)) != 0:
        raise RuntimeError("oracle: " + lib().sfo_last_error().decode())


def mfe(seq, hc=None, sc_stack=None, max_span=0, structure=True, temperature=37.0):
    """-> (energy_dcal, dot-bracket or None).  sc_stack: 1-based int array of length n+1."""
    L = lib()
    set_temperature(temperature)
    n = len(seq)
    buf = C.create_string_buffer(n + 1) if structure else None
    keep, scp = _sc_ptr(sc_stack)
    e = L.sfo_mfe(seq.encode(), n, hc.encode() if hc else None, scp, int(max_span or 0), buf)
    if e >= INF:
        raise RuntimeError("oracle mfe: " + L.sfo_last_error().decode())
    return e, (buf.value.decode() if structure else None)


def eval_structure(seq, structure, sc_stack=None):
    keep, scp = _sc_ptr(sc_stack)
    return lib().sfo_eval(seq.encode(), len(seq), structure.encode(), scp)


def pf(seq, hc=None, sc_stack=None, max_span=0, temperature=37.0, want_bpp=False, pf_scale=None):
    """-> dict(dG, ed, centroid, bpp).  pf_scale None: the tables' per-nucleotide scale, and exp(-1.07 mfe / (kT n)) where
    Z leaves the fp64 range with it; a number forces that scale (0: the tables') and raises if Z leaves the range."""
    L = lib()
    n = len(seq)
    dG = C.c_double()
    ed = C.c_double()
    cen = C.create_string_buffer(n + 1)
    bpp = np.zeros((n, n), dtype=np.float64) if want_bpp else None
    keep, scp = _sc_ptr(sc_stack)
    args = (C.addressof(dG), C.addressof(ed), cen, bpp.ctypes.data if want_bpp else None)
    if pf_scale is None:
        rc = L.sfo_pf(seq.encode(), n, hc.encode() if hc else None, scp, int(max_span or 0), float(temperature), *args)
    else:
        rc = L.sfo_pf_scaled(seq.encode(), n, hc.encode() if hc else None, scp, int(max_span or 0), float(temperature),
                             float(pf_scale), *args)
    if rc != 0:
        raise RuntimeError("oracle pf: " + L.sfo_last_error().decode())
    return {"dG": dG.value, "ed": ed.value, "centroid": cen.value.decode(), "bpp": bpp}


def eval_weight(seq, structure, temperature=37.0):
    return lib().sfo_eval_weight(seq.encode(), len(seq), structure.encode(), float(temperature))


def deigan(react1, m, b):
    """react1: 1-based float array (index 0 ignored) -> 1-based int32 array of stacking pseudo-energies."""
    r = np.ascontiguousarray(react1, dtype=np.float64)
    n = len(r) - 1
    out = np.zeros(n + 1, dtype=np.int32)
    lib().sfo_deigan(r.ctypes.data, n, float(m), float(b), out.ctypes.data)
    return out


def fold_batch(seqs, n_threads=1, fast=False, temperature=37.0):
    """seqs: uint8/bytes array [n_seq, len] of ASCII -> int32 energies (dcal).  fast: the tuned CPU path."""
    set_temperature(temperature)
    a = np.ascontiguousarray(seqs, dtype=np.uint8)
    n_seq, ln = a.shape
    out = np.zeros(n_seq, dtype=np.int32)
    fn = lib().sfo_fold_batch_fast if fast else lib().sfo_fold_batch
    if fn(a.tobytes(), n_seq, ln, out.ctypes.data, int(n_threads)) != 0:
        raise RuntimeError("oracle fold_batch: " + lib().sfo_last_error().decode())
    return out


def pf_batch(seqs, n_threads=1):
    set_temperature(37.0)
    a = np.ascontiguousarray(seqs, dtype=np.uint8)
    n_seq, ln = a.shape
    ed = np.zeros(n_seq, dtype=np.float64)
    dG = np.zeros(n_seq, dtype=np.float64)
    cen = np.zeros((n_seq, ln + 1), dtype=np.uint8)
    if lib().sfo_pf_batch(a.tobytes(), n_seq, ln, ed.ctypes.data, dG.ctypes.data, cen.ctypes.data, int(n_threads)) != 0:
        raise RuntimeError("oracle pf_batch: " + lib().sfo_last_error().decode())
    return ed, dG, [bytes(c[:ln]).decode() for c in cen]


def counters():
    d = C.c_longlong()
    u = C.c_longlong()
    lib().sfo_counters(C.addressof(d), C.addressof(u))
    return d.value, u.value
