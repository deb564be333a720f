"""Banded global alignment on the CPU, for the tests: tests/band_port_global.c (the global recurrence and traceback of
oracle/at_oracle.c with the band of include/aligntools_b200.h) compiled with gcc into tests/_build.  Results come in
the oracle's own types (oracle.Result, oracle.BatchOut), so the tests compare them the same way."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "band_port_global.c")
SO = os.path.join(HERE, "_build", "libband_port_global.so")
_lib = None


def _load():
    global _lib
    if _lib is None:
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        if not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(SRC):
            subprocess.run(["gcc", "-O2", "-std=gnu11", "-shared", "-fPIC", "-o", SO, SRC, "-lpthread"], check=True)
        lib = C.CDLL(SO)
        lib.band_port_global.restype = C.c_int
        lib.band_port_global.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t] + [C.c_int] * 5 + \
            [C.c_int64, C.c_int64, C.POINTER(C.c_int64), C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_size_t)]
        lib.band_port_global_batch.restype = C.c_int
        lib.band_port_global_batch.argtypes = [C.c_int] * 4 + [C.c_size_t] + [C.c_void_p] * 15 + [C.c_int]
        _lib = lib
    return _lib


def align(s1: bytes, s2: bytes, p: oracle.Params = oracle.Params(), band=None) -> oracle.Result:
    """One global pair (affine gaps); band = (lo, hi) on d = j - i, or None for the unbanded recurrence."""
    lib = _load()
    cap = len(s1) + len(s2) + 1
    r1, r2, ops = (C.create_string_buffer(cap) for _ in range(3))
    sc, al = C.c_int64(), C.c_size_t()
    coords = (C.c_int32 * 4)()
    lo, hi = band if band is not None else (0, 0)
    rc = lib.band_port_global(s1, len(s1), s2, len(s2), p.m, p.u, p.o, p.e, int(band is not None), int(lo), int(hi),
                              C.byref(sc), C.cast(coords, C.c_void_p), r1, r2, ops, C.byref(al))
    if rc:
        raise RuntimeError(f"band_port_global rc={rc}")
    n = al.value
    return oracle.Result(int(sc.value), r1.raw[:n], r2.raw[:n], ops.raw[:n], tuple(coords))


def batch(p: oracle.Params, q, q_off, q_len, t, t_off, t_len, band=None, threads=8) -> oracle.BatchOut:
    """Many global pairs (uint8 q / t, uint64 offsets, uint32 lengths); band = (lo, hi) int32 arrays or None."""
    lib = _load()
    n = len(q_len)
    out = oracle.BatchOut(n, q_len, t_len, want_aln=True, want_ops=True)
    lo = hi = None
    if band is not None:
        lo, hi = (np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=np.int32), (n,))) for x in band)
    ptr = lambda a: None if a is None else a.ctypes.data      # noqa: E731
    rc = lib.band_port_global_batch(p.m, p.u, p.o, p.e, n, ptr(q), ptr(q_off), ptr(q_len), ptr(t), ptr(t_off), ptr(t_len),
                                    ptr(lo), ptr(hi), ptr(out.score), ptr(out.coords), ptr(out.r1), ptr(out.r2), ptr(out.ops),
                                    ptr(out.aln_off), ptr(out.aln_len), threads)
    if rc:
        raise RuntimeError(f"band_port_global_batch rc={rc}")
    return out
