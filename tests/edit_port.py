"""Edit distance with a path on the CPU, for the tests: tests/edit_port.c (edit_dist of oracle/at_oracle.c with the
AT_OUT_EDIT_PATH traceback of include/aligntools_b200.h) compiled with gcc into tests/_build.  Results come in the
oracle's own types (oracle.Result, oracle.BatchOut), so the tests compare them the same way."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "edit_port.c")
SO = os.path.join(HERE, "_build", "libedit_port.so")
_lib = None


def _load():
    global _lib
    if _lib is None:
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        if not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(SRC):
            subprocess.run(["gcc", "-O2", "-std=gnu11", "-shared", "-fPIC", "-o", SO, SRC, "-lpthread"], check=True)
        lib = C.CDLL(SO)
        lib.edit_port_align.restype = C.c_int
        lib.edit_port_align.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_int64), C.c_void_p,
                                        C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_size_t)]
        lib.edit_port_batch.restype = C.c_int
        lib.edit_port_batch.argtypes = [C.c_int, C.c_size_t] + [C.c_void_p] * 13 + [C.c_int]
        _lib = lib
    return _lib


def align(s1: bytes, s2: bytes, u: int = -2) -> oracle.Result:
    """One pair: score, gapped strings, per-column ops (M / I / D), coords (end_i, end_j, beg_i, beg_j)."""
    lib = _load()
    cap = len(s1) + len(s2) + 1
    r1, r2, ops = (C.create_string_buffer(cap) for _ in range(3))
    sc, al = C.c_int64(), C.c_size_t()
    coords = (C.c_int32 * 4)()
    rc = lib.edit_port_align(s1, len(s1), s2, len(s2), int(u), C.byref(sc), C.cast(coords, C.c_void_p), r1, r2, ops, C.byref(al))
    if rc:
        raise RuntimeError(f"edit_port_align rc={rc}")
    n = al.value
    return oracle.Result(int(sc.value), r1.raw[:n], r2.raw[:n], ops.raw[:n], tuple(coords))


def batch(u: int, q, q_off, q_len, t, t_off, t_len, threads=8) -> oracle.BatchOut:
    """Many pairs (uint8 q / t, uint64 offsets, uint32 lengths)."""
    lib = _load()
    n = len(q_len)
    out = oracle.BatchOut(n, q_len, t_len, want_aln=True, want_ops=True)
    ptr = lambda a: a.ctypes.data      # noqa: E731
    rc = lib.edit_port_batch(int(u), n, ptr(q), ptr(q_off), ptr(q_len), ptr(t), ptr(t_off), ptr(t_len), ptr(out.score), ptr(out.coords),
                             ptr(out.r1), ptr(out.r2), ptr(out.ops), ptr(out.aln_off), ptr(out.aln_len), threads)
    if rc:
        raise RuntimeError(f"edit_port_batch rc={rc}")
    return out
