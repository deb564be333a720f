"""Substitution-matrix scoring on the CPU, for the tests: tests/subst_port.c (oracle/at_oracle.c's affine and overlap
alignments with s(i, j) = matrix[s1[i-1], s2[j-1]]) compiled with gcc into tests/_build.  Results come in the oracle's own
types (oracle.Result, oracle.BatchOut), so the tests compare them the same way."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "subst_port.c")
SO = os.path.join(HERE, "_build", "libsubst_port.so")
MODES = {"global": 0, "local": 1, "fit": 2, "overlap": 3}
_lib = None


def _load():
    global _lib
    if _lib is None:
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        if not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(SRC):
            subprocess.run(["gcc", "-O2", "-std=gnu11", "-shared", "-fPIC", "-o", SO, SRC, "-lpthread"], check=True)
        lib = C.CDLL(SO)
        lib.subst_port_align.restype = C.c_int
        lib.subst_port_align.argtypes = [C.c_int, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_void_p] + [C.c_int] * 4 + \
            [C.c_void_p, C.c_size_t, C.POINTER(C.c_int64), C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_size_t)]
        lib.subst_port_batch.restype = C.c_int
        lib.subst_port_batch.argtypes = [C.c_int, C.c_void_p] + [C.c_int] * 4 + [C.c_size_t] + [C.c_void_p] * 15 + [C.c_int]
        _lib = lib
    return _lib


def _mat(matrix):
    m = np.ascontiguousarray(np.asarray(matrix, dtype=np.int8))
    assert m.shape == (256, 256)
    return m


def align(mode, s1: bytes, s2: bytes, matrix, p: oracle.Params = oracle.Params(), sites=None) -> oracle.Result:
    """One pair; p.m / p.u are not used, p.o / p.e / p.j / p.jump are (jump: 0, 1 blacklist, 2 whitelist)."""
    lib = _load()
    mat = _mat(matrix)
    cap = len(s1) + len(s2) + 1
    r1, r2, ops = (C.create_string_buffer(cap) for _ in range(3))
    sc, al = C.c_int64(), C.c_size_t()
    coords = (C.c_int32 * 4)()
    sa = np.ascontiguousarray(np.asarray(sites if sites is not None else [0], dtype=np.int32))
    ns = len(sites) if sites is not None else 0
    rc = lib.subst_port_align(MODES[mode], s1, len(s1), s2, len(s2), mat.ctypes.data, p.o, p.e, p.j, int(p.jump),
                              sa.ctypes.data if ns else None, ns, C.byref(sc), C.cast(coords, C.c_void_p), r1, r2, ops, C.byref(al))
    if rc:
        raise RuntimeError(f"subst_port_align rc={rc}")
    n = al.value
    return oracle.Result(int(sc.value), r1.raw[:n], r2.raw[:n], ops.raw[:n], tuple(coords))


def batch(mode, matrix, p: oracle.Params, q, q_off, q_len, t, t_off, t_len, sites=None, site_off=None, threads=8) -> oracle.BatchOut:
    """Many pairs (uint8 q / t, uint64 offsets, uint32 lengths; fit + jump: int32 sites with uint64 site_off[n + 1])."""
    lib = _load()
    mat = _mat(matrix)
    n = len(q_len)
    out = oracle.BatchOut(n, q_len, t_len, want_aln=True, want_ops=True)
    ptr = lambda a: None if a is None else a.ctypes.data      # noqa: E731
    rc = lib.subst_port_batch(MODES[mode], mat.ctypes.data, p.o, p.e, p.j, int(p.jump), n, ptr(q), ptr(q_off), ptr(q_len), ptr(t),
                              ptr(t_off), ptr(t_len), ptr(sites), ptr(site_off), ptr(out.score), ptr(out.coords), ptr(out.r1),
                              ptr(out.r2), ptr(out.ops), ptr(out.aln_off), ptr(out.aln_len), threads)
    if rc:
        raise RuntimeError(f"subst_port_batch rc={rc}")
    return out


def rescore(mode, r1: bytes, r2: bytes, ops: bytes, matrix, p: oracle.Params) -> int:
    """The score of an alignment, column by column, from the recurrences of oracle/at_oracle.c:
    - an (x, y) column adds matrix[x, y]; in local mode the first column adds max(matrix[x, y], 0) (a HOME cell, or a cell
      next to the zero border);
    - overlap: every gap column adds o;
    - affine modes: a gap column opens with o and extends with e; a run at the very start of a global alignment extends the
      border (o + e per column from the first), one at the start of a local alignment grows from the zero border (max(o, e));
    - jump columns (N): j for the first of a run, 0 for the rest."""
    m = np.asarray(matrix, dtype=np.int64)
    total, prev = 0, None
    for k, (a, b) in enumerate(zip(r1, r2)):
        op = chr(ops[k])
        if op == "M":
            c = int(m[a, b])
            if mode == "local" and k == 0:
                c = max(c, 0)
        elif mode == "overlap":
            c = p.o
        elif op == "N":
            c = p.j if prev != "N" else 0
        elif prev == op:
            c = p.e
        elif k == 0:
            c = {"global": p.o + p.e, "local": max(p.o, p.e)}.get(mode, p.o)
        else:
            c = p.o
        total += c
        prev = op
    return total
