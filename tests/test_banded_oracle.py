"""Banded overlap alignment without a GPU: the banded CPU restatement (tests/band_port.c) against the reference (full
band, and the identity property on bands derived from the reference's own path), and the stripe geometry of aligntools/c_b200/csrc/at_band.h compiled
with g++ -- windows, hand-off (deadlock freedom), pointer offsets, in-band cell counts."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import band_port
from helpers import load_fuzz

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libband_model.so")
SRC = os.path.join(HERE, "band_model.cpp")
HDRS = [os.path.join(HERE, "..", "aligntools", "c_b200", "csrc", h) for h in ("at_band.h", "at_cell.cuh")]
I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1


@pytest.fixture(scope="module")
def band_lib():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(x) for x in [SRC] + HDRS):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-o", SO, SRC], check=True)
    lib = C.CDLL(SO)
    u32, i32, i64, u64 = C.c_uint32, C.c_int32, C.c_int64, C.c_uint64
    lib.band_model_clip.argtypes = [u32, u32, i64, i64, C.c_void_p]
    lib.band_model_stripe.argtypes = [u32, u32, i32, i32, u32, u32, C.c_void_p]
    for f in ("band_model_words", "band_model_off"):
        getattr(lib, f).argtypes = [u32, u32, i32, i32, u32, u32]
        getattr(lib, f).restype = u64
    lib.band_model_pair_words.argtypes = [u32, u32, i32, i32, u32]
    lib.band_model_pair_words.restype = u64
    lib.band_model_cells.argtypes = [u32, u32, i32, i32]
    lib.band_model_cells.restype = u64
    lib.band_model_first_wait.argtypes = [u32, u32, u32, u32]
    lib.band_model_first_wait.restype = u32
    return lib


def clip(lib, l1, l2, lo, hi):
    out = (C.c_int32 * 2)()
    lib.band_model_clip(l1, l2, lo, hi, C.cast(out, C.c_void_p))
    return out[0], out[1]


def stripe(lib, l1, l2, elo, ehi, rpp, s):
    out = (C.c_uint32 * 5)()
    return tuple(out) if lib.band_model_stripe(l1, l2, elo, ehi, rpp, s, C.cast(out, C.c_void_p)) else None


def path_diagonals(res):
    """d = j - i of every cell of the path after its column-0 start, the end cell included."""
    i, j = res.coords[2], res.coords[3]
    ds = []
    for op in res.ops:
        if op == ord("M"):
            i, j = i + 1, j + 1
        elif op == ord("I"):
            i += 1
        else:
            j += 1
        ds.append(j - i)
    assert (i, j) == tuple(res.coords[:2])
    return ds


def test_full_band_matches_stored_reference(oracle_mod):
    """A band covering the whole matrix -- the int32 extremes, clipped -- gives the reference's answers."""
    cases = [c for c in load_fuzz() if c["mode"] == "overlap"]
    assert len(cases) >= 100
    for c in cases:
        p = oracle_mod.Params(c["m"], c["u"], c["o"], c["e"], c["j"], False)
        s1, s2 = c["s1"].encode("latin-1"), c["s2"].encode("latin-1")
        for band in (None, (I32_MIN, I32_MAX), (-len(s1) + 1, len(s2) - 1)):
            r = band_port.align(s1, s2, p, band=band)
            assert r.score == c["score"], (c, band)
            assert r.r1 == c["r1"].encode("latin-1") and r.r2 == c["r2"].encode("latin-1"), (c, band)


def c4_like_pair(rng, lmin, lmax):
    l1, l2 = rng.randint(lmin, lmax), rng.randint(lmin, lmax)
    s1 = bytes(rng.choice(b"ACGT") for _ in range(l1))
    ov = rng.randint(min(l1, l2) // 5, min(l1, l2))
    pre = bytearray()
    for ch in s1[l1 - ov:]:
        r = rng.random()
        if r < 0.025:
            continue
        pre.append(rng.choice(b"ACGT") if r < 0.075 else ch)
        if rng.random() < 0.025:
            pre.append(rng.choice(b"ACGT"))
    s2 = (bytes(pre) + bytes(rng.choice(b"ACGT") for _ in range(l2)))[:l2]
    return s1, s2


def test_identity_on_reference_path(oracle_mod):
    """Band = [min d, max d] of the reference's path, widened by random margins (0 included): the banded port equals the
    reference in every field."""
    rng = random.Random(2024)
    p = oracle_mod.Params()
    for k in range(36):
        s1, s2 = c4_like_pair(rng, 200, 3000 if k % 3 == 0 else 1200)
        ref = oracle_mod.port_align("overlap", s1, s2, p)
        if oracle_mod.have_ref():
            live = oracle_mod.ref_align("overlap", s1, s2, p)
            assert (live.score, live.r1, live.r2) == (ref.score, ref.r1, ref.r2)
        ds = path_diagonals(ref) or [0]
        m_lo, m_hi = (0, 0) if k % 4 == 0 else (rng.choice([0, 0, 1, 3, 40, 500]), rng.choice([0, 0, 2, 17, 300]))
        band = (min(ds) - m_lo, max(ds) + m_hi)
        assert band_port.align(s1, s2, p) == ref                          # the restatement without a band is the port
        got = band_port.align(s1, s2, p, band=band)
        assert (got.score, got.r1, got.r2, got.ops, got.coords) == (ref.score, ref.r1, ref.r2, ref.ops, ref.coords), (k, band)


def test_empty_band_is_column_zero(oracle_mod):
    p = oracle_mod.Params()
    for band in ((50, 60), (-500, -200), (I32_MAX, I32_MAX), (I32_MIN, I32_MIN)):
        r = band_port.align(b"ACGTACGTAC", b"ACGTAC", p, band=band)
        assert (r.score, r.r1, r.coords) == (0, b"", (10, 0, 10, 0)), band


def band_cases(rng, n):
    extremes = [I32_MIN, I32_MIN + 1, -(1 << 30), 0, 1, (1 << 30), I32_MAX]
    for k in range(n):
        l1, l2 = rng.randint(1, 700), rng.randint(1, 700)
        rpp = 32 * rng.randint(1, 8)
        kind = k % 6
        if kind == 0:                                        # width 1
            lo = hi = rng.randint(-l1 - 5, l2 + 5)
        elif kind == 1:                                      # wider than the matrix / int32 extremes
            lo, hi = sorted((rng.choice(extremes), rng.choice(extremes)))
        elif kind == 2:                                      # entirely outside
            lo = rng.choice([l2 + rng.randint(0, 50), -l1 - 400])
            hi = lo + rng.randint(0, 300)
        else:
            lo = rng.randint(-l1 - 20, l2 + 20)
            hi = lo + rng.choice([0, 1, 5, 31, 64, 255, 256, 600, 2000])
        yield l1, l2, rpp, lo, min(hi, I32_MAX)


def test_band_geometry(band_lib):
    """at_band.h: windows hold every in-band cell of their stripe and no more, stripes with a window are contiguous,
    pointer offsets are contiguous and sum to the pair's words, the cell count is exact."""
    rng = random.Random(7)
    for l1, l2, rpp, lo, hi in band_cases(rng, 600):
        elo, ehi = clip(band_lib, l1, l2, lo, hi)
        assert elo > ehi or (max(lo, 1 - l1), min(hi, l2 - 1)) == (elo, ehi)
        ns = (l1 + rpp - 1) // rpp
        i = np.arange(1, l1 + 1)
        jlo, jhi = np.maximum(1, i + elo), np.minimum(l2, i + ehi)
        ok = (jlo <= jhi) & (elo <= ehi)
        assert band_lib.band_model_cells(l1, l2, elo, ehi) == int((jhi - jlo + 1)[ok].sum()), (l1, l2, lo, hi)
        have, off = [], 0
        for s in range(ns):
            w = stripe(band_lib, l1, l2, elo, ehi, rpp, s)
            rows = slice(s * rpp, min((s + 1) * rpp, l1))
            cells = ok[rows]
            assert (w is not None) == bool(cells.any()), (l1, l2, lo, hi, rpp, s)
            assert band_lib.band_model_off(l1, l2, elo, ehi, rpp, s) == off
            words = band_lib.band_model_words(l1, l2, elo, ehi, rpp, s)
            off += words
            if w is None:
                assert words == 0
                continue
            have.append(s)
            c0, c1, t0, groups, t_last = w
            assert (c0, c1) == (int(jlo[rows][cells].min()), int(jhi[rows][cells].max()))
            assert 1 <= c0 <= c1 <= l2 and t0 % 32 == 0 and t0 <= c0 - 1 < t0 + 32
            assert t_last == (c1 + 31) | 31 and t0 + 16 * groups - 1 >= c1 + 31 and words == groups * rpp
        assert band_lib.band_model_pair_words(l1, l2, elo, ehi, rpp) == off
        assert have == list(range(have[0], have[-1] + 1)) if have else True


def published(c0, c1, t0, t_last):
    """Columns K2's stripe stores to its hand-off slab: every 32 steps from t0 the block 63..32 columns behind, then the
    tail after the loop -- each restricted to the window."""
    cols = set()
    for tb in range(t0, t_last + 1, 32):
        if tb >= 64:
            cols.update(range(max(tb - 63, c0), min(tb - 32, c1) + 1))
    cols.update(range(max(t_last - 62, c0), min(t_last - 31, c1) + 1))
    return cols


def test_band_hand_off_never_waits_on_unpublished_columns(band_lib):
    """Deadlock freedom: a stripe waits only for columns its predecessor publishes -- its first wait and every ring
    block -- and every column it does not wait for is out of band in the predecessor's last row (-inf is its value)."""
    rng = random.Random(11)
    for l1, l2, rpp, lo, hi in band_cases(rng, 400):
        elo, ehi = clip(band_lib, l1, l2, lo, hi)
        ns = (l1 + rpp - 1) // rpp
        wins = [stripe(band_lib, l1, l2, elo, ehi, rpp, s) for s in range(ns)]
        for s in range(1, ns):
            prod, cons = wins[s - 1], wins[s]
            if prod is None or cons is None:
                continue
            pub = published(prod[0], prod[1], prod[2], prod[4])
            assert pub == set(range(prod[0], prod[1] + 1)), (l1, l2, lo, hi, rpp, s)
            for lag in (0, 500):
                c = band_lib.band_model_first_wait(prod[0], prod[1], cons[2], lag)
                assert c in pub
            last_row = s * rpp
            for col in range(cons[2], cons[4] + 1):              # lane 0's boundary input of every step
                waited = prod[0] <= col <= prod[1]
                in_band = 1 <= col <= l2 and elo <= col - last_row <= ehi
                assert waited or not in_band, (l1, l2, lo, hi, rpp, s, col)
                assert not waited or col in pub


def test_config4_with_diag_keeps_default_output():
    from aligntools.c_b200 import synth
    a = synth.config4_overlap(n_pairs=6, lo=300, hi=900)
    b = synth.config4_overlap(n_pairs=6, lo=300, hi=900, with_diag=True)
    assert set(b) == set(a) | {"diag"}
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k
        else:
            assert a[k] == b[k], k
    assert b["diag"].dtype == np.int32
    for p in range(6):
        assert -int(a["q_len"][p]) < int(b["diag"][p]) <= 0
