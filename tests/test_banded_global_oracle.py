"""Banded global alignment without a GPU: the banded CPU restatement (tests/band_port_global.c) against the
reference (full band, stored reference answers, the identity property on bands derived from the reference's own path,
banded <= unbanded on random bands), and at_band.h compiled with g++ at the affine kernel's 8 steps per pointer word
(wsh = 3, 256 rows per stripe) -- windows, pointer offsets against a brute-force count, the stripe hand-off -- and at
wsh = 4, where it must give the numbers the overlap path has always used."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import band_port_global
from helpers import load_fuzz

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "_build")
HDRS = [os.path.join(HERE, "..", "aligntools", "c_b200", "csrc", h) for h in ("at_band.h", "at_cell.cuh")]
I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1
RPP = 256


def _so(name):
    src, so = os.path.join(HERE, name + ".cpp"), os.path.join(BUILD, "lib" + name + ".so")
    os.makedirs(BUILD, exist_ok=True)
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(x) for x in [src] + HDRS):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-o", so, src], check=True)
    return C.CDLL(so)


@pytest.fixture(scope="module")
def libs():
    u32, i32, u64 = C.c_uint32, C.c_int32, C.c_uint64
    w = _so("band_model_wsh")
    w.band_wsh_stripe.argtypes = [u32, u32, i32, i32, u32, u32, u32, C.c_void_p]
    for f in ("band_wsh_words", "band_wsh_off"):
        getattr(w, f).argtypes = [u32, u32, i32, i32, u32, u32, u32]
        getattr(w, f).restype = u64
    w.band_wsh_pair_words.argtypes = [u32, u32, i32, i32, u32, u32]
    w.band_wsh_pair_words.restype = u64
    m = _so("band_model")            # the overlap path's entry points (at_band.h's defaults)
    m.band_model_clip.argtypes = [u32, u32, C.c_int64, C.c_int64, C.c_void_p]
    m.band_model_stripe.argtypes = [u32, u32, i32, i32, u32, u32, C.c_void_p]
    for f in ("band_model_words", "band_model_off"):
        getattr(m, f).argtypes = [u32, u32, i32, i32, u32, u32]
        getattr(m, f).restype = u64
    m.band_model_pair_words.argtypes = [u32, u32, i32, i32, u32]
    m.band_model_pair_words.restype = u64
    return w, m


def clip(m, l1, l2, lo, hi):
    out = (C.c_int32 * 2)()
    m.band_model_clip(l1, l2, lo, hi, C.cast(out, C.c_void_p))
    return out[0], out[1]


def stripe(w, l1, l2, elo, ehi, rpp, s, wsh):
    out = (C.c_uint32 * 5)()
    return tuple(out) if w.band_wsh_stripe(l1, l2, elo, ehi, rpp, s, wsh, C.cast(out, C.c_void_p)) else None


def inner_path_diagonals(res):
    """d = j - i of every cell (i >= 1, j >= 1) of a global path, the end cell (l1, l2) included; the flushed run on
    row 0 or column 0 is left out."""
    i = j = 0
    ds = []
    for op in res.ops:
        if op == ord("M"):
            i, j = i + 1, j + 1
        elif op == ord("I"):
            i += 1
        else:
            j += 1
        if i >= 1 and j >= 1:
            ds.append(j - i)
    assert (i, j) == tuple(res.coords[:2])
    return ds


def mutated(rng, l1, div=0.03, alphabet=b"ACGT"):
    s1 = bytes(rng.choice(alphabet) for _ in range(l1))
    out = bytearray()
    for ch in s1:
        r = rng.random()
        if r < div:
            continue                                          # deletion
        out.append(rng.choice(alphabet) if r < 2 * div else ch)
        if rng.random() < div:
            out.append(rng.choice(alphabet))                  # insertion
    return s1, bytes(out) or s1[:1]


def test_full_band_matches_port_and_stored_reference(oracle_mod):
    """A band covering the whole matrix -- the int32 extremes, or exactly [1 - l1, l2 - 1] -- gives the oracle port's
    result in every field and the reference's stored answers."""
    cases = [c for c in load_fuzz() if c["mode"] == "global" and c["s1"] and c["s2"]]
    assert len(cases) >= 100
    for c in cases:
        p = oracle_mod.Params(c["m"], c["u"], c["o"], c["e"], c["j"], False)
        s1, s2 = c["s1"].encode("latin-1"), c["s2"].encode("latin-1")
        port = oracle_mod.port_align("global", s1, s2, p)
        for band in (None, (I32_MIN, I32_MAX), (-len(s1) + 1, len(s2) - 1)):
            r = band_port_global.align(s1, s2, p, band=band)
            assert r.score == c["score"], (c, band)
            assert r.r1 == c["r1"].encode("latin-1") and r.r2 == c["r2"].encode("latin-1"), (c, band)
            assert (r.score, r.r1, r.r2, r.ops, r.coords) == (port.score, port.r1, port.r2, port.ops, port.coords), (c, band)


def test_identity_on_reference_path(oracle_mod):
    """Band = [min d, max d] over the reference path's cells with i, j >= 1, widened by random margins (0 included):
    the banded restatement equals the reference in every field."""
    rng = random.Random(2025)
    for k in range(40):
        p = oracle_mod.Params() if k % 2 else oracle_mod.Params(2, -3, -4, -1, -10, False)
        s1, s2 = mutated(rng, rng.randint(1, 2500 if k % 4 == 0 else 700), div=rng.choice([0.01, 0.03, 0.1]))
        if k % 5 == 1:
            s2 = s2[rng.randint(0, len(s2) // 2):] or s2          # a target much shorter than the read
        ref = oracle_mod.port_align("global", s1, s2, p)
        if oracle_mod.have_ref():
            live = oracle_mod.ref_align("global", s1, s2, p)
            assert (live.score, live.r1, live.r2) == (ref.score, ref.r1, ref.r2)
        ds = inner_path_diagonals(ref)
        assert ds[-1] == len(s2) - len(s1)
        m_lo, m_hi = (0, 0) if k % 3 == 0 else (rng.choice([0, 0, 1, 3, 40, 500]), rng.choice([0, 0, 2, 17, 300]))
        band = (min(ds) - m_lo, max(ds) + m_hi)
        assert band_port_global.align(s1, s2, p) == ref                  # the restatement without a band is the port
        got = band_port_global.align(s1, s2, p, band=band)
        assert (got.score, got.r1, got.r2, got.ops, got.coords) == (ref.score, ref.r1, ref.r2, ref.ops, ref.coords), (k, band)


def test_banded_score_never_exceeds_unbanded(oracle_mod):
    """Random bands holding the end diagonal: a banded global score is never above the unbanded one, and the banded
    alignment is a valid global alignment of the pair that stays in its band."""
    rng = random.Random(31)
    p = oracle_mod.Params()
    for k in range(120):
        s1, s2 = mutated(rng, rng.randint(1, 400), div=rng.choice([0.02, 0.1, 0.3]))
        l1, l2 = len(s1), len(s2)
        d = l2 - l1
        lo, hi = d - rng.choice([0, 0, 1, 5, 30, 300]), d + rng.choice([0, 0, 1, 5, 30, 300])
        if k % 4 == 0:
            lo = hi = d
        full = band_port_global.align(s1, s2, p)
        got = band_port_global.align(s1, s2, p, band=(lo, hi))
        assert got.score <= full.score, (k, lo, hi)
        assert got.r1.replace(b"-", b"") == s1 and got.r2.replace(b"-", b"") == s2
        assert all(lo <= x <= hi for x in inner_path_diagonals(got)), (k, lo, hi)


def band_cases(rng, n):
    """(l1, l2, lo, hi) with lo <= l2 - l1 <= hi: the bands banded global admits."""
    for k in range(n):
        l1, l2 = rng.randint(1, 1500), rng.randint(1, 1500)
        d = l2 - l1
        kind = k % 5
        if kind == 0:
            lo = hi = d                                                         # the end diagonal alone
        elif kind == 1:
            lo, hi = I32_MIN, rng.choice([d, d + 3, I32_MAX])                   # int32 extremes
        elif kind == 2:
            s = rng.randint(1, max(1, l1 // RPP + 1))                           # lo = hi = 1 - 256 s: window at column 1
            lo = hi = 1 - RPP * s
            l2 = max(1, l1 + lo)
            if l2 - l1 != lo:
                lo = hi = l2 - l1
        else:
            lo, hi = d - rng.choice([0, 1, 31, 64, 255, 256, 600]), d + rng.choice([0, 1, 31, 64, 255, 256, 600])
        yield l1, l2, lo, hi


def test_geometry_wsh3(libs):
    """at_band.h at 8 steps per pointer word: windows hold exactly their stripe's in-band cells, empty stripes are a
    run at the top, every window's pointer groups cover its steps with none to spare, offsets and pair words equal a
    brute-force count."""
    w, m = libs
    rng = random.Random(3)
    for l1, l2, lo, hi in band_cases(rng, 500):
        elo, ehi = clip(m, l1, l2, lo, hi)
        assert elo <= l2 - l1 <= ehi
        ns = (l1 + RPP - 1) // RPP
        i = np.arange(1, l1 + 1)
        jlo, jhi = np.maximum(1, i + elo), np.minimum(l2, i + ehi)
        ok = jlo <= jhi
        assert ok[-1] and (ok.all() or ok[np.argmax(ok):].all())              # in-band rows: a bottom run
        brute, off = 0, 0
        have = []
        for s in range(ns):
            win = stripe(w, l1, l2, elo, ehi, RPP, s, 3)
            rows = slice(s * RPP, min((s + 1) * RPP, l1))
            cells = ok[rows]
            assert (win is not None) == bool(cells.any()), (l1, l2, lo, hi, s)
            assert w.band_wsh_off(l1, l2, elo, ehi, RPP, s, 3) == off
            words = w.band_wsh_words(l1, l2, elo, ehi, RPP, s, 3)
            off += words
            if win is None:
                assert words == 0
                continue
            have.append(s)
            c0, c1, t0, groups, t_last = win
            assert (c0, c1) == (int(jlo[rows][cells].min()), int(jhi[rows][cells].max()))
            assert t0 % 32 == 0 and t0 <= c0 - 1 < t0 + 32 and t_last == (c1 + 31) | 31
            last_step = c1 + 31                                                  # lane 31 reaches column c1
            g = (last_step - t0) // 8 + 1                                        # 8-step groups from t0 up to it
            assert groups == g and words == g * RPP
            brute += g * RPP
        assert have == list(range(have[0], ns))                                   # the last stripe always has a window
        assert w.band_wsh_pair_words(l1, l2, elo, ehi, RPP, 3) == off == brute


def published(c0, c1, t0, t_last):
    """Columns K2's affine stripe stores to its hand-off slab: every 32 steps from t0 the block 63..32 columns behind,
    then the tail after the loop -- each restricted to the window."""
    cols = set()
    for tb in range(t0, t_last + 1, 32):
        if tb >= 64:
            cols.update(range(max(tb - 63, c0), min(tb - 32, c1) + 1))
    cols.update(range(max(t_last - 62, c0), min(t_last - 31, c1) + 1))
    return cols


def consumer(prod, cons, lag):
    """What K2's affine stripe waits for and loads from the stripe above: (awaited column, columns loaded after it)
    -- the first block before the loop, then one block ahead every 32 steps (at_wave_affine, BANDED)."""
    in0, in1 = prod[0], prod[1]
    t0, t_last = cons[2], cons[4]
    yield min(max(t0 + max(31, lag), in0), in1), [c for c in range(t0, t0 + 32) if in0 <= c <= in1]
    for tb in range(t0, t_last + 1, 32):
        loads = [c for c in range(tb + 32, tb + 64) if in0 <= c <= in1]
        if tb + 32 <= in1 and tb + 63 >= in0:
            yield min(in1, tb + 63), loads
        else:
            assert not loads


def test_hand_off_never_waits_on_unpublished_columns(libs):
    """Deadlock freedom and no stale reads: a stripe waits only for columns its predecessor publishes, loads only
    columns it has waited for, and every column it takes as -inf instead is out of band in the predecessor's last row."""
    w, m = libs
    rng = random.Random(13)
    for l1, l2, lo, hi in band_cases(rng, 400):
        elo, ehi = clip(m, l1, l2, lo, hi)
        ns = (l1 + RPP - 1) // RPP
        wins = [stripe(w, l1, l2, elo, ehi, RPP, s, 3) for s in range(ns)]
        for s in range(1, ns):
            prod, cons = wins[s - 1], wins[s]
            if prod is None:
                continue
            pub = published(prod[0], prod[1], prod[2], prod[4])
            assert pub == set(range(prod[0], prod[1] + 1)), (l1, l2, lo, hi, s)
            for lag in (0, 500):
                for need, loads in consumer(prod, cons, lag):
                    assert need in pub and all(c <= need for c in loads), (l1, l2, lo, hi, s, lag)
            last_row = s * RPP
            for col in range(max(1, cons[2]), min(l2, cons[4]) + 1):
                loaded = prod[0] <= col <= prod[1]
                assert loaded or not elo <= col - last_row <= ehi, (l1, l2, lo, hi, s, col)


def test_wsh4_gives_the_overlap_numbers(libs):
    """The word shift's default (4) is what the overlap path has always used: the explicit wsh = 4 entry points and
    the unchanged band_model ones agree on every stripe."""
    w, m = libs
    rng = random.Random(5)
    for _ in range(400):
        l1, l2 = rng.randint(1, 900), rng.randint(1, 900)
        rpp = 32 * rng.randint(1, 8)
        lo = rng.randint(-l1 - 20, l2 + 20)
        hi = lo + rng.choice([0, 1, 31, 255, 600, 3000])
        elo, ehi = clip(m, l1, l2, lo, hi)
        for s in range((l1 + rpp - 1) // rpp):
            out = (C.c_uint32 * 5)()
            old = tuple(out) if m.band_model_stripe(l1, l2, elo, ehi, rpp, s, C.cast(out, C.c_void_p)) else None
            assert stripe(w, l1, l2, elo, ehi, rpp, s, 4) == old
            assert w.band_wsh_words(l1, l2, elo, ehi, rpp, s, 4) == m.band_model_words(l1, l2, elo, ehi, rpp, s)
            assert w.band_wsh_off(l1, l2, elo, ehi, rpp, s, 4) == m.band_model_off(l1, l2, elo, ehi, rpp, s)
        assert w.band_wsh_pair_words(l1, l2, elo, ehi, rpp, 4) == m.band_model_pair_words(l1, l2, elo, ehi, rpp)


def test_long_global_is_seeded_and_full_length():
    from aligntools.c_b200 import synth
    a, b = synth.long_global(n_pairs=4, lo=2000, hi=3000), synth.long_global(n_pairs=4, lo=2000, hi=3000)
    for k in ("q", "q_off", "q_len", "t", "t_off", "t_len"):
        assert np.array_equal(a[k], b[k]), k
    assert ((a["q_len"] >= 2000) & (a["q_len"] <= 3000)).all()
    assert (np.abs(a["t_len"].astype(np.int64) - a["q_len"]) < 0.03 * a["q_len"]).all()
    lo, hi = synth.global_corridor(a["q_len"], a["t_len"], 64)
    d = a["t_len"].astype(np.int64) - a["q_len"]
    assert lo.dtype == hi.dtype == np.int32
    assert (lo == np.minimum(0, d) - 64).all() and (hi == np.maximum(0, d) + 64).all()
