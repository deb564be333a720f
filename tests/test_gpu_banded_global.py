"""Banded global alignment on the GPU (at_batch_create_banded / at_batch_align_banded with AT_GLOBAL): the full band
reproduces the unbanded path (bytes and 2-bit input, short pairs that the unbanded path packs two per warp on K1),
random band shapes match the banded CPU restatement in every field (DNA and protein alphabets, single diagonals, a
window at column 1 below an empty stripe, long runs of empty stripes, every window start mod 256), the long-pair shape
with a corridor band, sub-slices and small arenas, score-only runs and the band's argument errors."""
import ctypes as C
import random

import numpy as np
import pytest

import band_port_global
from helpers import pack_batch
from test_gpu_banded import in_band_cells, rle

pytestmark = pytest.mark.gpu
I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1
PRM = dict(m=1, u=-2, o=-5, e=-1, j=-10, jump=False)
FIELDS = ("score", "end_i", "end_j", "beg_i", "beg_j", "cigar_off", "aln_off")


@pytest.fixture(scope="module")
def A():
    import aligntools.c_b200 as A
    return A


@pytest.fixture(scope="module")
def aligner(A):
    al = A.Aligner()
    yield al
    al.close()


def pairs(rng, shapes, alphabet=b"ACGT", div=0.06):
    """Global pairs: s2 is a mutated copy of s1 cut or padded to l2."""
    q, t = [], []
    for l1, l2 in shapes:
        s1 = bytes(rng.choice(alphabet) for _ in range(l1))
        s2 = bytearray()
        for c in s1:
            r = rng.random()
            if r < div / 3:
                continue
            s2.append(rng.choice(alphabet) if r < div else c)
            if rng.random() < div / 3:
                s2.append(rng.choice(alphabet))
        s2 = bytes(s2[:l2]) + bytes(rng.choice(alphabet) for _ in range(max(0, l2 - len(s2))))
        q.append(s1); t.append(s2)
    qb, qo, ql = pack_batch(q)
    tb, to, tl = pack_batch(t)
    return qb, qo[:-1].copy(), ql, tb, to[:-1].copy(), tl


def run(A, aligner, prm, qb, qo, ql, tb, to, tl, band, encoding=0, flags=3, dev=None):
    q_, qo_, t_, to_ = dev if dev else (qb, qo, tb, to)
    b = aligner.batch("global", A.Opt(**prm), q_, qo_, ql, t_, to_, tl, out_flags=flags, encoding=encoding, band=band)
    tm = b.run()
    res = b.fetch()
    b.free()
    res.timing = tm
    return res


def same(got, ref):
    for name in FIELDS:
        assert np.array_equal(getattr(got, name), getattr(ref, name)), name
    no, nc = int(ref.cigar_off[-1]), int(ref.aln_off[-1])
    assert np.array_equal(got.cigar[:no], ref.cigar[:no])
    assert np.array_equal(got.aln1[:nc], ref.aln1[:nc]) and np.array_equal(got.aln2[:nc], ref.aln2[:nc])


def check_vs_port(A, aligner, oracle_mod, prm, qb, qo, ql, tb, to, tl, lo, hi, encoding=0, dev=None):
    p = oracle_mod.Params(prm["m"], prm["u"], prm["o"], prm["e"], prm["j"], False)
    ref = band_port_global.batch(p, qb, qo, ql, tb, to, tl, band=(lo, hi), threads=8)
    res = run(A, aligner, prm, qb, qo, ql, tb, to, tl, (lo, hi), encoding=encoding, dev=dev)
    assert res.timing.cells == in_band_cells(ql, tl, lo, hi)
    assert np.array_equal(res.score.astype(np.int64), ref.score)
    for k, name in enumerate(("end_i", "end_j", "beg_i", "beg_j")):
        bad = np.nonzero(getattr(res, name) != ref.coords[:, k].astype(np.uint32))[0]
        assert bad.size == 0, (name, bad[:5], lo[bad[:5]], hi[bad[:5]])
    for k in range(len(ql)):
        assert res.aln(k) == ref.aln(k), (k, int(ql[k]), int(tl[k]), lo[k], hi[k])
        assert res.cigar_string(k) == rle(ref.op(k)), k
    return res


# short pairs with repeated shapes (the unbanded path packs those two per warp on K1) and long ones (K2 either way)
SHAPES = [(1, 1), (1, 40), (40, 1), (40, 70), (150, 150), (200, 150), (256, 300), (257, 1), (300, 700), (513, 400),
          (1000, 33), (1003, 1200), (2049, 1500), (4000, 256), (700, 4097)]


@pytest.mark.parametrize("enc", ["bytes", "2bit1", "2bit16"])
def test_full_band_equals_unbanded(A, aligner, enc):
    """The whole matrix as the band (int32 extremes, or exactly [1 - l1, l2 - 1]): the unbanded results in every field."""
    qb, qo, ql, tb, to, tl = pairs(random.Random(3), SHAPES * 3)
    encoding, dev = 0, None
    if enc != "bytes":
        align = 1 if enc == "2bit1" else 16
        q2, qo2, _ = A.pack_2bit(qb, qo, ql, align=align)
        t2, to2, _ = A.pack_2bit(tb, to, tl, align=align)
        encoding, dev = A.SEQ_2BIT, (q2, qo2, t2, to2)
    ref = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, None, encoding=encoding, dev=dev)
    n = len(ql)
    for band in ((np.full(n, I32_MIN, np.int32), np.full(n, I32_MAX, np.int32)), (1 - ql.astype(np.int32), tl.astype(np.int32) - 1)):
        res = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, band, encoding=encoding, dev=dev)
        assert res.timing.cells == ref.timing.cells
        same(res, ref)


def band_shapes(rng, n, lmax=2500):
    """(l1, l2, lo, hi) with lo <= l2 - l1 <= hi, cycling through the band shapes banded global must handle."""
    out = []
    for k in range(n):
        kind = k % 9
        l1, l2 = rng.randint(1, lmax), rng.randint(1, lmax)
        if kind == 1:                                           # lo = hi = 1 - 256 s: stripe s - 1 has one cell, at column 1
            s = rng.randint(1, 6)
            l1 = rng.randint(256 * s, 256 * s + 900)
            l2 = l1 + 1 - 256 * s
        elif kind == 2:                                         # first in-band row 256 s + 1 starts a stripe
            s = rng.randint(1, 6)
            l1 = rng.randint(256 * s + 1, 256 * s + 900)
            l2 = rng.randint(1, l1 - 256 * s)
        elif kind == 3:                                         # a long run of empty stripes on top
            l1, l2 = rng.randint(2000, 4500), rng.randint(1, 300)
        d = l2 - l1
        if kind in (0, 1):
            lo = hi = d
        elif kind == 2:
            hi = -256 * s
            lo = d - rng.choice([0, 3, 100])
        elif kind == 3:
            lo, hi = d - rng.randint(0, 60), d + rng.randint(0, 60)
        elif kind == 4:
            lo, hi = d - rng.randint(0, 100), d + rng.randint(0, 100)       # narrower than a stripe
        elif kind == 5:
            lo, hi = d - rng.randint(256, 900), d + rng.randint(256, 900)   # wider than a stripe
        elif kind == 6:
            lo, hi = I32_MIN, I32_MAX
        elif kind == 7:
            lo, hi = (I32_MIN, d + rng.randint(0, 40)) if k % 2 else (d - rng.randint(0, 40), I32_MAX)
        else:
            w = rng.choice([0, 16, 64])
            lo, hi = min(0, d) - w, max(0, d) + w                         # corridor from the start to the end cell
        out.append((l1, l2, lo, hi))
    return out


def shaped_batch(rng, cases, alphabet=b"ACGT"):
    qb, qo, ql, tb, to, tl = pairs(rng, [(a, b) for a, b, _, _ in cases], alphabet)
    return qb, qo, ql, tb, to, tl, np.array([c[2] for c in cases], np.int32), np.array([c[3] for c in cases], np.int32)


@pytest.mark.parametrize("alphabet", ["dna", "protein"])
def test_random_bands_vs_port(A, aligner, oracle_mod, alphabet):
    """Band shapes: single diagonals, lo = hi = 1 - 256 s, a first in-band row that starts a stripe, long runs of empty
    stripes, narrower / wider than a stripe, int32 extremes, corridors -- against the banded restatement, every field.
    DNA runs the query-profile kernel, a protein alphabet the xor / min form."""
    rng = random.Random(27 if alphabet == "dna" else 28)
    ab = b"ACGT" if alphabet == "dna" else b"ACDEFGHIKLMNPQRSTVWY"
    cases = band_shapes(rng, 108) + [(l1, l2, l2 - l1 - 5, l2 - l1 + 5) for l1, l2 in SHAPES]
    qb, qo, ql, tb, to, tl, lo, hi = shaped_batch(rng, cases, ab)
    check_vs_port(A, aligner, oracle_mod, PRM, qb, qo, ql, tb, to, tl, lo, hi)


@pytest.mark.parametrize("align", [1, 16])
def test_window_start_every_residue_2bit(A, aligner, oracle_mod, align):
    """2-bit targets, first windows starting at every column mod 256 (stripe 0: c0 = 1 + lo), with records at every
    ring shift: K2's tile schedule starts mid-tile."""
    rng = random.Random(199 + align)
    cases = []
    for k in range(256):
        lo = k - 1 + 256 * rng.randint(0, 1)
        l1 = rng.randint(300, 900)
        l2 = l1 + max(lo, 0) + rng.randint(0, 500)
        cases.append((l1, l2, lo, l2 - l1 + rng.choice([0, 40, 200, 600])))
    qb, qo, ql, tb, to, tl, lo, hi = shaped_batch(rng, cases)
    q2, qo2, _ = A.pack_2bit(qb, qo, ql, align=align)
    t2, to2, _ = A.pack_2bit(tb, to, tl, align=align)
    res = check_vs_port(A, aligner, oracle_mod, PRM, qb, qo, ql, tb, to, tl, lo, hi, encoding=A.SEQ_2BIT, dev=(q2, qo2, t2, to2))
    assert res.timing.fill_kernel_flags & 4


def test_long_global_corridor(A, aligner, oracle_mod):
    """synth.long_global pairs with a +-64 corridor: the banded restatement's result, and the unbanded one wherever
    the unbanded path stays in the corridor."""
    from aligntools.c_b200 import synth
    w = synth.long_global(n_pairs=12, lo=3000, hi=7000)
    q, qo, ql, t, to, tl = w["q"], w["q_off"], w["q_len"], w["t"], w["t_off"], w["t_len"]
    lo, hi = synth.global_corridor(ql, tl, 64)
    res = check_vs_port(A, aligner, oracle_mod, w["params"], q, qo, ql, t, to, tl, lo, hi)
    full = run(A, aligner, w["params"], q, qo, ql, t, to, tl, None)
    assert res.timing.ptr_bytes < 0.1 * full.timing.ptr_bytes
    assert (res.score <= full.score).all()
    assert (res.score == full.score).sum() >= 10


def test_one_shot_subslices_and_small_arena(A, aligner, monkeypatch):
    """at_batch_align_banded cut into sub-slices, and the three-call path on a small pointer arena (several chunks):
    both equal the plain three-call banded result."""
    rng = random.Random(15)
    qb, qo, ql, tb, to, tl, lo, hi = shaped_batch(rng, band_shapes(rng, 400, lmax=3000))
    ref = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi))
    monkeypatch.setenv("AT_PIPE_MIN_CELLS", "1")
    monkeypatch.setenv("AT_PIPE_SLICE_CELLS", "3000000")
    monkeypatch.setenv("AT_PIPE_MIN_TASKS", "1")
    res = aligner.align_arrays("global", A.Opt(**PRM), qb, qo, ql, tb, to, tl, out_flags=3, band=(lo, hi))
    assert res.timing.launches > 8 and res.timing.cells == ref.timing.cells
    for name in ("AT_PIPE_MIN_CELLS", "AT_PIPE_SLICE_CELLS", "AT_PIPE_MIN_TASKS"):
        monkeypatch.delenv(name)
    monkeypatch.setenv("AT_PTR_BUDGET_MB", "8")      # several chunks; the largest pair (a full band) needs about 4.5 MB
    small = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi))
    for got in (res, small):
        same(got, ref)


def test_score_only(A, aligner):
    rng = random.Random(18)
    qb, qo, ql, tb, to, tl, lo, hi = shaped_batch(rng, band_shapes(rng, 60))
    full = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi))
    so = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi), flags=0)
    assert so.timing.ptr_bytes == 0 and full.timing.ptr_bytes > 0
    assert so.timing.cells == full.timing.cells == in_band_cells(ql, tl, lo, hi)
    for name in ("score", "end_i", "end_j"):
        assert np.array_equal(getattr(so, name), getattr(full, name)), name


def test_band_must_hold_end_diagonal(A, aligner):
    """A global band that misses l2 - l1 is AT_E_ARG naming the pair, for both entry points; lo > hi is reported first
    with its own message; local, fit (with and without jump) and edit still take no band."""
    qb, qo, ql, tb, to, tl = pairs(random.Random(1), [(30, 40), (50, 60), (70, 90)])
    lo, hi = np.array([0, 0, 0], np.int32), np.array([10, 5, 30], np.int32)        # pair 1: l2 - l1 = 10 > 5
    with pytest.raises(A.AtError) as e:
        aligner.batch("global", A.Opt(), qb, qo, ql, tb, to, tl, band=(lo, hi))
    assert e.value.rc == -1 and "band" in str(e.value) and "pair 1" in str(e.value) and "10" in str(e.value)
    with pytest.raises(A.AtError) as e:
        aligner.align_arrays("global", A.Opt(), qb, qo, ql, tb, to, tl, out_flags=3, band=(lo, hi))
    assert e.value.rc == -1 and "pair 1" in str(e.value)
    with pytest.raises(A.AtError) as e:
        aligner.batch("global", A.Opt(), qb, qo, ql, tb, to, tl, band=(np.array([0, 11, 40], np.int32), hi))
    assert e.value.rc == -1 and "lo > hi at pair 1" in str(e.value)
    ok = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, np.array([10, 10, 20], np.int32)))
    assert ok.timing.cells > 0
    for mode, opt in (("local", A.Opt()), ("fit", A.Opt()), ("fit", A.Opt(jump=True)), ("edit", A.Opt(u=1))):
        with pytest.raises(A.AtError) as e:
            aligner.batch(mode, opt, qb, qo, ql, tb, to, tl, band=(np.full(3, -100, np.int32), np.full(3, 100, np.int32)))
        assert e.value.rc == -1 and "band" in str(e.value), mode
    lib = aligner.lib
    inp = A._Input(3, 0, qb.ctypes.data, qo.ctypes.data, ql.ctypes.data, tb.ctypes.data, to.ctypes.data, tl.ctypes.data, None, None)
    prm = A.Opt().c()
    bd = A._Band(None, hi.ctypes.data)
    h = C.c_void_p()
    assert lib.at_batch_create_banded(aligner.h, 0, C.byref(prm), C.byref(inp), C.byref(bd), 0, C.byref(h)) == -1
    assert "NULL" in aligner.last_error()
