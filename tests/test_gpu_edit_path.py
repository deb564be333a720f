"""Edit distance paths on the GPU (AT_OUT_EDIT_PATH): every field, the CIGAR and the gapped strings against the CPU
restatement (tests/edit_port.c) on the shapes that hit the stripe and step-block edges of both fill kernels -- the
bit-parallel one (u = 1, DNA) and the cell-by-cell one (other u, protein) -- for bytes and 2-bit input; the two kernels
agree at u = 1; without the flag edit is score-only as before; sub-slices and small arenas; a 20 kbp pair and a
100 kbp x 100 kbp pair."""
import random

import numpy as np
import pytest

import edit_port
from helpers import pack_batch
from test_gpu_banded import rle

pytestmark = pytest.mark.gpu
FIELDS = ("score", "end_i", "end_j", "beg_i", "beg_j", "cigar_off", "aln_off")
DNA, PROTEIN = b"ACGT", b"ACDEFGHIKLMNPQRSTVWY"
PATH = 1 | 2 | 4


@pytest.fixture(scope="module")
def A():
    import aligntools.c_b200 as A
    return A


@pytest.fixture(scope="module")
def aligner(A):
    al = A.Aligner()
    yield al
    al.close()


def pairs(rng, shapes, alphabet=DNA, div=0.08):
    """s2 is a mutated copy of s1, cut or padded to l2."""
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


def run(A, aligner, u, w, flags=PATH, encoding=0, dev=None):
    qb, qo, ql, tb, to, tl = w
    q_, qo_, t_, to_ = dev if dev else (qb, qo, tb, to)
    b = aligner.batch("edit", A.Opt(u=u), q_, qo_, ql, t_, to_, tl, out_flags=flags, encoding=encoding)
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


def check_vs_port(res, u, w):
    qb, qo, ql, tb, to, tl = w
    ref = edit_port.batch(u, qb, qo, ql, tb, to, tl, threads=8)
    assert np.array_equal(res.score.astype(np.int64), ref.score)
    assert np.array_equal(res.end_i, ql) and np.array_equal(res.end_j, tl)
    for k, name in enumerate(("beg_i", "beg_j")):
        bad = np.nonzero(getattr(res, name) != ref.coords[:, 2 + k].astype(np.uint32))[0]
        assert bad.size == 0, (name, bad[:5])
    for k in range(len(ql)):
        assert res.aln(k) == ref.aln(k), (k, int(ql[k]), int(tl[k]))
        assert res.cigar_string(k) == rle(ref.op(k)), k


# 1 x 1, 1 x n, n x 1; the cell-by-cell kernel's stripe edges (32 R rows, R = 8 from 225 rows on) and the bit-parallel
# kernel's (1024 R, R = 1 for a batch this small) +- 1, multi-stripe reads; targets at the 16-step block edges
# (63 / 64 / 65: the bit-parallel kernel's steps16 path against its tail) and the 256-column tiles
ROWS = [1, 2, 31, 33, 255, 256, 257, 1023, 1024, 1025, 3000]
COLS = [1, 63, 64, 65, 255, 256, 257, 700]
SHAPES = [(l1, l2) for l1 in ROWS for l2 in COLS] + [(1, 1500), (1500, 1), (2049, 2100), (5000, 300)]


@pytest.mark.parametrize("alphabet", ["dna", "protein"])
@pytest.mark.parametrize("u", [1, 2, 3, 0, -2])
def test_shapes_vs_port(A, aligner, u, alphabet):
    rng = random.Random(10 * u + len(alphabet))
    w = pairs(rng, SHAPES, DNA if alphabet == "dna" else PROTEIN)
    res = run(A, aligner, u, w)
    check_vs_port(res, u, w)
    bitpar = u == 1 and alphabet == "dna"
    assert res.timing.fill_kernel_kind == (3 if bitpar else 2)
    assert res.timing.ptr_bytes > 0


@pytest.mark.parametrize("align", [1, 16])
@pytest.mark.parametrize("u", [1, 2, -2])
def test_two_bit_vs_port(A, aligner, u, align):
    rng = random.Random(70 + u + align)
    w = pairs(rng, SHAPES)
    qb, qo, ql, tb, to, tl = w
    q2, qo2, _ = A.pack_2bit(qb, qo, ql, align=align)
    t2, to2, _ = A.pack_2bit(tb, to, tl, align=align)
    res = run(A, aligner, u, w, encoding=A.SEQ_2BIT, dev=(q2, qo2, t2, to2))
    assert res.timing.fill_kernel_flags & 4
    check_vs_port(res, u, w)


def test_bit_parallel_equals_cell_by_cell(A, aligner, monkeypatch):
    """u = 1: the bit-parallel kernel and the cell-by-cell one give identical results in every field."""
    w = pairs(random.Random(3), SHAPES)
    bits = run(A, aligner, 1, w)
    monkeypatch.setenv("AT_NO_BITPAR", "1")
    cell = run(A, aligner, 1, w)
    assert bits.timing.fill_kernel_kind == 3 and cell.timing.fill_kernel_kind == 2
    same(cell, bits)


@pytest.mark.parametrize("u", [1, 2])
def test_without_path_flag_is_score_only(A, aligner, u):
    """Flags 0 and CIGAR | ALN without AT_OUT_EDIT_PATH: no pointers, no alignments (at_batch_fetch leaves cigar_off /
    aln_off all zero) -- today's edit results; with the path, the same scores."""
    import ctypes as C
    w = pairs(random.Random(9 + u), SHAPES)
    path = run(A, aligner, u, w)
    for flags in (0, 3):
        res = run(A, aligner, u, w, flags=flags)
        assert res.timing.ptr_bytes == 0
        assert np.array_equal(res.score, path.score)
        assert np.array_equal(res.end_i, path.end_i) and np.array_equal(res.end_j, path.end_j)
        assert res.cigar is None and res.aln1 is None
    # the C-ABI with CIGAR | ALN buffers but without the path flag: offsets come back zero
    qb, qo, ql, tb, to, tl = w
    b = aligner.batch("edit", A.Opt(u=u), qb, qo, ql, tb, to, tl, out_flags=3)
    b.run()
    n = len(ql)
    score, cig, coff = np.zeros(n, np.int32), np.zeros(64, np.uint32), np.full(n + 1, 7, np.uint64)
    a1, a2, aoff = np.zeros(64, np.uint8), np.zeros(64, np.uint8), np.full(n + 1, 7, np.uint64)
    out = A._Output()
    out.score = score.ctypes.data
    out.cigar, out.cigar_cap, out.cigar_off = cig.ctypes.data, cig.size, coff.ctypes.data
    out.aln1, out.aln2, out.aln_cap, out.aln_off = a1.ctypes.data, a2.ctypes.data, a1.size, aoff.ctypes.data
    assert aligner.lib.at_batch_fetch(b.h, C.byref(out)) == 0
    b.free()
    assert np.array_equal(score, path.score) and not coff.any() and not aoff.any()
    one = aligner.align_arrays("edit", A.Opt(u=u), *w, out_flags=3)
    assert np.array_equal(one.score, path.score) and one.cigar is None and one.timing.ptr_bytes == 0


@pytest.mark.parametrize("u", [1, 2])
def test_one_shot_subslices_and_small_arena(A, aligner, monkeypatch, u):
    """at_batch_align cut into sub-slices, and the three-call path on a small pointer arena (several chunks): both equal
    the plain three-call result."""
    rng = random.Random(21 + u)
    w = pairs(rng, [(rng.randint(200, 3000), rng.randint(200, 3000)) for _ in range(60)])
    ref = run(A, aligner, u, w)
    monkeypatch.setenv("AT_PIPE_MIN_CELLS", "1")
    monkeypatch.setenv("AT_PIPE_SLICE_CELLS", "20000000")
    monkeypatch.setenv("AT_PIPE_MIN_TASKS", "1")
    one = aligner.align_arrays("edit", A.Opt(u=u), *w, out_flags=PATH)
    assert one.timing.launches > 8
    for name in ("AT_PIPE_MIN_CELLS", "AT_PIPE_SLICE_CELLS", "AT_PIPE_MIN_TASKS"):
        monkeypatch.delenv(name)
    monkeypatch.setenv("AT_PTR_BUDGET_MB", "8")
    small = run(A, aligner, u, w)
    for got in (one, small):
        for name in FIELDS:
            assert np.array_equal(getattr(got, name), getattr(ref, name)), name
        no, nc = int(ref.cigar_off[-1]), int(ref.aln_off[-1])
        assert np.array_equal(got.cigar[:no], ref.cigar[:no])
        assert np.array_equal(got.aln1[:nc], ref.aln1[:nc]) and np.array_equal(got.aln2[:nc], ref.aln2[:nc])
    monkeypatch.setenv("AT_PTR_BUDGET_MB", "1")
    with pytest.raises(A.AtError, match="traceback pointers"):
        run(A, aligner, u, w)


def test_long_pair_vs_port(A, aligner):
    w = pairs(random.Random(2), [(20000, 20000)])
    check_vs_port(run(A, aligner, 1, w), 1, w)


def path_cost(res, p, u):
    a1, a2 = (np.frombuffer(x, np.uint8) for x in res.aln(p))
    gap = (a1 == ord("-")) | (a2 == ord("-"))
    return int(gap.sum()) + u * int(((a1 != a2) & ~gap).sum())


def test_c5_size_pair(A, aligner):
    """100 kbp x 100 kbp, u = 1 (bit-parallel): the score equals the score-only run's, the path consumes exactly l1 and
    l2 and costs the score, the pointers take about l1 l2 / 4 bytes."""
    w = pairs(random.Random(5), [(100000, 100000)], div=0.1)
    qb, qo, ql, tb, to, tl = w
    score_only = run(A, aligner, 1, w, flags=0)
    res = run(A, aligner, 1, w)
    assert res.timing.fill_kernel_kind == 3
    assert res.score[0] == score_only.score[0]
    ops = res.cigar_ops(0)
    n, code = ops >> 4, ops & 15
    assert int(n[code != 2].sum()) == 100000 and int(n[code != 1].sum()) == 100000
    a1, a2 = res.aln(0)
    assert a1.replace(b"-", b"") == qb.tobytes() and a2.replace(b"-", b"") == tb.tobytes()
    assert path_cost(res, 0, 1) == res.score[0]
    assert 1.0 <= res.timing.ptr_bytes / (100000 * 100000 / 4) < 1.02
