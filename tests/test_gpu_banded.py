"""Banded overlap alignment on the GPU (at_batch_create_banded / at_batch_align_banded): the full band reproduces the
unbanded path, random bands match the banded port in every field (bytes and 2-bit input, DNA and protein alphabets,
every window start mod 256), the C4 shape with a band around the true path, sub-slices and small arenas, score-only
runs and the band's argument errors."""
import ctypes as C
import random

import numpy as np
import pytest

import band_port
from helpers import pack_batch

pytestmark = pytest.mark.gpu
I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1


@pytest.fixture(scope="module")
def A():
    import aligntools.c_b200 as A
    return A


@pytest.fixture(scope="module")
def aligner(A):
    al = A.Aligner()
    yield al
    al.close()


def rle(ops: bytes) -> str:
    out, k = [], 0
    while k < len(ops):
        j = k
        while j < len(ops) and ops[j] == ops[k]:
            j += 1
        out.append(f"{j - k}{chr(ops[k])}")
        k = j
    return "".join(out)


def in_band_cells(ql, tl, lo, hi):
    n = 0
    for l1, l2, a, b in zip(ql.tolist(), tl.tolist(), lo.tolist(), hi.tolist()):
        a, b = max(a, 1 - l1), min(b, l2 - 1)
        for d in range(a, b + 1):
            n += max(0, min(l1, l2 - d) - max(1, 1 - d) + 1)
    return n


def pairs(rng, shapes, alphabet=b"ACGT", div=0.08):
    q, t = [], []
    for l1, l2 in shapes:
        base = bytes(rng.choice(alphabet) for _ in range(l1 + l2))
        s1 = bytes(c if rng.random() > div else rng.choice(alphabet) for c in base[:l1])
        sh = rng.randint(0, l1 - 1)
        s2 = bytes(c if rng.random() > div else rng.choice(alphabet) for c in base[sh:sh + l2])
        q.append(s1); t.append(s2)
    qb, qo, ql = pack_batch(q)
    tb, to, tl = pack_batch(t)
    return qb, qo[:-1].copy(), ql, tb, to[:-1].copy(), tl


def run(A, aligner, prm, qb, qo, ql, tb, to, tl, band, encoding=0, flags=3, dev=None):
    q_, qo_, t_, to_ = dev if dev else (qb, qo, tb, to)
    b = aligner.batch("overlap", A.Opt(**prm), q_, qo_, ql, t_, to_, tl, out_flags=flags, encoding=encoding, band=band)
    tm = b.run()
    res = b.fetch()
    b.free()
    res.timing = tm
    return res


def check_vs_port(A, aligner, oracle_mod, prm, qb, qo, ql, tb, to, tl, lo, hi, encoding=0, dev=None):
    p = oracle_mod.Params(prm["m"], prm["u"], prm["o"], prm["e"], prm["j"], False)
    ref = band_port.batch(p, qb, qo, ql, tb, to, tl, band=(lo, hi), threads=8)
    res = run(A, aligner, prm, qb, qo, ql, tb, to, tl, (lo, hi), encoding=encoding, dev=dev)
    assert res.timing.cells == in_band_cells(ql, tl, lo, hi)
    assert np.array_equal(res.score.astype(np.int64), ref.score)
    for k, name in enumerate(("end_i", "end_j", "beg_i", "beg_j")):
        bad = np.nonzero(getattr(res, name) != ref.coords[:, k].astype(np.uint32))[0]
        assert bad.size == 0, (name, bad[:5], lo[bad[:5]], hi[bad[:5]])
    for k in range(len(ql)):
        assert res.aln(k) == ref.aln(k), (k, lo[k], hi[k])
        assert res.cigar_string(k) == rle(ref.op(k)), k
    return res


PRM = dict(m=1, u=-2, o=-3, e=-1, j=-5, jump=False)
SHAPES = [(1, 1), (40, 70), (200, 150), (256, 300), (257, 1), (300, 700), (513, 400), (1000, 33), (1003, 1200),
          (2049, 1500), (4000, 256), (700, 4097)]


@pytest.mark.parametrize("enc", ["bytes", "2bit1", "2bit16"])
def test_full_band_equals_unbanded(A, aligner, enc):
    """The whole matrix as the band (int32 extremes, clipped): the unbanded path's results in every field."""
    qb, qo, ql, tb, to, tl = pairs(random.Random(3), SHAPES * 2)
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
        for name in ("score", "end_i", "end_j", "beg_i", "beg_j", "cigar_off", "aln_off"):
            assert np.array_equal(getattr(res, name), getattr(ref, name)), name
        no, nc = int(ref.cigar_off[-1]), int(ref.aln_off[-1])
        assert np.array_equal(res.cigar[:no], ref.cigar[:no])
        assert np.array_equal(res.aln1[:nc], ref.aln1[:nc]) and np.array_equal(res.aln2[:nc], ref.aln2[:nc])


def random_bands(rng, ql, tl):
    lo, hi = [], []
    for k, (l1, l2) in enumerate(zip(ql.tolist(), tl.tolist())):
        kind = k % 9
        if kind == 0:
            a = b = rng.randint(-l1, l2)                                   # width 1
        elif kind == 1:
            a, b = l2 + rng.randint(0, 40), l2 + 300                        # entirely right of the matrix: empty
        elif kind == 2:
            a, b = -l1 - 300, -l1 - rng.randint(0, 40)                      # entirely below: empty
        elif kind == 3:
            a, b = I32_MIN, rng.randint(-l1, l2)                            # cuts the first stripes away (upper part kept)
        elif kind == 4:
            a, b = rng.randint(-l1, l2), I32_MAX                            # cuts the last stripes away
        elif kind == 5:
            a = rng.randint(-l1, l2); b = a + rng.randint(1, 100)          # narrower than a stripe
        elif kind == 6:
            a = rng.randint(-l1, l2); b = a + rng.randint(256, 900)        # wider than a stripe
        elif kind == 7:
            a, b = I32_MIN, I32_MAX
        else:
            a = b = 0
        lo.append(a); hi.append(min(b, I32_MAX))
    return np.array(lo, np.int32), np.array(hi, np.int32)


@pytest.mark.parametrize("alphabet", ["dna", "protein"])
def test_random_bands_vs_port(A, aligner, oracle_mod, alphabet):
    """Band shapes: empty, width 1, narrower / wider than a stripe, outside the matrix, cutting the first or last
    stripes away, int32 extremes -- against the banded port, every field.  DNA runs the query-profile kernel, a
    protein alphabet the fallback."""
    rng = random.Random(17 if alphabet == "dna" else 18)
    ab = b"ACGT" if alphabet == "dna" else b"ACDEFGHIKLMNPQRSTVWY"
    shapes = [(rng.randint(1, 2500), rng.randint(1, 2500)) for _ in range(90)] + SHAPES
    qb, qo, ql, tb, to, tl = pairs(rng, shapes, ab)
    lo, hi = random_bands(rng, ql, tl)
    check_vs_port(A, aligner, oracle_mod, PRM, qb, qo, ql, tb, to, tl, lo, hi)


@pytest.mark.parametrize("align", [1, 16])
def test_window_start_every_residue_2bit(A, aligner, oracle_mod, align):
    """2-bit targets, windows starting at every column mod 256 (first stripe: c0 = 1 + lo), with records at every ring
    shift: K2's tile schedule starts mid-tile."""
    rng = random.Random(99 + align)
    shapes = [(rng.randint(300, 900), rng.randint(700, 1400)) for _ in range(256)]
    qb, qo, ql, tb, to, tl = pairs(rng, shapes)
    lo = np.array([k - 1 + 256 * rng.randint(0, 1) for k in range(256)], np.int32)
    hi = lo + np.array([rng.choice([0, 40, 200, 600]) for _ in range(256)], np.int32)
    q2, qo2, _ = A.pack_2bit(qb, qo, ql, align=align)
    t2, to2, _ = A.pack_2bit(tb, to, tl, align=align)
    res = check_vs_port(A, aligner, oracle_mod, PRM, qb, qo, ql, tb, to, tl, lo, hi, encoding=A.SEQ_2BIT, dev=(q2, qo2, t2, to2))
    assert res.timing.fill_kernel_flags & 4


def path_band(coords, ops, margin):
    i, j = int(coords[2]), int(coords[3])
    ds = []
    for op in ops:
        if op == ord("M"):
            i, j = i + 1, j + 1
        elif op == ord("I"):
            i += 1
        else:
            j += 1
        ds.append(j - i)
    ds = ds or [0]
    return min(ds) - margin, max(ds) + margin


def test_config4_band_around_path(A, aligner, oracle_mod):
    """C4 shape (10-20 kbp), band = the port's path +- 64: the port's result; two pairs also against the compiled
    reference where it is present."""
    from aligntools.c_b200 import synth
    w = synth.config4_overlap(n_pairs=32)
    q, qo, ql, t, to, tl = w["q"], w["q_off"], w["q_len"], w["t"], w["t_off"], w["t_len"]
    p = oracle_mod.Params(**{k: w["params"][k] for k in "muoej"}, jump=False)
    ref = oracle_mod.port_batch("overlap", p, q, np.append(qo, 0).astype(np.uint64), ql, t, np.append(to, 0).astype(np.uint64), tl,
                                want_aln=True, want_ops=True, threads=16)
    bands = [path_band(ref.coords[k], ref.op(k), 64) for k in range(32)]
    lo = np.array([b[0] for b in bands], np.int32)
    hi = np.array([b[1] for b in bands], np.int32)
    res = check_vs_port(A, aligner, oracle_mod, w["params"], q, qo, ql, t, to, tl, lo, hi)
    assert np.array_equal(res.score.astype(np.int64), ref.score)          # identity: the unbanded answer
    for k in range(32):
        assert res.aln(k) == ref.aln(k), k
    assert res.timing.ptr_bytes < 0.2 * 4 * sum(int(a) * int(b) for a, b in zip(ql, tl)) / 16
    if oracle_mod.have_ref():
        for k in (0, 17):
            s1 = q[int(qo[k]):int(qo[k]) + int(ql[k])].tobytes()
            s2 = t[int(to[k]):int(to[k]) + int(tl[k])].tobytes()
            r = oracle_mod.ref_align("overlap", s1, s2, p)
            assert (int(res.score[k]),) + res.aln(k) == (r.score, r.r1, r.r2), k


def test_one_shot_subslices_and_small_arena(A, aligner, monkeypatch):
    """at_batch_align_banded cut into sub-slices, and the three-call path on a small pointer arena (several chunks):
    both equal the plain three-call banded result."""
    rng = random.Random(5)
    shapes = [(rng.randint(20, 3000), rng.randint(20, 3000)) for _ in range(400)]
    qb, qo, ql, tb, to, tl = pairs(rng, shapes)
    lo, hi = random_bands(rng, ql, tl)
    ref = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi))
    monkeypatch.setenv("AT_PIPE_MIN_CELLS", "1")
    monkeypatch.setenv("AT_PIPE_SLICE_CELLS", "3000000")
    monkeypatch.setenv("AT_PIPE_MIN_TASKS", "1")
    res = aligner.align_arrays("overlap", A.Opt(**PRM), qb, qo, ql, tb, to, tl, out_flags=3, band=(lo, hi))
    assert res.timing.launches > 8 and res.timing.cells == ref.timing.cells
    for name in ("AT_PIPE_MIN_CELLS", "AT_PIPE_SLICE_CELLS", "AT_PIPE_MIN_TASKS"):
        monkeypatch.delenv(name)
    monkeypatch.setenv("AT_PTR_BUDGET_MB", "4")      # several chunks; the largest pair (a full band) needs 2.3 MB
    small = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi))
    for got in (res, small):
        for name in ("score", "end_i", "end_j", "beg_i", "beg_j", "cigar_off", "aln_off"):
            assert np.array_equal(getattr(got, name), getattr(ref, name)), name
        no, nc = int(ref.cigar_off[-1]), int(ref.aln_off[-1])
        assert np.array_equal(got.cigar[:no], ref.cigar[:no])
        assert np.array_equal(got.aln1[:nc], ref.aln1[:nc]) and np.array_equal(got.aln2[:nc], ref.aln2[:nc])


def test_score_only(A, aligner):
    rng = random.Random(8)
    qb, qo, ql, tb, to, tl = pairs(rng, SHAPES * 3)
    lo, hi = random_bands(rng, ql, tl)
    full = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi))
    so = run(A, aligner, PRM, qb, qo, ql, tb, to, tl, (lo, hi), flags=0)
    assert so.timing.ptr_bytes == 0 and full.timing.ptr_bytes > 0
    assert so.timing.cells == full.timing.cells == in_band_cells(ql, tl, lo, hi)
    for name in ("score", "end_i", "end_j"):
        assert np.array_equal(getattr(so, name), getattr(full, name)), name


def test_band_argument_errors(A, aligner):
    qb, qo, ql, tb, to, tl = pairs(random.Random(1), [(30, 40), (50, 60)])
    lo, hi = np.array([-5, -5], np.int32), np.array([5, 5], np.int32)
    for mode in ("global", "local", "fit", "edit"):
        with pytest.raises(A.AtError) as e:
            aligner.batch(mode, A.Opt(u=1) if mode == "edit" else A.Opt(), qb, qo, ql, tb, to, tl, band=(lo, hi))
        assert e.value.rc == -1 and "band" in str(e.value)
    with pytest.raises(A.AtError) as e:
        aligner.batch("overlap", A.Opt(), qb, qo, ql, tb, to, tl, band=(lo, np.array([5, -6], np.int32)))
    assert e.value.rc == -1 and "pair 1" in str(e.value)
    # NULL lo / hi, through the C-ABI directly, for both entry points
    lib = aligner.lib
    inp = A._Input(2, 0, qb.ctypes.data, qo.ctypes.data, ql.ctypes.data, tb.ctypes.data, to.ctypes.data, tl.ctypes.data, None, None)
    prm = A.Opt().c()
    score = np.zeros(2, np.int32)
    out = A._Output()
    out.score = score.ctypes.data
    for bd in (A._Band(None, hi.ctypes.data), A._Band(lo.ctypes.data, None)):
        h = C.c_void_p()
        assert lib.at_batch_create_banded(aligner.h, 3, C.byref(prm), C.byref(inp), C.byref(bd), 0, C.byref(h)) == -1
        assert "NULL" in aligner.last_error()
        assert lib.at_batch_align_banded(aligner.h, 3, C.byref(prm), C.byref(inp), C.byref(bd), 0, C.byref(out), None) == -1
