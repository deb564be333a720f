"""Substitution-matrix scoring on the GPU (at_batch_create_scored / at_batch_align_scored): the match / mismatch table
reproduces the unscored results in every field (every mode, bytes and 2-bit input, K1 int32 and packed lanes, K2 with
multi-stripe reads, the profile and table variants, the three-call and pipelined one-shot paths); random tables match the
CPU restatement (tests/subst_port.c) on ACGT targets (profile variants), ACGTN, 20-, 40-, 150- and 256-letter alphabets
(table variants, up to a 128 KB table) and with AT_NO_PROFILE; score-only runs, the score-range bound and the argument
errors."""
import ctypes as C
import random
import zlib

import numpy as np
import pytest

import subst_port
from helpers import pack_batch

pytestmark = pytest.mark.gpu
FIELDS = ("score", "end_i", "end_j", "beg_i", "beg_j", "cigar_off", "aln_off")
VARIANTS = {"global": ("global", 0), "local": ("local", 0), "fit": ("fit", 0), "fitjump": ("fit", 1), "fitwhite": ("fit", 2),
            "overlap": ("overlap", 0)}
PROTEIN = b"ACDEFGHIKLMNPQRSTVWY"
WIDE = bytes(range(48, 88))      # 40 letters: more than 32 on either side


@pytest.fixture(scope="module")
def A():
    import aligntools.c_b200 as A
    return A


@pytest.fixture(scope="module")
def aligner(A):
    al = A.Aligner()
    yield al
    al.close()


def rle(ops):
    out, k = "", 0
    while k < len(ops):
        r = k
        while r < len(ops) and ops[r] == ops[k]:
            r += 1
        out += f"{r - k}{chr(ops[k])}"
        k = r
    return out


def make_pairs(rng, shapes, alphabet, mode):
    q, t, sites = [], [], []
    for l1, l2 in shapes:
        if mode == "fit":
            l2 = max(l2, l1, 2)
        s1 = bytes(rng.choice(alphabet) for _ in range(l1))
        s2 = bytearray(rng.choice(alphabet) for _ in range(l2))
        if l2 >= l1:
            at = rng.randint(0, l2 - l1)
            for k, c in enumerate(s1):
                s2[at + k] = c if rng.random() > 0.1 else rng.choice(alphabet)
        q.append(s1); t.append(bytes(s2))
        sites.append(sorted(rng.sample(range(l2), min(l2, 5))))
    return q, t, sites


class Inputs:
    def __init__(self, A, q, t, sites, jump, enc="bytes"):
        self.q, self.t, self.sites = q, t, sites
        self.qb, qo, self.ql = pack_batch(q)
        self.tb, to, self.tl = pack_batch(t)
        self.qo, self.to = qo[:-1].copy(), to[:-1].copy()
        self.sa = self.so = None
        if jump:
            self.sa = np.array([x for s in sites for x in s] + [0], dtype=np.int32)
            self.so = np.zeros(len(q) + 1, np.uint64)
            np.cumsum([len(s) for s in sites], out=self.so[1:])
        self.encoding, self.dev = 0, (self.qb, self.qo, self.tb, self.to)
        if enc != "bytes":
            align = 1 if enc == "2bit1" else 16
            q2, qo2, _ = A.pack_2bit(self.qb, self.qo, self.ql, align=align)
            t2, to2, _ = A.pack_2bit(self.tb, self.to, self.tl, align=align)
            self.encoding, self.dev = A.SEQ_2BIT, (q2, qo2, t2, to2)


def opt(A, v, m=2, u=-3, o=-4, e=-1, j=-9):
    return A.Opt(m=m, u=u, o=o, e=e, j=j, jump=VARIANTS[v][1] > 0, whitelist=VARIANTS[v][1] == 2)


def run3(A, aligner, v, op, x, scoring=None, flags=3):
    """create + run + fetch"""
    q_, qo_, t_, to_ = x.dev
    b = aligner.batch(VARIANTS[v][0], op, q_, qo_, x.ql, t_, to_, x.tl, sites=x.sa, site_off=x.so, out_flags=flags,
                      encoding=x.encoding, scoring=scoring)
    tm = b.run()
    res = b.fetch()
    b.free()
    res.timing = tm
    return res


def run1(A, aligner, v, op, x, scoring=None, flags=3):
    """one-shot at_batch_align(_scored)"""
    q_, qo_, t_, to_ = x.dev
    return aligner.align_arrays(VARIANTS[v][0], op, q_, qo_, x.ql, t_, to_, x.tl, sites=x.sa, site_off=x.so, out_flags=flags,
                                encoding=x.encoding, scoring=scoring)


def same(got, ref):
    for name in FIELDS:
        assert np.array_equal(getattr(got, name), getattr(ref, name)), name
    no, nc = int(ref.cigar_off[-1]), int(ref.aln_off[-1])
    assert np.array_equal(got.cigar[:no], ref.cigar[:no])
    assert np.array_equal(got.aln1[:nc], ref.aln1[:nc]) and np.array_equal(got.aln2[:nc], ref.aln2[:nc])


def vs_port(A, v, op, x, mat, res):
    import oracle
    p = oracle.Params(op.m, op.u, op.o, op.e, op.j, VARIANTS[v][1])
    ref = subst_port.batch(VARIANTS[v][0], mat, p, x.qb, x.qo, x.ql, x.tb, x.to, x.tl, sites=x.sa, site_off=x.so)
    assert np.array_equal(res.score.astype(np.int64), ref.score)
    for k, name in enumerate(("end_i", "end_j", "beg_i", "beg_j")):
        bad = np.nonzero(getattr(res, name) != ref.coords[:, k].astype(np.uint32))[0]
        assert bad.size == 0, (name, bad[:5])
    for k in range(len(x.ql)):
        assert res.aln(k) == ref.aln(k), k
        assert res.cigar_string(k) == rle(ref.op(k)), k


SHORT = [(1, 1), (7, 30), (40, 70), (150, 500), (150, 500), (150, 500), (150, 500), (200, 150), (256, 300), (100, 100), (100, 100)]
LONG = [(257, 1), (300, 700), (513, 400), (1000, 1200), (2049, 1500), (700, 4097)]


@pytest.mark.parametrize("v", list(VARIANTS))
@pytest.mark.parametrize("enc", ["bytes", "2bit1", "2bit16"])
def test_identity_matrix_equals_unscored(A, aligner, v, enc):
    """m / u as a table: every field of the unscored call, short (K1) and long (K2, several stripes) pairs, both entries."""
    rng = random.Random(zlib.crc32(f"{v}{enc}".encode()))
    q, t, sites = make_pairs(rng, SHORT * 3 + LONG, b"ACGT", VARIANTS[v][0])
    x = Inputs(A, q, t, sites, VARIANTS[v][1], enc)
    op = opt(A, v)
    ident = A.identity_scoring(op.m, op.u)
    ref = run3(A, aligner, v, op, x)
    got = run3(A, aligner, v, op, x, scoring=ident)
    same(got, ref)
    assert got.timing.fill_kernel_flags & 9 == 9      # profile variant, scored
    same(run1(A, aligner, v, op, x, scoring=ident), ref)


@pytest.mark.parametrize("v", list(VARIANTS))
@pytest.mark.parametrize("alphabet", [b"ACGTN", PROTEIN])
def test_identity_matrix_table_variant_equals_unscored(A, aligner, v, alphabet):
    """Targets of more than four bytes run the table variants: still every field of the unscored call."""
    rng = random.Random(zlib.crc32(v.encode() + alphabet))
    q, t, sites = make_pairs(rng, SHORT * 3 + LONG, alphabet, VARIANTS[v][0])
    x = Inputs(A, q, t, sites, VARIANTS[v][1])
    op = opt(A, v)
    ref = run3(A, aligner, v, op, x)
    got = run3(A, aligner, v, op, x, scoring=A.identity_scoring(op.m, op.u))
    same(got, ref)
    assert got.timing.fill_kernel_flags & 9 == 8      # table variant, scored


@pytest.mark.parametrize("v", ["global", "local", "fit"])
def test_identity_matrix_int32_and_packed_lanes(A, aligner, v, monkeypatch):
    """150 x 500 pairs run on K1's packed lanes with a profile; without them (AT_NO_P16) on int32 lanes: both as unscored."""
    rng = random.Random(11)
    q, t, sites = make_pairs(rng, [(150, 500)] * 512, b"ACGT", v)
    x = Inputs(A, q, t, sites, 0)
    op = opt(A, v)
    ident = A.identity_scoring(op.m, op.u)
    ref = run3(A, aligner, v, op, x)
    got = run3(A, aligner, v, op, x, scoring=ident)
    assert got.timing.fill_kernel_kind == ref.timing.fill_kernel_kind == 1
    same(got, ref)
    monkeypatch.setenv("AT_NO_P16", "1")
    got = run3(A, aligner, v, op, x, scoring=ident)
    assert got.timing.fill_kernel_kind == 0
    same(got, ref)


def test_identity_matrix_one_shot_subslices_and_small_arena(A, aligner, monkeypatch):
    rng = random.Random(5)
    for v, alphabet in (("local", b"ACGT"), ("global", PROTEIN), ("overlap", b"ACGTN"), ("fitjump", b"ACGT")):
        q, t, sites = make_pairs(rng, (SHORT + LONG) * 6, alphabet, VARIANTS[v][0])
        x = Inputs(A, q, t, sites, VARIANTS[v][1])
        op = opt(A, v)
        ident = A.identity_scoring(op.m, op.u)
        ref = run1(A, aligner, v, op, x)
        monkeypatch.setenv("AT_PIPE_MIN_CELLS", "1")
        monkeypatch.setenv("AT_PIPE_SLICE_CELLS", "2000000")
        monkeypatch.setenv("AT_PIPE_MIN_TASKS", "1")
        same(run1(A, aligner, v, op, x, scoring=ident), ref)
        for name in ("AT_PIPE_MIN_CELLS", "AT_PIPE_SLICE_CELLS", "AT_PIPE_MIN_TASKS"):
            monkeypatch.delenv(name)
        monkeypatch.setenv("AT_PTR_BUDGET_MB", "4")
        same(run1(A, aligner, v, op, x, scoring=ident), ref)
        same(run3(A, aligner, v, op, x, scoring=ident), ref)
        monkeypatch.delenv("AT_PTR_BUDGET_MB")


def random_matrix(rng, alphabet, lo=-9, hi=9):
    mat = np.array([[rng.randint(lo, hi) for _ in range(256)] for _ in range(256)], dtype=np.int8)    # asymmetric
    for a in alphabet:
        mat[a, a] = rng.randint(2, hi)
    return mat


@pytest.mark.parametrize("v", list(VARIANTS))
@pytest.mark.parametrize("alphabet", [b"ACGT", b"ACGTN", PROTEIN, WIDE])
def test_random_matrix_matches_restatement(A, aligner, v, alphabet):
    rng = random.Random(zlib.crc32(v.encode() + alphabet + b"1"))
    q, t, sites = make_pairs(rng, SHORT * 2 + LONG, alphabet, VARIANTS[v][0])
    x = Inputs(A, q, t, sites, VARIANTS[v][1])
    op = opt(A, v, o=rng.randint(-8, -2), e=rng.randint(-3, 0), j=rng.randint(-15, -5))
    mat = random_matrix(rng, alphabet)
    res = run3(A, aligner, v, op, x, scoring=mat)
    assert bool(res.timing.fill_kernel_flags & 1) == (alphabet == b"ACGT")
    vs_port(A, v, op, x, mat, res)


@pytest.mark.parametrize("v", list(VARIANTS))
@pytest.mark.parametrize("n_sym", [150, 256])
def test_large_alphabets_match_restatement(A, aligner, v, n_sym):
    """Every byte on both sides (a 128 KB table) and 150 symbols (a 45 KB table: with K2's static shared memory above the
    48 KB a launch gets without opting in), on K1 and on K2 with several stripes."""
    rng = random.Random(zlib.crc32(f"{v}{n_sym}".encode()))
    alphabet = bytes(range(256)) if n_sym == 256 else bytes(range(40, 190))
    q, t, sites = make_pairs(rng, SHORT + LONG, alphabet, VARIANTS[v][0])
    every = bytes(rng.sample(list(alphabet), len(alphabet)))
    q.append(every); t.append(bytes(rng.sample(list(alphabet), len(alphabet))) * 2)     # every symbol in the reads and the targets
    sites.append([3, 70])
    x = Inputs(A, q, t, sites, VARIANTS[v][1])
    assert len(set(x.qb.tobytes())) == len(set(x.tb.tobytes())) == n_sym
    op = opt(A, v, o=rng.randint(-8, -2), e=rng.randint(-3, 0), j=rng.randint(-15, -5))
    mat = random_matrix(rng, alphabet)
    res = run3(A, aligner, v, op, x, scoring=mat)
    assert res.timing.fill_kernel_flags & 9 == 8
    vs_port(A, v, op, x, mat, res)


@pytest.mark.parametrize("v", ["local", "fitjump", "overlap"])
@pytest.mark.parametrize("enc", ["bytes", "2bit16"])
def test_no_profile_takes_the_table_variant(A, aligner, v, enc, monkeypatch):
    """AT_NO_PROFILE: DNA targets run the table variants too (2-bit input is then expanded to bytes)."""
    rng = random.Random(41)
    q, t, sites = make_pairs(rng, SHORT + LONG, b"ACGT", VARIANTS[v][0])
    x = Inputs(A, q, t, sites, VARIANTS[v][1], enc)
    op = opt(A, v)
    mat = random_matrix(rng, b"ACGT")
    monkeypatch.setenv("AT_NO_PROFILE", "1")
    res = run3(A, aligner, v, op, x, scoring=mat)
    assert res.timing.fill_kernel_flags & 13 == 8      # table variant, bytes in HBM
    vs_port(A, v, op, Inputs(A, q, t, sites, VARIANTS[v][1]), mat, res)


@pytest.mark.parametrize("v", ["global", "local", "overlap"])
def test_random_matrix_2bit_profile(A, aligner, v):
    """2-bit input: codes stand for A C G T when the profile reads the matrix."""
    rng = random.Random(21)
    q, t, sites = make_pairs(rng, SHORT * 2 + LONG, b"ACGT", v)
    x = Inputs(A, q, t, sites, 0, "2bit16")
    op = opt(A, v)
    mat = random_matrix(rng, b"ACGT")
    res = run3(A, aligner, v, op, x, scoring=mat)
    x8 = Inputs(A, q, t, sites, 0)
    vs_port(A, v, op, x8, mat, res)


@pytest.mark.parametrize("v", ["local", "fitjump", "overlap"])
def test_score_only_equals_traceback_run(A, aligner, v):
    rng = random.Random(31)
    q, t, sites = make_pairs(rng, SHORT + LONG, PROTEIN, VARIANTS[v][0])
    x = Inputs(A, q, t, sites, VARIANTS[v][1])
    op = opt(A, v)
    mat = random_matrix(rng, PROTEIN)
    full = run3(A, aligner, v, op, x, scoring=mat)
    only = run3(A, aligner, v, op, x, scoring=mat, flags=0)
    for name in ("score", "end_i", "end_j"):
        assert np.array_equal(getattr(only, name), getattr(full, name)), name
    assert only.timing.ptr_bytes == 0


def test_score_range_bound(A, aligner):
    """(l1 + l2 + 2) * maxabs must stay below 2^25 (with K1's 40 columns of slack), maxabs taken over o, e, j and the matrix."""
    n = 1
    mat = np.zeros((256, 256), np.int8)
    mat[65, 65] = 100
    op = A.Opt(m=1, u=-1, o=-1, e=-1, j=-1)
    limit = ((1 << 25) - 1) // 100      # l1 + l2 + 42 <= limit
    l1 = 300
    for l2, ok in ((limit - 42 - l1, True), (limit - 41 - l1, False)):
        x = Inputs(A, [b"A" * l1], [b"A" * l2], [[]], 0)
        if ok:
            res = run3(A, aligner, "local", op, x, scoring=mat, flags=0)
            assert res.score[0] == 100 * l1
        else:
            with pytest.raises(A.AtError) as e:
                run3(A, aligner, "local", op, x, scoring=mat, flags=0)
            assert e.value.rc == -6
            res = run3(A, aligner, "local", op, x, flags=0)      # the same pair without the matrix: m, u, o, e, j of 1
            assert res.score[0] == l1


def test_argument_errors(A, aligner):
    x = Inputs(A, [b"ACGT"], [b"ACGA"], [[]], 0)
    lib = aligner.lib
    inp = A._Input(1, 0, x.qb.ctypes.data, x.qo.ctypes.data, x.ql.ctypes.data, x.tb.ctypes.data, x.to.ctypes.data, x.tl.ctypes.data, None, None)
    prm = A.Opt().c()
    good = A.identity_scoring(1, -2)
    res = A.BatchResult(1)
    out = A._Output()
    out.score = res.score.ctypes.data
    for mode, sc in ((4, A._Scoring(good.ctypes.data)), (1, A._Scoring(None))):
        h = C.c_void_p()
        assert lib.at_batch_create_scored(aligner.h, mode, C.byref(prm), C.byref(inp), C.byref(sc), 0, C.byref(h)) == -1
        assert aligner.last_error().startswith("scoring")
        assert lib.at_batch_align_scored(aligner.h, mode, C.byref(prm), C.byref(inp), C.byref(sc), 0, C.byref(out), None) == -1
        assert aligner.last_error().startswith("scoring")
    # sc == NULL is the unscored call
    h = C.c_void_p()
    assert lib.at_batch_create_scored(aligner.h, 1, C.byref(prm), C.byref(inp), None, 3, C.byref(h)) == 0
    lib.at_batch_free(h)
