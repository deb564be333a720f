"""Substitution-matrix scoring on the CPU (tests/subst_port.c, the restatement the GPU tests compare with): with the
match / mismatch table it is the oracle port and reproduces the stored reference answers on every mode variant; with random
asymmetric tables every returned path, rescored column by column, gives the returned score and spells the sequences."""
import random
import zlib

import numpy as np
import pytest

import subst_port
from helpers import load_fuzz, pack_batch

VARIANTS = ["global", "local", "fit", "fitjump", "fitwhite", "overlap"]


@pytest.fixture(scope="module")
def oracle_mod():
    import oracle
    oracle.build()
    return oracle


def identity(m, u):
    t = np.full((256, 256), u, dtype=np.int8)
    np.fill_diagonal(t, m)
    return t


def mode_of(v):
    return "fit" if v.startswith("fit") else v


def params(oracle_mod, v, rng):
    jump = {"fitjump": 1, "fitwhite": 2}.get(v, 0)
    return oracle_mod.Params(rng.randint(1, 4), rng.randint(-5, -1), rng.randint(-6, 0), rng.randint(-3, 0), rng.randint(-12, -1), jump)


def random_pairs(rng, n, alphabet, mode, lmax=60):
    q, t, sites = [], [], []
    for _ in range(n):
        l1 = rng.randint(1, lmax)
        l2 = rng.randint(max(2, l1) if mode == "fit" else 1, lmax + (lmax if mode == "fit" else 0))
        s1 = bytes(rng.choice(alphabet) for _ in range(l1))
        s2 = bytearray(rng.choice(alphabet) for _ in range(l2))
        if l2 >= l1 and rng.random() < 0.7:      # related pairs: s1 planted in s2 with a few changes
            at = rng.randint(0, l2 - l1)
            for k, c in enumerate(s1):
                s2[at + k] = c if rng.random() > 0.15 else rng.choice(alphabet)
        q.append(s1); t.append(bytes(s2))
        sites.append(sorted(rng.sample(range(l2), min(l2, rng.randint(0, 4)))))
    return q, t, sites


def run_port(oracle_mod, v, matrix, p, q, t, sites):
    qb, qo, ql = pack_batch(q)
    tb, to, tl = pack_batch(t)
    sa = so = None
    if p.jump:
        sa = np.array([x for s in sites for x in s] + [0], dtype=np.int32)
        so = np.zeros(len(q) + 1, np.uint64)
        np.cumsum([len(s) for s in sites], out=so[1:])
    return subst_port.batch(mode_of(v), matrix, p, qb, qo[:-1].copy(), ql, tb, to[:-1].copy(), tl, sites=sa, site_off=so), (qb, qo, ql, tb, to, tl, sa, so)


@pytest.mark.parametrize("v", VARIANTS)
def test_identity_matrix_is_the_oracle(oracle_mod, v):
    rng = random.Random(zlib.crc32(v.encode()))
    for alphabet in (b"ACGT", b"ACDEFGHIKLMNPQRSTVWY"):
        p = params(oracle_mod, v, rng)
        q, t, sites = random_pairs(rng, 120, alphabet, mode_of(v))
        got, (qb, qo, ql, tb, to, tl, sa, so) = run_port(oracle_mod, v, identity(p.m, p.u), p, q, t, sites)
        ref = oracle_mod.port_batch(mode_of(v), p, qb, qo[:-1].copy(), ql, tb, to[:-1].copy(), tl, sites=sa, site_off=so,
                                    want_aln=True, want_ops=True, threads=8)
        assert np.array_equal(got.score, ref.score)
        assert np.array_equal(got.coords, ref.coords)
        for k in range(len(q)):
            assert got.aln(k) == ref.aln(k) and got.op(k) == ref.op(k), k


@pytest.mark.parametrize("v", VARIANTS[:4] + ["overlap"])
def test_identity_matrix_reproduces_stored_answers(v):
    cases = [c for c in load_fuzz() if ("fitjump" if c["jump"] else c["mode"]) == v]
    assert cases
    import oracle
    for c in cases:
        p = oracle.Params(c["m"], c["u"], c["o"], c["e"], c["j"], bool(c["jump"]))
        r = subst_port.align(c["mode"], c["s1"].encode(), c["s2"].encode(), identity(c["m"], c["u"]), p, sites=c["sites"] if c["jump"] else None)
        assert (r.score, r.r1, r.r2) == (c["score"], c["r1"].encode(), c["r2"].encode())


@pytest.mark.parametrize("v", VARIANTS)
def test_random_matrix_paths_rescore_to_the_score(oracle_mod, v):
    rng = random.Random(7 + VARIANTS.index(v))
    mode = mode_of(v)
    for alphabet in (b"ACGT", b"ACGTN", bytes(range(65, 105))):
        p = params(oracle_mod, v, rng)
        mat = np.array([[rng.randint(-9, 9) for _ in range(256)] for _ in range(256)], dtype=np.int8)   # asymmetric
        for a in alphabet:
            mat[a, a] = rng.randint(1, 9)
        q, t, sites = random_pairs(rng, 150, alphabet, mode)
        got, _ = run_port(oracle_mod, v, mat, p, q, t, sites)
        for k in range(len(q)):
            r1, r2 = got.aln(k)
            ops = got.op(k)
            assert subst_port.rescore(mode, r1, r2, ops, mat, p) == int(got.score[k]), (k, ops)
            ei, ej, bi, bj = (int(x) for x in got.coords[k])
            s1, s2 = r1.replace(b"-", b""), r2.replace(b"-", b"")
            if mode == "global":
                assert (s1, s2) == (q[k], t[k])
            else:      # the path spells the sequences between its begin and end cells
                assert s1 == q[k][bi:ei] and s2 == t[k][bj:ej], k
