"""CPU tests: pin the oracle port (oracle/at_oracle.c) against the reference's golden
vectors (SURVEY.md Appendix B), the committed fuzz fixtures and -- where it was built --
the compiled, unmodified reference itself."""
import hashlib
import random

import numpy as np
import pytest

from helpers import (expected_stdout, load_cli, load_fuzz, pack_batch, parse_cli_argv,
                     sites_from_comment)


def test_port_matches_golden_cli(oracle_mod):
    gold = load_cli()
    checked = 0
    for v in gold["vectors"]:
        if v["rc"] != 0:
            continue
        mode, prm, fname = parse_cli_argv(v["argv"])
        recs = gold["files"][fname.split("/")[-1]]["records"]
        s1, s2 = recs[0]["seq"].encode(), recs[1]["seq"].encode()
        comment = recs[1]["comment"] or ""
        p = oracle_mod.Params(**{k: prm[k] for k in "muoej"}, jump=prm["jump"])
        sites = sites_from_comment(comment) if (mode == "fit" and prm["jump"]) else None
        r = oracle_mod.port_align(mode, s1, s2, p, sites)
        out = expected_stdout(mode, prm, comment, r.score, r.r1, r.r2)
        assert hashlib.md5(out).hexdigest() == v["stdout_md5"], v["id"]
        assert out == v["stdout"].encode("latin-1"), v["id"]
        checked += 1
    assert checked >= 27


def test_port_matches_fuzz_fixtures(oracle_mod):
    cases = load_fuzz()
    assert len(cases) >= 900
    for c in cases:
        p = oracle_mod.Params(c["m"], c["u"], c["o"], c["e"], c["j"], bool(c["jump"]))
        r = oracle_mod.port_align(c["mode"], c["s1"].encode("latin-1"), c["s2"].encode("latin-1"), p, c["sites"])
        assert r.score == c["score"], c
        if c["mode"] != "edit":
            assert r.r1 == c["r1"].encode("latin-1") and r.r2 == c["r2"].encode("latin-1"), c


def _rescore(mode, p, ops, r1, r2):
    """Recompute the score from the emitted columns (SURVEY.md A.8): gap run from M costs
    o + (k-1) e; jump run costs j once."""
    sc, prev = 0, None
    for k, op in enumerate(ops):
        ch = chr(op)
        if ch == "M":
            sc += p.m if r1[k] == r2[k] else p.u
        elif ch in "ID":
            sc += p.e if prev == ch else p.o
        elif ch == "N":
            sc += 0 if prev == "N" else p.j
        prev = ch
    return sc


def test_port_ops_rescore(oracle_mod):
    """fit / fit+jump: the alignment starts in row 0 (M or U = 0) so Σ column scores == score."""
    cases = [c for c in load_fuzz() if c["mode"] == "fit"]
    n = 0
    for c in cases:
        p = oracle_mod.Params(c["m"], c["u"], c["o"], c["e"], c["j"], bool(c["jump"]))
        r = oracle_mod.port_align("fit", c["s1"].encode("latin-1"), c["s2"].encode("latin-1"), p, c["sites"])
        assert len(r.ops) == len(r.r1)
        # a leading run of D columns started from U[0][j] = 0 extends at e without an open
        ops = r.ops
        lead = 0
        while lead < len(ops) and chr(ops[lead]) == "D":
            lead += 1
        sc = _rescore("fit", p, ops[lead:], r.r1[lead:], r.r2[lead:]) + lead * p.e
        if lead and lead < len(ops) and False:
            pass
        assert sc == r.score, (c, r)
        n += 1
    assert n >= 200


def _stored_reference_cases(mode):
    """The compiled reference's answers kept in tests/golden/fuzz_vectors.json for one mode variant."""
    return [c for c in load_fuzz() if ("fitjump" if c["jump"] else c["mode"]) == mode]


def _port_batch_vs_stored_reference(oracle_mod, mode):
    cases = _stored_reference_cases(mode)
    assert len(cases) >= 100
    for c in cases:
        s1, s2 = c["s1"].encode("latin-1"), c["s2"].encode("latin-1")
        qb, qo, ql = pack_batch([s1])
        tb, to, tl = pack_batch([s2])
        sa = so = None
        if c["jump"]:
            sites = c["sites"] or []
            sa = np.array(sites + [0], dtype=np.int32)
            so = np.array([0, len(sites)], dtype=np.uint64)
        p = oracle_mod.Params(c["m"], c["u"], c["o"], c["e"], c["j"], bool(c["jump"]))
        a = oracle_mod.port_batch(c["mode"], p, qb, qo, ql, tb, to, tl, sa, so, threads=2)
        assert int(a.score[0]) == c["score"], c
        if c["mode"] != "edit":
            assert a.aln(0) == (c["r1"].encode("latin-1"), c["r2"].encode("latin-1")), c


@pytest.mark.parametrize("mode", ["global", "local", "fit", "fitjump", "overlap", "edit"])
def test_port_matches_live_reference(oracle_mod, mode):
    """The port's batch entry point against the reference: live on random batches where oracle/_ref was built,
    otherwise against the reference's stored answers for this mode."""
    if not oracle_mod.have_ref():
        _port_batch_vs_stored_reference(oracle_mod, mode)
        return
    rng = random.Random(hash(mode) & 0xffff)
    q, t, sites, site_off = [], [], [], [0]
    for _ in range(120):
        l1 = rng.randint(1, 200)
        s1 = bytes(rng.choice(b"ACGT") for _ in range(l1))
        mut = bytearray()
        for ch in s1:
            r = rng.random()
            if r < 0.08:
                mut.append(rng.choice(b"ACGT"))
            elif r < 0.11:
                continue
            elif r < 0.14:
                mut.append(ch); mut.append(rng.choice(b"ACGT"))
            else:
                mut.append(ch)
        s2 = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 150))) + bytes(mut) + \
            bytes(rng.choice(b"ACGT") for _ in range(rng.randint(1, 150)))
        if mode.startswith("fit") and len(s1) > len(s2):
            s1, s2 = s2, s1
        q.append(s1); t.append(s2)
        ss = sorted(rng.randrange(len(s2)) for _ in range(rng.choice([0, 2, 6])))
        sites += ss; site_off.append(len(sites))
    p = oracle_mod.Params(m=2, u=-3, o=-4, e=-1, j=-6, jump=(mode == "fitjump"))
    md = "fit" if mode == "fitjump" else mode
    qb, qo, ql = pack_batch(q)
    tb, to, tl = pack_batch(t)
    sa = np.array(sites + [0], dtype=np.int32) if mode == "fitjump" else None
    so = np.array(site_off, dtype=np.uint64) if mode == "fitjump" else None
    a = oracle_mod.port_batch(md, p, qb, qo, ql, tb, to, tl, sa, so, threads=2)
    b = oracle_mod.ref_batch(md, p, qb, qo, ql, tb, to, tl, sa, so, threads=2)
    assert np.array_equal(a.score, b.score)
    if md != "edit":
        for k in range(len(q)):
            assert a.aln(k) == b.aln(k), k


def test_port_medium_vs_reference(oracle_mod):
    """One 2 000 x 6 000 fit+jump pair and one 3 000 x 3 000 overlap pair vs the reference."""
    if not oracle_mod.have_ref():
        pytest.skip("oracle/_ref not built")
    rng = np.random.default_rng(7)
    tgt = rng.choice(np.frombuffer(b"ACGT", np.uint8), 6000).tobytes()
    read = tgt[500:1500] + tgt[3000:4000]
    p = oracle_mod.Params(1, -2, -5, -1, -10, True)
    sites = [1499, 1500, 2999, 3000]
    a = oracle_mod.port_align("fit", read, tgt, p, sites)
    b = oracle_mod.ref_align("fit", read, tgt, p, sites)
    assert (a.score, a.r1, a.r2) == (b.score, b.r1, b.r2)
    assert a.ops.count(b"N") > 0
    s1 = rng.choice(np.frombuffer(b"ACGT", np.uint8), 3000).tobytes()
    s2 = s1[1800:] + rng.choice(np.frombuffer(b"ACGT", np.uint8), 1800).tobytes()
    p = oracle_mod.Params()
    a = oracle_mod.port_align("overlap", s1, s2, p)
    b = oracle_mod.ref_align("overlap", s1, s2, p)
    assert (a.score, a.r1, a.r2) == (b.score, b.r1, b.r2)
    assert a.score > 1000


@pytest.mark.parametrize("mode", ["global", "local", "fitjump", "overlap", "edit"])
def test_port_20kbp_vs_reference(oracle_mod, mode):
    """SURVEY.md 8(c): the port is the checker of the long-sequence GPU tests, so it is itself pinned against the
    compiled reference at the largest size the reference's 48 B/cell matrices allow here: one 20 kbp x 20 kbp pair
    per mode (fit: 16 kbp x 20 kbp, with junction sites)."""
    if not oracle_mod.have_ref():
        pytest.skip("oracle/_ref not built")
    rng = np.random.default_rng(2026 + len(mode))
    acgt = np.frombuffer(b"ACGT", np.uint8)
    l2 = 20000
    s2 = acgt[rng.integers(0, 4, l2)]
    if mode == "fitjump":                      # transcript of two "exons" of the target, 3 % substitutions
        s1 = np.concatenate([s2[1000:9000], s2[11000:19000]]).copy()
        sites = [8999, 9000, 10999, 11000, 15000]
    else:
        s1 = s2.copy()
        cut = np.sort(rng.choice(l2, 400, replace=False))
        s1 = np.delete(s1, cut[:200])                                  # 1 % deletions, 1 % insertions
        s1 = np.insert(s1, np.sort(rng.choice(s1.size, 200)), acgt[rng.integers(0, 4, 200)])
        sites = None
    sub = rng.random(s1.size) < 0.03
    s1[sub] = acgt[rng.integers(0, 4, int(sub.sum()))]
    if mode == "overlap":                      # s2's prefix overlaps s1's suffix
        s1 = np.concatenate([acgt[rng.integers(0, 4, 6000)], s1[:14000]])
    p = oracle_mod.Params(1, -2, -5, -1, -10, mode == "fitjump") if mode != "edit" else oracle_mod.Params(1, 1, -5, -1, -10, False)
    md = "fit" if mode == "fitjump" else mode
    a = oracle_mod.port_align(md, s1.tobytes(), s2.tobytes(), p, sites)
    b = oracle_mod.ref_align(md, s1.tobytes(), s2.tobytes(), p, sites)
    assert a.score == b.score
    if md != "edit":
        assert (a.r1, a.r2) == (b.r1, b.r2)
        assert len(a.r1) > 10000
    if mode == "fitjump":
        assert a.ops.count(b"N") > 1000


def test_port_whitelist_mode_is_blacklist_of_the_complement(oracle_mod):
    """SURVEY.md 8(f) #3: the "intended" junction semantics (src/alignment.h:542-544: entering J only AT the listed
    target indices).  The reference cannot run it, but it is its own blacklist mode on the complement of the list --
    which pins the port's whitelist restatement on the compiled reference (live where oracle/_ref was built,
    otherwise on the reference's stored fit -s answers, whose site lists are blacklists)."""
    if not oracle_mod.have_ref():
        n_jump = 0
        for c in _stored_reference_cases("fitjump"):
            s1, s2 = c["s1"].encode("latin-1"), c["s2"].encode("latin-1")
            black = set(c["sites"] or [])
            white = [x for x in range(len(s2)) if x not in black]
            w = oracle_mod.port_align("fit", s1, s2, oracle_mod.Params(c["m"], c["u"], c["o"], c["e"], c["j"], jump=2), white)
            assert (w.score, w.r1, w.r2) == (c["score"], c["r1"].encode("latin-1"), c["r2"].encode("latin-1")), c
            n_jump += w.ops.count(b"N") > 0
        assert n_jump > 20
        return
    rng = random.Random(8)
    n_jump = 0
    for k in range(120):
        l2 = rng.randint(30, 220)
        s2 = bytes(rng.choice(b"ACGT") for _ in range(l2))
        a, b = sorted(rng.sample(range(5, l2 - 5), 2))
        s1 = (s2[max(0, a - rng.randint(3, 25)):a] + s2[b:b + rng.randint(3, 25)]) or b"A"      # two "exons" around an "intron"
        s1 = bytes(c if rng.random() > 0.05 else rng.choice(b"ACGT") for c in s1)
        white = sorted(set([a, b - 1, b] + [rng.randrange(l2) for _ in range(rng.choice([0, 2, 5]))]))
        black = [x for x in range(l2) if x not in white]
        prm = dict(m=rng.randint(1, 4), u=rng.randint(-4, -1), o=rng.randint(-8, -2), e=rng.randint(-3, -1), j=rng.randint(-12, -2))
        w = oracle_mod.port_align("fit", s1, s2, oracle_mod.Params(**prm, jump=2), white)
        r = oracle_mod.ref_align("fit", s1, s2, oracle_mod.Params(**prm, jump=True), black)
        assert (w.score, w.r1, w.r2) == (r.score, r.r1, r.r2), (k, prm, s1, s2, white)
        n_jump += w.ops.count(b"N") > 0
    assert n_jump > 20
