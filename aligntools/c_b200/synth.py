"""Synthetic workloads of BASELINE.json / SURVEY.md 8(d): uniform random ACGT, reads derived
from their targets so that alignments are non-trivial.  Deterministic: numpy PCG64 seeded with
0xA11C0000 + config id (+ rank for weak scaling).  All generators return byte batches
(uint8 concat, uint64 offsets, uint32 lengths) for both sides."""
from __future__ import annotations

import numpy as np

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
SEED0 = 0xA11C0000


def _rng(cfg, stream=0):
    return np.random.default_rng([SEED0 + cfg, stream])


def _fixed_batch(mat):
    n, L = mat.shape
    off = (np.arange(n, dtype=np.uint64) * np.uint64(L))
    lens = np.full(n, L, dtype=np.uint32)
    return np.ascontiguousarray(mat.reshape(-1)), off, lens


def _ragged_batch(seqs):
    lens = np.fromiter((len(s) for s in seqs), dtype=np.uint32, count=len(seqs))
    off = np.zeros(len(seqs), dtype=np.uint64)
    if len(seqs) > 1:
        np.cumsum(lens[:-1], out=off[1:])
    return np.ascontiguousarray(np.concatenate(seqs)), off, lens


# the two protein records of the reference's test/test_global.fa (BASELINE.json configs[0]); the same strings
# are kept with their md5 in tests/golden/cli_vectors.json
C1_S1 = b"PAKKFQIFWEKQHMIYHFTFIYVDTLICILFIVAKAGTLRFEHPHSWCRHVVDYSIGNYWSVWTVNEAYRSG"
C1_S2 = b"PAKKLCHDCTDPIVWEKQHMIYHFTFIYVDTLICILFIVAKAGTLRDEHPVSWCRHVVEDYSIGNYWSVWTVNEAYRSG"


def config1_global(n_pairs=1):
    """C1: global alignment of test/test_global.fa with -m 1 -u -1 -o -4 -e -1 (72 x 79, protein bytes)."""
    q, qo, ql = _ragged_batch([np.frombuffer(C1_S1, np.uint8)] * n_pairs)
    t, to, tl = _ragged_batch([np.frombuffer(C1_S2, np.uint8)] * n_pairs)
    return dict(mode="global", params=dict(m=1, u=-1, o=-4, e=-1, j=-10, jump=False),
                q=q, q_off=qo, q_len=ql, t=t, t_off=to, t_len=tl, sites=None, site_off=None)


def config2_local(n_pairs=1 << 20, l1=150, l2=500, stream=0):
    """C2: local, reads of l1 bp against l2 bp target windows: read = window of the target with
    4 % substitutions, 1 % insertions, 1 % deletions; 10 % of the pairs are unrelated."""
    rng = _rng(2, stream)
    tgt = rng.integers(0, 4, size=(n_pairs, l2), dtype=np.uint8)
    span = l1 + 16
    w = rng.integers(0, max(1, l2 - span), size=n_pairs)
    ev = rng.random((n_pairs, l1), dtype=np.float32)
    ins = ev < 0.01
    dele = (ev >= 0.01) & (ev < 0.02)
    adv = np.ones((n_pairs, l1), dtype=np.int32)
    adv[ins] = 0
    adv[dele] = 2
    src = np.cumsum(adv, axis=1) - adv + dele.astype(np.int32) + w[:, None]
    np.clip(src, 0, l2 - 1, out=src)
    reads = np.take_along_axis(tgt, src, axis=1)
    rnd = rng.integers(0, 4, size=(n_pairs, l1), dtype=np.uint8)
    reads[ins] = rnd[ins]
    sub = rng.random((n_pairs, l1), dtype=np.float32) < 0.04
    reads[sub] = (reads[sub] + 1 + rnd[sub] % 3) % 4
    unrelated = rng.random(n_pairs) < 0.10
    reads[unrelated] = rng.integers(0, 4, size=(int(unrelated.sum()), l1), dtype=np.uint8)
    q, qo, ql = _fixed_batch(ACGT[reads])
    t, to, tl = _fixed_batch(ACGT[tgt])
    return dict(mode="local", params=dict(m=2, u=-2, o=-5, e=-2, j=-10, jump=False),
                q=q, q_off=qo, q_len=ql, t=t, t_off=to, t_len=tl, sites=None, site_off=None)


def config3_fit_jump(n_pairs=64, l1=2000, l2=20000, stream=0):
    """C3: fit -s -j -10: two-gene target (geneA + geneB, 4-6 exons of 150-400 bp each),
    transcript = exons of A (prefix) + exons of B (suffix), 2 % substitutions; sites = intron
    start / end-exclusive indices as in test/test_fit.fa's header."""
    rng = _rng(3, stream)
    reads, tgts, sites, site_off = [], [], [], [0]
    half = l2 // 2
    for _ in range(n_pairs):
        tgt = rng.integers(0, 4, size=l2, dtype=np.uint8)
        exons = []
        st = []
        for g in range(2):
            ne = int(rng.integers(4, 7))
            lens = rng.integers(150, 401, size=ne)
            gaps_total = half - int(lens.sum()) - 20
            cuts = np.sort(rng.integers(0, max(1, gaps_total), size=ne))
            pos = g * half + 10
            prev = 0
            for k in range(ne):
                pos += int(cuts[k] - prev)
                prev = int(cuts[k])
                exons.append((pos, pos + int(lens[k])))
                pos += int(lens[k])
        # junction list: every exon end (intron start) and exon start (intron end, exclusive)
        for a, b in exons:
            st.append(b)
            st.append(a)
        tx = np.concatenate([tgt[a:b] for a, b in exons])
        if tx.size >= l1:
            lo = int(rng.integers(0, tx.size - l1 + 1))
            tx = tx[lo:lo + l1]
        else:
            tx = np.concatenate([tx, rng.integers(0, 4, size=l1 - tx.size, dtype=np.uint8)])
        sub = rng.random(l1) < 0.02
        tx = tx.copy()
        tx[sub] = (tx[sub] + 1 + rng.integers(0, 3, size=int(sub.sum()))) % 4
        reads.append(ACGT[tx])
        tgts.append(ACGT[tgt])
        st = sorted(set(int(x) for x in st if 0 <= x < l2))
        sites += st
        site_off.append(len(sites))
    q, qo, ql = _ragged_batch(reads)
    t, to, tl = _ragged_batch(tgts)
    return dict(mode="fit", params=dict(m=1, u=-2, o=-5, e=-1, j=-10, jump=True),
                q=q, q_off=qo, q_len=ql, t=t, t_off=to, t_len=tl,
                sites=np.array(sites + [0], dtype=np.int32), site_off=np.array(site_off, dtype=np.uint64))


def _mutate(rng, s, sub, ins, dele):
    ev = rng.random(s.size)
    keep = ev >= dele
    out = s[keep].copy()
    evk = ev[keep]
    m = (evk >= dele) & (evk < dele + sub)
    out[m] = (out[m] + 1 + rng.integers(0, 3, size=int(m.sum()))) % 4
    n_ins = int(rng.binomial(out.size, ins))
    if n_ins:
        pos = np.sort(rng.integers(0, out.size + 1, size=n_ins))
        out = np.insert(out, pos, rng.integers(0, 4, size=n_ins, dtype=np.uint8))
    return out


def config4_overlap(n_pairs=32, lo=10000, hi=20000, stream=0, with_diag=False):
    """C4: overlap (defaults m=1 u=-2 o=-5): s2's prefix is a mutated (5 % sub, 2.5 % ins,
    2.5 % del) copy of a suffix of s1.  with_diag: the result also carries `diag`, each pair's true start
    diagonal -(l1 - ov) (int32; what a seed chain would give a banded overlap alignment)."""
    rng = _rng(4, stream)
    reads, tgts, diag = [], [], []
    for _ in range(n_pairs):
        l1 = int(rng.integers(lo, hi + 1))
        l2 = int(rng.integers(lo, hi + 1))
        s1 = rng.integers(0, 4, size=l1, dtype=np.uint8)
        ov = int(rng.integers(min(2000, lo // 5), min(l1, l2) + 1))
        pre = _mutate(rng, s1[l1 - ov:], 0.05, 0.025, 0.025)[:l2]
        s2 = np.concatenate([pre, rng.integers(0, 4, size=max(0, l2 - pre.size), dtype=np.uint8)])
        reads.append(ACGT[s1])
        tgts.append(ACGT[s2])
        diag.append(-(l1 - ov))
    q, qo, ql = _ragged_batch(reads)
    t, to, tl = _ragged_batch(tgts)
    out = dict(mode="overlap", params=dict(m=1, u=-2, o=-5, e=-1, j=-10, jump=False),
               q=q, q_off=qo, q_len=ql, t=t, t_off=to, t_len=tl, sites=None, site_off=None)
    if with_diag:
        out["diag"] = np.array(diag, dtype=np.int32)
    return out


def config5_edit(n_pairs=8, length=100000, stream=0):
    """C5: edit -u 1: s2 = s1 with 5 % sub, 2.5 % ins, 2.5 % del, re-trimmed to `length`."""
    rng = _rng(5, stream)
    reads, tgts = [], []
    for _ in range(n_pairs):
        s1 = rng.integers(0, 4, size=length, dtype=np.uint8)
        s2 = _mutate(rng, s1, 0.05, 0.025, 0.025)
        if s2.size >= length:
            s2 = s2[:length]
        else:
            s2 = np.concatenate([s2, rng.integers(0, 4, size=length - s2.size, dtype=np.uint8)])
        reads.append(ACGT[s1])
        tgts.append(ACGT[s2])
    q, qo, ql = _ragged_batch(reads)
    t, to, tl = _ragged_batch(tgts)
    return dict(mode="edit", params=dict(m=1, u=1, o=-5, e=-1, j=-10, jump=False),
                q=q, q_off=qo, q_len=ql, t=t, t_off=to, t_len=tl, sites=None, site_off=None)


def long_global(n_pairs=256, lo=10000, hi=20000, stream=0):
    """Long global pairs (defaults m=1 u=-2 o=-5 e=-1): s1 random of lo..hi bp, s2 a mutated full-length copy of it (1 %
    substitutions, 1 % insertions, 1 % deletions) -- a read against its reference window, or one assembly against
    another.  The path keeps close to the diagonals between 0 and l2 - l1: global_corridor() gives a band around them."""
    rng = _rng(6, stream)
    reads, tgts = [], []
    for _ in range(n_pairs):
        s1 = rng.integers(0, 4, size=int(rng.integers(lo, hi + 1)), dtype=np.uint8)
        reads.append(ACGT[s1])
        tgts.append(ACGT[_mutate(rng, s1, 0.01, 0.01, 0.01)])
    q, qo, ql = _ragged_batch(reads)
    t, to, tl = _ragged_batch(tgts)
    return dict(mode="global", params=dict(m=1, u=-2, o=-5, e=-1, j=-10, jump=False),
                q=q, q_off=qo, q_len=ql, t=t, t_off=to, t_len=tl, sites=None, site_off=None)


def global_corridor(q_len, t_len, w):
    """Per-pair band (lo, hi) = (min(0, l2 - l1) - w, max(0, l2 - l1) + w) as int32 arrays: the diagonals between the
    start and the end cell of a global alignment, widened by w on both sides."""
    d = t_len.astype(np.int64) - q_len.astype(np.int64)
    return (np.minimum(0, d) - w).astype(np.int32), (np.maximum(0, d) + w).astype(np.int32)


def global_short(n_pairs=4096, l1=150, l2=150, stream=0):
    """Extra parity workload: global, l1 x l2 with ~8 % divergence."""
    rng = _rng(1, stream)
    reads, tgts = [], []
    for _ in range(n_pairs):
        s2 = rng.integers(0, 4, size=l2, dtype=np.uint8)
        s1 = _mutate(rng, s2, 0.04, 0.02, 0.02)[:l1]
        if s1.size == 0:
            s1 = s2[:1]
        reads.append(ACGT[s1])
        tgts.append(ACGT[s2])
    q, qo, ql = _ragged_batch(reads)
    t, to, tl = _ragged_batch(tgts)
    return dict(mode="global", params=dict(m=1, u=-1, o=-4, e=-1, j=-10, jump=False),
                q=q, q_off=qo, q_len=ql, t=t, t_off=to, t_len=tl, sites=None, site_off=None)
