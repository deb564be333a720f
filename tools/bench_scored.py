"""Substitution-matrix scoring against match / mismatch scoring on the same pairs, one JSON line on stdout.

Legs, each a scored batch (at_batch_create_scored) and an unscored batch (at_batch_create) of the same pairs, run in turn
step after step (alternating: drifts of the shared machine hit both alike):
  c2_identity  BASELINE C2 (local, 150 x 500, 2-bit input), the m / u table: the profile variant of K1's packed lanes;
  c2_tstv      the same pairs, a DNA table with transitions scored above transversions;
  c2_n         C2 with about 1 % N in the targets, byte input, a ts/tv table with N neutral: 5 target bytes, the table variant
               (int32 lanes; the unscored batch runs packed lanes, so a third arm runs it on int32 lanes too, AT_NO_P16);
  protein      2 048 global pairs of 1 kbp x 1 kbp over a 20-letter alphabet, a random symmetric table: K2's table variant;
  c4_overlap   BASELINE C4 (overlap, 10-20 kbp), the ts/tv table: K2's single-plane profile variant.
Per leg: fill device ms of both (medians over the steps), GCUPS, the fill kernel, and scored over unscored.  The GPU's name
and power limit are read (nvidia-smi --query-gpu, read-only) in the same run.

    python tools/bench_scored.py [--steps 5] [--warmup 1] [--legs ...] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import aligntools.c_b200 as A              # noqa: E402
from aligntools.c_b200 import synth        # noqa: E402
from bench_banded import gpu_info          # noqa: E402

LEGS = ["c2_identity", "c2_tstv", "c2_n", "protein", "c4_overlap"]
PROTEIN = b"ACDEFGHIKLMNPQRSTVWY"
# transitions (A<->G, C<->T) -1, transversions -3, match +2; N scores 0 against everything
TSTV = A.scoring_matrix("ACGTN", [[2, -3, -1, -3, 0], [-3, 2, -3, -1, 0], [-1, -3, 2, -3, 0], [-3, -1, -3, 2, 0], [0] * 5])


def c2(n_pairs, two_bit, n_frac=0.0):
    w = synth.config2_local(n_pairs=n_pairs)
    t = w["t"].copy()
    if n_frac:
        rng = np.random.default_rng(12)
        t[rng.random(t.size) < n_frac] = ord("N")
    arrays = (w["q"], w["q_off"], w["q_len"], t, w["t_off"], w["t_len"])
    if two_bit:
        q2, qo2, _ = A.pack_2bit(w["q"], w["q_off"], w["q_len"], align=16)
        t2, to2, _ = A.pack_2bit(t, w["t_off"], w["t_len"], align=16)
        arrays = (q2, qo2, w["q_len"], t2, to2, w["t_len"])
    return arrays


def workload(leg, n_c2):
    if leg in ("c2_identity", "c2_tstv"):
        opt = A.Opt()
        mat = A.identity_scoring(opt.m, opt.u) if leg == "c2_identity" else TSTV
        return dict(mode="local", opt=opt, arrays=c2(n_c2, True), encoding=A.SEQ_2BIT, matrix=mat, shape=f"{n_c2} x 150 x 500, 2-bit")
    if leg == "c2_n":
        return dict(mode="local", opt=A.Opt(), arrays=c2(n_c2, False, 0.01), encoding=A.SEQ_BYTES, matrix=TSTV,
                    shape=f"{n_c2} x 150 x 500, 1 % N in the targets, bytes")
    if leg == "protein":
        rng = np.random.default_rng(20)
        n, L = 2048, 1000
        alpha = np.frombuffer(PROTEIN, np.uint8)
        q = alpha[rng.integers(0, 20, n * L)]
        t = q.copy()
        mut = rng.random(t.size) < 0.2
        t[mut] = alpha[rng.integers(0, 20, int(mut.sum()))]
        off = np.arange(n, dtype=np.uint64) * L
        lens = np.full(n, L, np.uint32)
        k = rng.integers(-4, 5, (20, 20))
        k = np.triu(k) + np.triu(k, 1).T
        np.fill_diagonal(k, rng.integers(4, 12, 20))
        return dict(mode="global", opt=A.Opt(m=5, u=-1, o=-10, e=-1), arrays=(q, off, lens, t.copy(), off.copy(), lens.copy()),
                    encoding=A.SEQ_BYTES, matrix=A.scoring_matrix(PROTEIN, k, -4), shape=f"{n} x {L} x {L}, 20 letters")
    w = synth.config4_overlap()
    return dict(mode="overlap", opt=A.Opt(), arrays=(w["q"], w["q_off"], w["q_len"], w["t"], w["t_off"], w["t_len"]),
                encoding=A.SEQ_BYTES, matrix=TSTV, shape="C4: 32 x 10-20 kbp")


def run_leg(al, leg, steps, warmup, n_c2):
    w = workload(leg, n_c2)
    kinds = ("unscored", "scored") + (("unscored_int32",) if leg == "c2_n" else ())
    batches = {}
    for k in kinds:
        if k == "unscored_int32":
            os.environ["AT_NO_P16"] = "1"      # read when the batch is planned
        batches[k] = al.batch(w["mode"], w["opt"], *w["arrays"], out_flags=A.OUT_CIGAR, encoding=w["encoding"],
                              scoring=w["matrix"] if k == "scored" else None)
        os.environ.pop("AT_NO_P16", None)
    times = {k: [] for k in kinds}
    for step in range(warmup + steps):
        for k in kinds:
            tm = batches[k].run()
            if step >= warmup:
                times[k].append(tm)
    res = {k: batches[k].fetch() for k in kinds}
    for b in batches.values():
        b.free()
    out = dict(shape=w["shape"], mode=w["mode"])
    if leg == "c2_identity":
        out["identity_scores_equal"] = bool(np.array_equal(res["scored"].score, res["unscored"].score))
    for k in kinds:
        ts = times[k]
        fill = float(np.median([t.fill_ms for t in ts]))
        out[k] = dict(fill_ms=round(fill, 3), fill_ms_all=[round(t.fill_ms, 3) for t in ts], cells=int(ts[0].cells),
                      gcups=round(ts[0].cells / fill / 1e6, 1), fill_kernel_kind=int(ts[0].fill_kernel_kind),
                      fill_kernel_flags=int(ts[0].fill_kernel_flags))
    out["scored_over_unscored"] = round(out["scored"]["fill_ms"] / out["unscored"]["fill_ms"], 3)
    if "unscored_int32" in out:
        out["scored_over_unscored_int32"] = round(out["scored"]["fill_ms"] / out["unscored_int32"]["fill_ms"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--legs", nargs="+", default=LEGS, choices=LEGS)
    ap.add_argument("--c2-pairs", type=int, default=1 << 18)
    ap.add_argument("--out")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    out = dict(tool="bench_scored", steps=a.steps, warmup=a.warmup, metric="fill device ms, median over steps", **gpu_info())
    al = A.Aligner(devices=[0])
    out["legs"] = {leg: run_leg(al, leg, a.steps, a.warmup, a.c2_pairs) for leg in a.legs}
    al.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
