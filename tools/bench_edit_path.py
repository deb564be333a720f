"""Edit distance paths (AT_OUT_EDIT_PATH) against score-only edit runs, one JSON line on stdout.

Legs, each a score-only batch and a path batch (CIGAR | ALN | EDIT_PATH) of the same pairs, run in turn step after step:
  c5     BASELINE C5: 8 pairs of 100 kbp x 100 kbp, u = 1, 2-bit input (the bit-parallel kernel);
  short  65 536 pairs of 150 x 500 (the C2 reads and windows), u = 1 (bit-parallel);
  cell   2 048 pairs of 10 kbp x 10 kbp (C5's generator), u = 2 (the cell-by-cell kernel).
Per leg and output kind: fill and traceback device ms (medians over the steps), GCUPS of the fill, pointer bytes, the
fill kernel, and the path's fill time over the score-only one.  The GPU's name and power limit are read (nvidia-smi
--query-gpu, read-only) in the same run.

    python tools/bench_edit_path.py [--steps 5] [--warmup 1] [--legs c5 short cell] [--out FILE]
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

PATH = A.OUT_CIGAR | A.OUT_ALN | A.OUT_EDIT_PATH


def workload(leg):
    if leg == "c5":
        w = synth.config5_edit(n_pairs=8)
        q2, qo2, _ = A.pack_2bit(w["q"], w["q_off"], w["q_len"], align=16)
        t2, to2, _ = A.pack_2bit(w["t"], w["t_off"], w["t_len"], align=16)
        return dict(u=1, encoding=A.SEQ_2BIT, arrays=(q2, qo2, w["q_len"], t2, to2, w["t_len"]), shape="8 x 100 kbp^2, 2-bit")
    if leg == "short":
        w = synth.config2_local(n_pairs=65536)
        return dict(u=1, encoding=A.SEQ_BYTES, arrays=(w["q"], w["q_off"], w["q_len"], w["t"], w["t_off"], w["t_len"]), shape="65536 x 150 x 500")
    w = synth.config5_edit(n_pairs=2048, length=10000)
    return dict(u=2, encoding=A.SEQ_BYTES, arrays=(w["q"], w["q_off"], w["q_len"], w["t"], w["t_off"], w["t_len"]), shape="2048 x 10 kbp^2")


def run_leg(al, leg, steps, warmup):
    w = workload(leg)
    opt = A.Opt(u=w["u"])
    kinds = (("score_only", 0), ("path", PATH))
    batches = {k: al.batch("edit", opt, *w["arrays"], out_flags=f, encoding=w["encoding"]) for k, f in kinds}
    times = {k: [] for k, _ in kinds}
    for step in range(warmup + steps):
        for k, _ in kinds:                       # alternate: drifts of the shared machine hit both alike
            tm = batches[k].run()
            if step >= warmup:
                times[k].append(tm)
    res = {k: batches[k].fetch() for k, _ in kinds}
    for b in batches.values():
        b.free()
    out = dict(shape=w["shape"], u=w["u"], scores_equal=bool(np.array_equal(res["score_only"].score, res["path"].score)))
    for k, _ in kinds:
        ts = times[k]
        fill = float(np.median([t.fill_ms for t in ts]))
        out[k] = dict(fill_ms=round(fill, 3), traceback_ms=round(float(np.median([t.traceback_ms for t in ts])), 3),
                      cells=int(ts[0].cells), gcups=round(ts[0].cells / fill / 1e6, 1), ptr_bytes=int(ts[0].ptr_bytes),
                      fill_kernel_kind=int(ts[0].fill_kernel_kind), fill_kernel_rows=int(ts[0].fill_kernel_rows))
    out["path_fill_over_score_only"] = round(out["path"]["fill_ms"] / out["score_only"]["fill_ms"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--legs", nargs="+", default=["c5", "short", "cell"], choices=["c5", "short", "cell"])
    ap.add_argument("--out")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    out = dict(tool="bench_edit_path", steps=a.steps, warmup=a.warmup, **gpu_info())
    al = A.Aligner(devices=[0])
    out["legs"] = {leg: run_leg(al, leg, a.steps, a.warmup) for leg in a.legs}
    al.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
