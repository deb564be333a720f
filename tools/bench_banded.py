"""Banded overlap alignment on the C4 shape (BASELINE config 4: 10-20 kbp overlap pairs), one JSON line on stdout.

Legs on the same 256 pairs (config4_overlap(n_pairs=256, stream=0, with_diag=True)), run in turn step after step:
unbanded; banded with half-widths 64, 256 and 1024 around each pair's true start diagonal; score-only unbanded and +-256.
Per leg: fill and traceback device ms (medians over the steps), the band cells and GCUPS over them, the speed-up over
the unbanded leg of the same output kind, and the fraction of pairs whose banded result (score, end and begin cells,
CIGAR) equals the unbanded one.  Then one banded +-256 at_batch_align_banded pass over the full 10 000-pair C4.
The GPU's name and power limit are read (nvidia-smi --query-gpu, read-only) in the same run.

    python tools/bench_banded.py [--steps 7] [--warmup 2] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import aligntools.c_b200 as A              # noqa: E402
from aligntools.c_b200 import synth        # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return dict(gpu=name, power_limit=power)
    except Exception as e:      # the numbers stay valid; say what could not be read
        return dict(gpu="unknown", power_limit="unknown", nvidia_smi_error=str(e))


def same_as(res, ref, k, cigar):
    if (res.score[k], res.end_i[k], res.end_j[k], res.beg_i[k], res.beg_j[k]) != (ref.score[k], ref.end_i[k], ref.end_j[k], ref.beg_i[k], ref.beg_j[k]):
        return False
    return not cigar or np.array_equal(res.cigar_ops(k), ref.cigar_ops(k))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--pairs", type=int, default=256)
    ap.add_argument("--full-pairs", type=int, default=10000, help="pairs of the one-shot pass (BASELINE C4: 10 000)")
    ap.add_argument("--out")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    info = gpu_info()
    w = synth.config4_overlap(n_pairs=a.pairs, stream=0, with_diag=True)
    opt = A.Opt(**w["params"])
    diag = w["diag"].astype(np.int64)
    al = A.Aligner(devices=[0])
    legs = [("unbanded", None, A.OUT_CIGAR), ("band64", 64, A.OUT_CIGAR), ("band256", 256, A.OUT_CIGAR),
            ("band1024", 1024, A.OUT_CIGAR), ("unbanded_score", None, 0), ("band256_score", 256, 0)]
    batches = {}
    for name, hw, flags in legs:
        band = None if hw is None else ((diag - hw).astype(np.int32), (diag + hw).astype(np.int32))
        batches[name] = al.batch("overlap", opt, w["q"], w["q_off"], w["q_len"], w["t"], w["t_off"], w["t_len"], out_flags=flags, band=band)
    times = {name: [] for name, _, _ in legs}
    last = {}
    for step in range(a.warmup + a.steps):
        for name, _, _ in legs:                  # the legs alternate: drifts of the shared machine hit them alike
            tm = batches[name].run()
            if step >= a.warmup:
                times[name].append(tm)
    results = {name: batches[name].fetch() for name, _, _ in legs}
    for b in batches.values():
        b.free()
    out = dict(tool="bench_banded", shape="C4 overlap 10-20 kbp", pairs=a.pairs, steps=a.steps, warmup=a.warmup, **info, legs={})
    base = {}
    for name, hw, flags in legs:
        ts = times[name]
        fill = float(np.median([t.fill_ms for t in ts]))
        tb = float(np.median([t.traceback_ms for t in ts]))
        cells = int(ts[0].cells)
        ref_name = "unbanded" if flags else "unbanded_score"
        if hw is None:
            base[ref_name] = (fill, fill + tb)
        bf, bt = base[ref_name]
        res, ref = results[name], results[ref_name]
        ident = sum(same_as(res, ref, k, bool(flags)) for k in range(a.pairs)) / a.pairs
        out["legs"][name] = dict(half_width=hw, cigar=bool(flags), fill_ms=round(fill, 3), traceback_ms=round(tb, 3), cells=cells,
                                 gcups=round(cells / fill / 1e6, 1), ptr_bytes=int(ts[0].ptr_bytes),
                                 fill_speedup=round(bf / fill, 2), total_speedup=round(bt / (fill + tb), 2), identical_to_unbanded=ident)
    # one banded +-256 one-shot pass over BASELINE's full C4
    wf = synth.config4_overlap(n_pairs=a.full_pairs, stream=0, with_diag=True)
    df = wf["diag"].astype(np.int64)
    band = ((df - 256).astype(np.int32), (df + 256).astype(np.int32))
    t0 = time.perf_counter()
    res = al.align_arrays("overlap", opt, wf["q"], wf["q_off"], wf["q_len"], wf["t"], wf["t_off"], wf["t_len"], out_flags=A.OUT_CIGAR,
                          band=band, cigar_cap=1 << 26)
    wall = time.perf_counter() - t0
    tm = res.timing
    out["full_c4_band256"] = dict(pairs=a.full_pairs, wall_s=round(wall, 3), fill_ms=round(tm.fill_ms, 2), traceback_ms=round(tm.traceback_ms, 2),
                                  device_ms=round(tm.device_ms, 2), cells=int(tm.cells), gcups_fill=round(tm.cells / tm.fill_ms / 1e6, 1),
                                  ptr_bytes=int(tm.ptr_bytes), launches=int(tm.launches), ops=int(res.cigar_off[-1]))
    al.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
