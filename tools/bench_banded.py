"""Banded alignment on long pairs, one JSON line on stdout.

--mode overlap (default): the C4 shape (BASELINE config 4: 10-20 kbp overlap pairs).  Legs on the same 256 pairs
(config4_overlap(n_pairs=256, stream=0, with_diag=True)), run in turn step after step: unbanded; banded with half-widths
64, 256 and 1024 around each pair's true start diagonal; score-only unbanded and +-256.  Then one banded +-256
at_batch_align_banded pass over the full 10 000-pair C4.

--mode global: synth.long_global (10-20 kbp global pairs, s2 a 1 % sub / ins / del copy of s1), at 256 and at 2 048
pairs: at 256 pairs banded overlap was latency-bound (DESIGN.md section 5), the larger count shows whether more resident
stripes move that.  The same legs, with corridor bands [min(0, l2 - l1) - w, max(0, l2 - l1) + w] for w = 64, 256, 1024
(synth.global_corridor).  Then one banded w = 256 at_batch_align_banded pass over 10 000 pairs.

Per leg: fill and traceback device ms (medians over the steps), the band cells and GCUPS over them, pointer bytes, the
speed-up over the unbanded leg of the same output kind, and the fraction of pairs whose banded result (score, end and
begin cells, CIGAR) equals the unbanded one.  The GPU's name and power limit are read (nvidia-smi --query-gpu,
read-only) in the same run.

    python tools/bench_banded.py [--mode overlap|global] [--steps 7] [--warmup 2] [--pairs N ...] [--out FILE]
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


LEGS = [("unbanded", None, A.OUT_CIGAR), ("band64", 64, A.OUT_CIGAR), ("band256", 256, A.OUT_CIGAR),
        ("band1024", 1024, A.OUT_CIGAR), ("unbanded_score", None, 0), ("band256_score", 256, 0)]


def band_of(mode, w, hw):
    """overlap: +-hw around the true start diagonal; global: the corridor between the start and the end diagonal, +-hw"""
    if mode == "global":
        return synth.global_corridor(w["q_len"], w["t_len"], hw)
    diag = w["diag"].astype(np.int64)
    return (diag - hw).astype(np.int32), (diag + hw).astype(np.int32)


def workload(mode, n_pairs):
    return synth.long_global(n_pairs=n_pairs, stream=0) if mode == "global" else synth.config4_overlap(n_pairs=n_pairs, stream=0, with_diag=True)


def run_legs(al, mode, w, n_pairs, steps, warmup):
    """The legs on one batch of pairs, alternating step after step; returns {leg: stats}"""
    opt = A.Opt(**w["params"])
    legs = LEGS
    batches = {}
    for name, hw, flags in legs:
        band = None if hw is None else band_of(mode, w, hw)
        batches[name] = al.batch(mode, opt, w["q"], w["q_off"], w["q_len"], w["t"], w["t_off"], w["t_len"], out_flags=flags, band=band)
    times = {name: [] for name, _, _ in legs}
    last = {}
    for step in range(warmup + steps):
        for name, _, _ in legs:                  # the legs alternate: drifts of the shared machine hit them alike
            tm = batches[name].run()
            if step >= warmup:
                times[name].append(tm)
    results = {name: batches[name].fetch() for name, _, _ in legs}
    for b in batches.values():
        b.free()
    out = {}
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
        ident = sum(same_as(res, ref, k, bool(flags)) for k in range(n_pairs)) / n_pairs
        out[name] = dict(half_width=hw, cigar=bool(flags), fill_ms=round(fill, 3), traceback_ms=round(tb, 3), cells=cells,
                         gcups=round(cells / fill / 1e6, 1), ptr_bytes=int(ts[0].ptr_bytes),
                         fill_speedup=round(bf / fill, 2), total_speedup=round(bt / (fill + tb), 2), identical_to_unbanded=ident)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["overlap", "global"], default="overlap")
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--pairs", type=int, nargs="+", help="pair counts of the legs (overlap: 256; global: 256 2048)")
    ap.add_argument("--full-pairs", type=int, default=10000, help="pairs of the one-shot pass (BASELINE C4: 10 000)")
    ap.add_argument("--out")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    counts = a.pairs or ([256, 2048] if a.mode == "global" else [256])
    if a.mode == "overlap" and len(counts) != 1:
        ap.error("--mode overlap takes one --pairs count")
    info = gpu_info()
    al = A.Aligner(devices=[0])
    if a.mode == "overlap":
        out = dict(tool="bench_banded", shape="C4 overlap 10-20 kbp", pairs=counts[0], steps=a.steps, warmup=a.warmup, **info,
                   legs=run_legs(al, "overlap", workload("overlap", counts[0]), counts[0], a.steps, a.warmup))
    else:
        out = dict(tool="bench_banded", mode="global", shape="long_global 10-20 kbp, 1 % sub / ins / del", steps=a.steps, warmup=a.warmup,
                   **info, runs=[dict(pairs=n, legs=run_legs(al, "global", workload("global", n), n, a.steps, a.warmup)) for n in counts])
    # one banded +-256 one-shot pass over the full-size batch
    wf = workload(a.mode, a.full_pairs)
    t0 = time.perf_counter()
    res = al.align_arrays(a.mode, A.Opt(**wf["params"]), wf["q"], wf["q_off"], wf["q_len"], wf["t"], wf["t_off"], wf["t_len"],
                          out_flags=A.OUT_CIGAR, band=band_of(a.mode, wf, 256), cigar_cap=1 << 26)
    wall = time.perf_counter() - t0
    tm = res.timing
    out["full_c4_band256" if a.mode == "overlap" else "full_band256"] = dict(
        pairs=a.full_pairs, wall_s=round(wall, 3), fill_ms=round(tm.fill_ms, 2), traceback_ms=round(tm.traceback_ms, 2),
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
