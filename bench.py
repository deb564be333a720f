#!/usr/bin/env python
"""bench.py -- GCUPS (fill + traceback, device-timed) of the alignTools DP core on B200.

Headline workload (BASELINE.json configs[1], the configuration the metric is quoted on): batched local
(Smith-Waterman) affine-gap alignment of 1 Mi synthetic 150 bp reads against 500 bp target windows,
score + CIGAR, parameters -m 2 -u -2 -o -5 -e -2.  A "step" is one pass of the hot path (fill kernels +
device traceback) over that batch.  Weak scaling: every rank runs the full batch on its own GPU (pairs
are independent; no collective on the data path).

The same JSON line carries
  * `configs`: device-timed GCUPS, roofline fraction of the dominant kernel and the end-to-end number
    (host buffers through at_batch_align) of the OTHER BASELINE.json shapes -- C1 global 72 x 79, C3 fit
    with jump state 2 k x 20 k, C4 overlap 10-20 kbp, C5 edit 100 k x 100 k -- each timed in this run;
  * `sharded`: the multi-GPU split BASELINE.json's north star describes: ONE batch cut into contiguous
    slices by at_plan_slices, every rank aligns its slice through at_batch_align and the results are
    gathered on rank 0's host memory inside the clock (C2: 1 Mi pairs in total; C5: 64 pairs in total,
    8 per GPU at N = 8).  Strong scaling; no NCCL on the data path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--pairs P] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line on rank 0.  The oracle (oracle/) is executed only for the `cpu_baseline` objects and for
`--impl reference`; it is never on the measured GPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GCUPS (fill+traceback, device-timed)"       # BASELINE.json's metric; the SAME string in both arms
UNIT = "GCUPS"
C2_WORKLOAD = "C2 batched local SW affine: 150 bp reads vs 500 bp windows (-m 2 -u -2 -o -5 -e -2), score + CIGAR"

OPS_PER_CELL = {"global": 10, "local": 12, "fit": 10, "fitjump": 14, "overlap": 6, "edit": 6}   # SURVEY.md 8(d)
PTR_BYTES_PER_CELL = {"global": 0.5, "local": 0.5, "fit": 0.5, "fitjump": 0.625, "overlap": 0.25, "edit": 0.0}
# Integer roofline denominator (BASELINE.md 4 / SURVEY.md 8d): the ALU pipe issues 64 int32 lanes per clock per
# SM (profiles/int_peak_r02.txt: 58-59 lane-ops/clk/SM measured for VIMNMX / LOP3 / VIADDMNMX); one packed
# s16x2 instruction counts as two operations.
INT32_LANES_PER_SM = 64
N_SM = 148
# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per PAIR of the C2 batch, from the ncu
# --set full capture of ONE launch on the full 1 Mi-pair batch (see profiles/): scaled by the pairs of a launch.
NCU_TRAFFIC_BYTES_PER_PAIR = None          # filled from profiles/ncu_traffic_r02.json when present
KERNEL_KINDS = {0: "at_fill_affine<int32>", 1: "at_fill_affine<s16x2>", 2: "at_wave", 3: "at_wave_edit_bits"}


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("sm_max_mhz", 1965.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1965.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_pair():
    p = os.path.join(ROOT, "profiles", "ncu_traffic_r02.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("c2_fill_dram_bytes_per_pair"), d.get("source")
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        inside = [ln for ts, ln in self.lines if t_begin is None or (t_begin <= ts <= t_end + 0.12)]
        if not inside:                       # region shorter than one sampling period: take the sample nearest to it
            inside = [ln for ts, ln in self.lines[-1:]]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        hot = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(hot) if hot else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pinned_like(arr):
    """Copy a numpy array into pinned host memory (torch allocator) and return a numpy view."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(arr))
    try:
        t = t.pin_memory()
    except Exception:
        pass
    return t.numpy(), t


def make_workload(pairs, stream):
    from aligntools.c_b200 import synth
    return synth.config2_local(n_pairs=pairs, stream=stream)


def cpu_baseline_sample(w, n_sample, threads, kind_pref="reference"):
    """Time the reference's own CPU implementation (oracle/_ref) -- or the port when the compiled
    reference is absent -- on the first n_sample pairs of the workload."""
    import oracle
    p = oracle.Params(**{k: w["params"][k] for k in "muoej"}, jump=w["params"]["jump"])
    sl = slice(0, n_sample)
    so = w["site_off"][:n_sample + 1] if w.get("site_off") is not None else None
    args = (w["mode"], p, w["q"], w["q_off"][sl], w["q_len"][sl], w["t"], w["t_off"][sl], w["t_len"][sl])
    kw = dict(sites=w.get("sites"), site_off=so)
    cells = int((w["q_len"][sl].astype(np.uint64) * w["t_len"][sl].astype(np.uint64)).sum())
    if kind_pref == "reference" and oracle.have_ref():
        kind = "reference"
        t0 = time.perf_counter()
        out = oracle.ref_batch(*args, want_aln=True, threads=threads, **kw)
        dt = time.perf_counter() - t0
    else:
        kind = "port"
        oracle.build()
        t0 = time.perf_counter()
        out = oracle.port_batch(*args, want_aln=True, threads=threads, **kw)
        dt = time.perf_counter() - t0
    return kind, cells, dt, out


def run_reference_arm(args):
    rank, local_rank, world = env_rank()
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    w = make_workload(max(args.ref_pairs, 1024), 0)
    per_step = args.ref_pairs
    times = []
    for k in range(args.warmup + args.steps):
        kind, cells, dt, _ = cpu_baseline_sample(w, per_step, threads)
        if k >= args.warmup:
            times.append(dt)
    tot = sum(times)
    gcups = cells * len(times) / tot / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": gcups, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": C2_WORKLOAD, "pairs_per_step": per_step, "l1": 150, "l2": 500,
                   "note": "the reference's own CPU implementation (oracle/_ref, compiled from /root/reference/src) on a bounded "
                           "sample of the workload, one pthread per host core; wall-clock timed (there is no device)"},
        "cpu_baseline": {"value": gcups, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"{per_step} pairs of the C2 workload per step, one pthread per host core"},
        "e2e": {"value": gcups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def kernel_label(tm, mode_key):
    kind = KERNEL_KINDS.get(tm.fill_kernel_kind, "?")
    fl = tm.fill_kernel_flags
    return (f"{kind} mode={mode_key} rows_per_lane={tm.fill_kernel_rows}" + (" query-profile" if fl & 1 else " xor/min")
            + (" +jump" if fl & 2 else "") + (" 2-bit targets" if fl & 4 else ""))


def roofline_of(tm, mode_key, k_ms, sm_max_mhz, hbm_peak, peak_src, seq_bytes):
    """Integer-ALU roofline of the dominant fill launch (SURVEY.md 8d): algorithmic ops per cell x the cells of one
    launch / its CUDA-event duration, against 148 SM x 64 lanes x clock (x2 for packed s16x2 lanes)."""
    packed = 2 if tm.fill_kernel_kind == 1 else 1
    int_peak = N_SM * INT32_LANES_PER_SM * packed * sm_max_mhz * 1e6 / 1e12
    ops = OPS_PER_CELL[mode_key]
    achieved = tm.fill_kernel_cells * ops / (k_ms * 1e-3) / 1e12
    ptr_b = PTR_BYTES_PER_CELL[mode_key] * tm.fill_kernel_cells
    r = {"bound": "int_alu", "achieved": achieved, "peak": int_peak, "unit": "Tiop/s", "frac": achieved / int_peak,
         "traffic": None, "algorithmic_bytes": int(ptr_b) + int(seq_bytes),
         "kernel": kernel_label(tm, mode_key), "kernel_ms": k_ms, "kernel_cells": int(tm.fill_kernel_cells),
         "kernel_gcups": tm.fill_kernel_cells / (k_ms * 1e-3) / 1e9, "ops_per_cell": ops,
         "peak_note": (f"{N_SM} SM x {INT32_LANES_PER_SM} ALU lanes x {packed} ({'s16x2' if packed == 2 else 'int32'}) x "
                       f"{sm_max_mhz:.0f} MHz nominal (BASELINE.md 4); algorithmic ops/cell from SURVEY.md 8(d)"),
         "hbm": {"bound": "hbm", "achieved": ptr_b / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                 "frac": ptr_b / (k_ms * 1e-3) / 1e9 / hbm_peak, "what": "traceback-pointer writes", "peak_src": peak_src}}
    if tm.fill_kernel_kind == 3:
        r["note"] = ("bit-parallel kernel: one instruction advances 32 cells, so the fraction of the CELL-BY-CELL roofline "
                     "(6 ops per cell) exceeds 1; it is reported for comparison with the other modes only")
    return r


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(res, out_dir):
    """Write what the caller of the timed path receives (scores, start / end cells, CIGARs) as out_dir/<name>.npy, so
    that two builds run with the same arguments can be compared output for output.  When the whole result would exceed
    DUMP_MAX_BYTES, the dump is the largest prefix of a fixed, seeded permutation of the pairs that fits, in pair
    order (pair_index.npy).  Scores, cells and packed CIGAR ops are below 2^24, so float32 holds them exactly; CIGAR
    offsets are float64."""
    n = res.n
    off = res.cigar_off.astype(np.int64)
    lens_all = np.diff(off[:n + 1])
    # bytes per pair: five float32 fields, a float64 offset (and a float64 pair_index when sampled), 4 per CIGAR op;
    # the budget keeps room for the final offset and the .npy headers
    budget = DUMP_MAX_BYTES - 8 - 4096
    if 28 * n + 4 * int(lens_all.sum()) <= budget:
        idx = np.arange(n)
    else:
        perm = np.random.default_rng(0).permutation(n)
        cost = np.cumsum(36 + 4 * lens_all[perm])
        idx = np.sort(perm[:int(np.searchsorted(cost, budget, side="right"))])
    lens = lens_all[idx]
    sub_off = np.zeros(len(idx) + 1, np.int64)
    np.cumsum(lens, out=sub_off[1:])
    take = np.repeat(off[idx] - sub_off[:-1], lens) + np.arange(sub_off[-1])
    arrs = {k: getattr(res, k)[idx].astype(np.float32) for k in ("score", "end_i", "end_j", "beg_i", "beg_j")}
    arrs["cigar_off"] = sub_off.astype(np.float64)
    arrs["cigar"] = res.cigar[take].astype(np.float32)
    if len(idx) < n:
        arrs["pair_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def mode_key_of(w):
    return "fitjump" if (w["mode"] == "fit" and w["params"]["jump"]) else w["mode"]


def time_config(al, A, w, name, flags, steps, warmup, e2e_steps, peaks, barrier, encoding=0, want_e2e=True, twobit=False):
    """Device-timed GCUPS of one workload with inputs resident in HBM + the same through at_batch_align with
    host buffers (H2D / D2H inside the clock)."""
    hbm_peak, sm_max_mhz, peak_src = peaks
    opt = A.Opt(**w["params"])
    keep = []
    arrs = {}
    for k in ("q", "q_off", "q_len", "t", "t_off", "t_len", "sites", "site_off"):
        if w.get(k) is None:
            arrs[k] = None
        else:
            arrs[k], t_ = pinned_like(w[k]); keep.append(t_)
    if twobit:      # ACGT workloads: hand the sequences over as AT_SEQ_2BIT (records on 16-byte boundaries); they stay packed in HBM
        encoding = A.SEQ_2BIT
        for sq, so, sl in (("q", "q_off", "q_len"), ("t", "t_off", "t_len")):
            pk, po, _ = A.pack_2bit(w[sq], w[so], w[sl], align=16)
            arrs[sq], t_ = pinned_like(pk); keep.append(t_)
            arrs[so], t_ = pinned_like(po); keep.append(t_)
    batch = al.batch(w["mode"], opt, arrs["q"], arrs["q_off"], arrs["q_len"], arrs["t"], arrs["t_off"], arrs["t_len"],
                     sites=arrs["sites"], site_off=arrs["site_off"], out_flags=flags, encoding=encoding)
    for _ in range(warmup):
        batch.run()
    barrier()
    dev_ms = fill_ms = tb_ms = 0.0
    launches = 0
    kern_ms = []
    t0 = time.perf_counter()
    for _ in range(steps):
        tm = batch.run()
        dev_ms += tm.device_ms; fill_ms += tm.fill_ms; tb_ms += tm.traceback_ms; launches += tm.launches
        kern_ms.append(tm.fill_kernel_ms)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    res = batch.fetch()
    batch.free()
    mk = mode_key_of(w)
    seq_bytes = arrs["q"].nbytes + arrs["t"].nbytes
    k_ms = sum(kern_ms) / len(kern_ms)
    out = {"name": name, "mode": mk, "encoding": "2bit (resident)" if twobit else "bytes", "pairs": int(len(w["q_len"])), "cells": int(tm.cells), "steps": steps, "warmup": warmup,
           "value": tm.cells * steps / (dev_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": dev_ms / steps,
           "fill_ms_per_step": fill_ms / steps, "traceback_ms_per_step": tb_ms / steps, "wall_ms_per_step": wall_ms / steps,
           "gpu_launches": int(launches), "roofline": roofline_of(tm, mk, k_ms, sm_max_mhz, hbm_peak, peak_src, seq_bytes),
           "checks": {"score_sum": int(res.score.astype(np.int64).sum()),
                      "cigar_ops": int(res.cigar_off[-1]) if res.cigar_off is not None else 0}}
    raw = {"dev_ms": dev_ms, "wall_ms": wall_ms, "launches": launches, "res": res, "tm": tm, "arrs": arrs, "keep": keep}
    if want_e2e:
        h2d = sum(a.nbytes for a in arrs.values() if a is not None)
        n = len(w["q_len"])
        outb = A.BatchResult(n)
        cig_cap = None
        if flags & A.OUT_CIGAR and w["mode"] != "edit":
            cig_cap = max(2 * out["checks"]["cigar_ops"] + 1024, 1 << 16)
            outb.cigar, kc = pinned_like(np.zeros(cig_cap, np.uint32)); keep.append(kc)
            outb.cigar_off = np.zeros(n + 1, np.uint64)
        times = []
        e2e_warm = 2
        for k in range(e2e_warm + e2e_steps):
            barrier()
            t1 = time.perf_counter()
            r2 = al.align_arrays(w["mode"], opt, arrs["q"], arrs["q_off"], arrs["q_len"], arrs["t"], arrs["t_off"], arrs["t_len"],
                                 sites=arrs["sites"], site_off=arrs["site_off"], out_flags=flags, encoding=encoding,
                                 out=outb, cigar_cap=cig_cap)
            dt = time.perf_counter() - t1
            if k >= e2e_warm:
                times.append(dt)
            if os.environ.get("AT_BENCH_VERBOSE"):
                print(f"[bench] {name} e2e iteration {k}: {1e3 * dt:.2f} ms", file=sys.stderr, flush=True)
        assert np.array_equal(r2.score, res.score), f"{name}: e2e scores differ from the resident run"
        d2h = r2.score.nbytes + 4 * r2.end_i.nbytes
        if r2.cigar_off is not None and flags & A.OUT_CIGAR and w["mode"] != "edit":
            nops = int(r2.cigar_off[-1])
            assert nops == out["checks"]["cigar_ops"] and np.array_equal(r2.cigar[:nops], res.cigar[:nops]), f"{name}: e2e CIGARs differ"
            d2h += (r2.cigar_off.nbytes - 8) + nops * 4
        e2e_ms = 1e3 * sum(times) / len(times)
        out["e2e"] = {"value": tm.cells / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": e2e_ms,
                      "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                      "launches_per_step": int(r2.timing.launches)}
        raw["e2e_ms"] = e2e_ms
        raw["e2e_launches"] = int(r2.timing.launches)
    return out, raw


def sharded_leg(al, A, dist, w, name, flags, rank, world, steps, barrier, expect=None, twobit=False):
    """ONE batch, contiguous slices balanced by DP cells (at_plan_slices), each rank aligns its slice through
    at_batch_align with host buffers, results land in rank 0's host memory; all of it inside the clock."""
    n = len(w["q_len"])
    cut = A.plan_slices(w["q_len"], w["t_len"], world)
    lo, hi = int(cut[rank]), int(cut[rank + 1])
    opt = A.Opt(**w["params"])
    tb = bool(flags & A.OUT_CIGAR) and w["mode"] != "edit"
    worst = int(w["q_len"][lo:hi].astype(np.uint64).sum() + w["t_len"][lo:hi].astype(np.uint64).sum()) if tb else 0
    cap = min(worst, 40 * (hi - lo) + (1 << 16)) if tb else 1
    if world > 1:
        caps = [None] * world
        dist.all_gather_object(caps, cap)
        cap = max(caps)
    from aligntools.c_b200.sharding import HostGather
    hg = HostGather(dist, rank, world, n, cap, name, pin=True)
    keep = []
    arrs = {}
    enc = A.SEQ_BYTES
    q_off, t_off = w["q_off"], w["t_off"]
    if twobit:      # the library's input encoding for ACGT data: a quarter of the PCIe bytes, read by the fill as it is
        enc = A.SEQ_2BIT
        q2, q_off, _ = A.pack_2bit(w["q"], w["q_off"], w["q_len"], align=16)
        t2, t_off, _ = A.pack_2bit(w["t"], w["t_off"], w["t_len"], align=16)
        arrs["q"], k1 = pinned_like(q2); arrs["t"], k2 = pinned_like(t2); keep += [k1, k2]
    else:
        for k in ("q", "t"):
            arrs[k], t_ = pinned_like(w[k]); keep.append(t_)
    so = w["site_off"][lo:hi + 1] if w.get("site_off") is not None else None
    outb = hg.slice_out(lo, hi)
    full_cigar = np.zeros(cap * world + 1, np.uint32) if (rank == 0 and tb) else None
    full_off = np.zeros(n + 1, np.uint64) if rank == 0 else None
    times = []
    total_ops = 0
    for k in range(2 + steps):
        barrier()
        t1 = time.perf_counter()
        if hi > lo:
            al.align_arrays(w["mode"], opt, arrs["q"], q_off[lo:hi], w["q_len"][lo:hi], arrs["t"], t_off[lo:hi], w["t_len"][lo:hi],
                            sites=w.get("sites"), site_off=so, out_flags=flags, encoding=enc, out=outb, cigar_cap=cap if tb else None)
        barrier()                                   # every slice is in host memory
        if rank == 0 and tb:
            total_ops = hg.merge(cut, full_cigar, full_off)
        dt = time.perf_counter() - t1
        if k >= 2:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    if world > 1:
        import torch
        tt = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt[0])
    cells = int((w["q_len"].astype(np.uint64) * w["t_len"].astype(np.uint64)).sum())
    out = None
    if rank == 0:
        score_sum = int(hg.arr["score"][:n].astype(np.int64).sum())
        out = {"name": name, "pairs_total": n, "pairs_per_gpu": [int(cut[r + 1] - cut[r]) for r in range(world)], "cells": cells,
               "value": cells / (ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms, "steps": steps, "scaling": "strong",
               "gather": "rank 0 host memory (shared-memory output arrays; CIGARs concatenated in pair order), inside the clock",
               "encoding": "2bit" if twobit else "bytes",
               "checks": {"score_sum": score_sum, "cigar_ops": int(total_ops)}}
        if expect is not None:
            assert score_sum == expect["score_sum"], f"sharded {name}: score checksum differs from the single-GPU run"
            if tb:
                assert int(total_ops) == expect["cigar_ops"], f"sharded {name}: CIGAR total differs from the single-GPU run"
    barrier()
    hg.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=1 << 20, help="pairs per GPU (C2 = 1 Mi)")
    ap.add_argument("--ref-pairs", type=int, default=4096, help="pairs per step of the --impl reference arm")
    ap.add_argument("--cpu-sample", type=int, default=12000, help="pairs timed for cpu_baseline (about 14 s on one core)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1 / C3 / C4 / C5 lines")
    ap.add_argument("--no-sharded", action="store_true", help="skip the sharded (strong-scaling) legs")
    ap.add_argument("--c3-pairs", type=int, default=2048)
    ap.add_argument("--c4-pairs", type=int, default=256)
    ap.add_argument("--c5-pairs", type=int, default=8, help="C5 pairs per GPU (BASELINE: 64 pairs over 8 GPUs)")
    ap.add_argument("--cfg-steps", type=int, default=3)
    ap.add_argument("--bytes-e2e", action="store_true", help="C2 e2e leg hands over byte-encoded sequences instead of AT_SEQ_2BIT")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed C2 step's results (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)

    rank, local_rank, world = env_rank()
    import torch
    import torch.distributed as dist
    use_dist = world > 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if use_dist:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # NCCL logs (its version banner) go to stdout by default: rank 0 prints ONE JSON line there
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import aligntools.c_b200 as A
    from aligntools.c_b200 import synth
    al = A.Aligner(devices=[local_rank])
    peaks = measured_peaks()
    hbm_peak, sm_max_mhz, peak_src = peaks

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- headline: C2, inputs resident in HBM, device-timed ----------------
    w = make_workload(args.pairs, rank)
    sampler = ClockSampler(local_rank)
    sampler.start()                      # nvidia-smi needs a moment to start: begin before the warm-up, keep only the timed region
    t_begin = time.perf_counter()
    head, raw = time_config(al, A, w, "C2", A.OUT_CIGAR, args.steps, args.warmup, args.e2e_steps, peaks, barrier, want_e2e=False)
    t_end = time.perf_counter()
    clocks = sampler.stop(t_begin, t_end)
    dev_ms, wall_ms, launches, res, tm = raw["dev_ms"], raw["wall_ms"], raw["launches"], raw["res"], raw["tm"]
    if args.dump_outputs and rank == 0:
        dump_outputs(res, args.dump_outputs)
    cells = tm.cells
    if use_dist:
        tt = torch.tensor([dev_ms, wall_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms = float(tt[0]), float(tt[1])
        tl_ = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(tl_, op=dist.ReduceOp.SUM)
        launches = int(tl_[0])
    value = cells * world * args.steps / (dev_ms * 1e-3) / 1e9
    score_sum, cigar_ops = head["checks"]["score_sum"], head["checks"]["cigar_ops"]
    roofline = head["roofline"]
    traffic_pp, traffic_src = ncu_traffic_per_pair()
    if traffic_pp:
        roofline["traffic"] = traffic_pp * args.pairs
        roofline["traffic_note"] = f"ncu dram read+write of one launch ({traffic_src}), scaled by pairs"

    # ---------------- e2e: host buffers through the public C-ABI call ----------------
    # at_batch_align (one-shot): H2D of the sequences from pinned host memory, fill + traceback, D2H of scores /
    # cells / CIGARs into host buffers, all inside the timed region.  The sequences are handed over 2-bit packed
    # (AT_SEQ_2BIT, the library's input encoding for ACGT data): a quarter of the PCIe bytes.
    e2e = None
    if not args.no_e2e:
        arrs = raw["arrs"]
        enc = A.SEQ_BYTES
        q, qo, ql, t, to, tl = arrs["q"], arrs["q_off"], arrs["q_len"], arrs["t"], arrs["t_off"], arrs["t_len"]
        keep2 = []
        if not args.bytes_e2e:
            enc = A.SEQ_2BIT
            q2, qo2, _ = A.pack_2bit(w["q"], w["q_off"], w["q_len"], align=16)      # 16-byte aligned records: 128-bit loads in the fill
            t2, to2, _ = A.pack_2bit(w["t"], w["t_off"], w["t_len"], align=16)
            q, k1 = pinned_like(q2); t, k2 = pinned_like(t2); qo, k3 = pinned_like(qo2); to, k4 = pinned_like(to2)
            keep2 += [k1, k2, k3, k4]
        h2d = q.nbytes + t.nbytes + qo.nbytes + to.nbytes + ql.nbytes + tl.nbytes
        opt = A.Opt(**w["params"])
        out_bufs = A.BatchResult(args.pairs)
        cig_cap = max(2 * cigar_ops + 1024, 1 << 16)
        out_bufs.cigar, _kc = pinned_like(np.zeros(cig_cap, np.uint32))
        out_bufs.cigar_off = np.zeros(args.pairs + 1, np.uint64)
        e2e_warm = max(3, args.warmup)             # the first calls size the library's workspaces
        e2e_times = []
        for k in range(e2e_warm + args.e2e_steps):
            barrier()
            t1 = time.perf_counter()
            r2 = al.align_arrays("local", opt, q, qo, ql, t, to, tl, out_flags=A.OUT_CIGAR, encoding=enc, out=out_bufs, cigar_cap=cig_cap)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t1
            if k >= e2e_warm:
                e2e_times.append(dt)
            if os.environ.get("AT_BENCH_VERBOSE"):
                print(f"[bench] e2e iteration {k}: {1e3 * dt:.2f} ms", file=sys.stderr, flush=True)
        d2h = r2.score.nbytes + 4 * r2.end_i.nbytes + (r2.cigar_off.nbytes - 8) + int(r2.cigar_off[-1]) * 4
        e2e_ms = 1e3 * sum(e2e_times) / len(e2e_times)
        if use_dist:
            tt = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_ms = float(tt[0])
        assert int(r2.score.astype(np.int64).sum()) == score_sum and int(r2.cigar_off[-1]) == cigar_ops
        assert np.array_equal(r2.cigar[:cigar_ops], res.cigar[:cigar_ops]), "pipelined e2e CIGARs differ from the resident run"
        e2e = {"value": cells * world / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "encoding": "2bit (records on 16-byte boundaries; resident in HBM as handed over, read by the fill directly)" if enc == A.SEQ_2BIT else "bytes",
               "kernel_ms_sum": r2.timing.fill_ms + r2.timing.traceback_ms, "launches_per_step": int(r2.timing.launches),
               "api": "at_batch_align (one call: pinned host buffers in, host buffers out; sub-slices pipelined over 3 streams)"}
        del keep2

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        kind, ccells, dt, out = cpu_baseline_sample(w, args.cpu_sample, 1)
        assert np.array_equal(out.score[:args.cpu_sample], res.score[:args.cpu_sample].astype(np.int64)), "GPU/CPU score mismatch"
        cpu = {"value": ccells / dt / 1e9, "unit": UNIT, "cores": 1, "kind": kind,
               "sample": f"first {args.cpu_sample} pairs of the same C2 batch, single thread ({dt:.1f} s); scores cross-checked against the GPU run"}
    del raw, res

    # ---------------- the other BASELINE shapes, timed in the same run ----------------
    configs = []
    if not args.no_configs:
        c1 = synth.config1_global()
        shapes = [("C1 global 72x79 protein (-m 1 -u -1 -o -4 -e -1), test/test_global.fa", c1, A.OUT_CIGAR, max(args.cfg_steps, 10)),
                  (f"C3 fit -s -j -10: {args.c3_pairs} pairs 2 kbp x 20 kbp", synth.config3_fit_jump(n_pairs=args.c3_pairs, stream=rank), A.OUT_CIGAR, args.cfg_steps),
                  (f"C4 overlap: {args.c4_pairs} pairs U[10,20] kbp", synth.config4_overlap(n_pairs=args.c4_pairs, stream=rank), A.OUT_CIGAR, args.cfg_steps),
                  (f"C5 edit -u 1: {args.c5_pairs} pairs 100 kbp x 100 kbp", synth.config5_edit(n_pairs=args.c5_pairs, stream=rank), 0, args.cfg_steps)]
        for name, wc, fl, st in shapes:
            c, rw = time_config(al, A, wc, name, fl, st, 1, 2, peaks, barrier, twobit=name[:2] != "C1" and not args.bytes_e2e)
            vals = [c["value"], c["e2e"]["value"], c["ms_per_step"], c["e2e"]["ms_per_step"]]
            if use_dist:      # whole-job aggregate: ranks run replicas of the shape (weak scaling); time = max over ranks
                tt = torch.tensor([c["ms_per_step"], c["e2e"]["ms_per_step"]], device="cuda", dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                c["ms_per_step"], c["e2e"]["ms_per_step"] = float(tt[0]), float(tt[1])
                c["value"] = c["cells"] * world / (c["ms_per_step"] * 1e-3) / 1e9
                c["e2e"]["value"] = c["cells"] * world / (c["e2e"]["ms_per_step"] * 1e-3) / 1e9
            launches += c["gpu_launches"]
            # CPU reference beside it: one pair (C1: the pair; C3: the first pair), single thread, N = 1 only
            if rank == 0 and world == 1 and not args.no_cpu and name[:2] in ("C1", "C3"):
                reps = 200 if name[:2] == "C1" else 1
                t0 = time.perf_counter()
                for _ in range(reps):
                    kind, ccells, _, o1 = cpu_baseline_sample(wc, 1, 1)
                dt = (time.perf_counter() - t0) / reps
                assert int(o1.score[0]) == int(rw["res"].score[0]), f"{name}: GPU/CPU score mismatch"
                c["cpu_baseline"] = {"value": ccells / dt / 1e9, "unit": UNIT, "cores": 1, "kind": kind, "sample": "first pair, single thread"}
            configs.append(c)
            del rw

    # ---------------- sharded legs: one batch over all ranks, gathered on rank 0's host ----------------
    sharded = None
    if not args.no_sharded:
        sharded = []
        w_all = w if world == 1 else make_workload(args.pairs, 0)          # every rank generates the SAME batch
        s2 = sharded_leg(al, A, dist, w_all, "C2 1 Mi pairs in total" if args.pairs == 1 << 20 else f"C2 {args.pairs} pairs in total", A.OUT_CIGAR,
                         rank, world, 3, barrier, expect={"score_sum": score_sum, "cigar_ops": cigar_ops} if world == 1 else None, twobit=not args.bytes_e2e)
        w5 = synth.config5_edit(n_pairs=64, stream=0)
        s5 = sharded_leg(al, A, dist, w5, "C5 64 pairs in total", 0, rank, world, 2, barrier)
        if rank == 0:
            sharded = [s2, s5]
        del w_all

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "s16x2", "data": "synthetic",
            "config": {"workload": C2_WORKLOAD,
                       "pairs_per_gpu": args.pairs, "l1": 150, "l2": 500, "parallelism": f"pairs sharded x{world}, no collective",
                       "l2_policy": "inputs (650 MB sequences + 42 GB pointer arena) are larger than L2"},
            "fill_ms_per_step": head["fill_ms_per_step"], "traceback_ms_per_step": head["traceback_ms_per_step"],
            "wall_ms_per_step": wall_ms / args.steps,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "cpu_baseline": cpu,
            "checks": {"score_sum": score_sum, "cigar_ops": cigar_ops},
            "configs": configs, "sharded": sharded,
        }
        print(json.dumps(line), flush=True)
    al.close()
    if use_dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
