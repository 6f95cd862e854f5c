"""What the QC depth runs cost: HBM-resident steps (clb_rerun_resident) with no runs, raw runs, QC runs and both, on the
bench's chr1-size 30x workload and on BASELINE configs 4 (2000x piles, default cap) and 5 (long reads) at the sizes
bench.py's other_configs uses.

Each variant gets its own context with the contig resident; the steps of the four contexts alternate (off, raw, qc, both,
off, ...) so that drifts of the shared machine hit them alike.  The script checks on the same inputs that intervals, state
counts, sums and bins are identical across the variants, that the raw runs are the same with and without the QC runs, that
the QC runs are the same alone and with the raw runs, and that the QC runs hold their invariants (they start at the region
start, adjacent depths differ, sum (end - start) * depth is quality_bases).  For each variant it reports the median step
and pileup-kernel time, raw and QC runs per 1000 positions, the bytes and time of the runs' device-to-host copy (a copy of
the same size into pinned memory, CUDA events), and the bedGraph text bytes and the host time of
clb_bedgraph_writer_add_contig writing the runs to /dev/null (formatting and write calls, no disk).  One JSON line per
workload and variant, with the card's name, power limit and maximum SM clock read in the same run.  Needs a GPU; there is
no CPU path.

    python scripts/qc_depth_runs_cost.py [--steps 30] [--warmup 3] [--scale 1.0]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

VARIANTS = (("off", False, False), ("raw", True, False), ("qc", False, True), ("both", True, True))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().splitlines()[0].split(",")] + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def same_result(a, b):
    return bool(np.array_equal(a.intervals, b.intervals) and a.state_counts.tolist() == b.state_counts.tolist()
                and np.array_equal(a.bins, b.bins)
                and all(getattr(a, k) == getattr(b, k) for k in ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases")))


def qc_runs_hold(r):
    from decodingustools_b200.callable_loci import depth_run_ends
    runs = r.qc_depth_runs
    if runs is None or len(runs) == 0:
        return False
    starts = runs["start"].astype(np.int64)
    lens = depth_run_ends(runs, r.region_end) - starts
    depth = runs["depth"].astype(np.int64)
    return bool(starts[0] == r.region_start and (lens > 0).all() and (np.diff(depth) != 0).all()
                and int((lens * depth).sum()) == r.quality_bases)


def d2h_ms(n_bytes, reps=10):
    """Median time of one device-to-host copy of n_bytes into pinned memory (what fetch_result does for the runs)."""
    import torch
    src = torch.empty(max(n_bytes, 1), dtype=torch.uint8, device="cuda")
    dst = torch.empty(max(n_bytes, 1), dtype=torch.uint8, pin_memory=True)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(reps + 1):
        a.record(); dst.copy_(src, non_blocking=True); b.record(); b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts[1:]))


def bedgraph_bytes(name, runs, region_end):
    """Bytes of the bedGraph lines "name\\tstart\\tend\\tdepth\\n" of the runs."""
    from decodingustools_b200.callable_loci import depth_run_ends
    if runs is None or len(runs) == 0:
        return 0
    digits = lambda v: np.floor(np.log10(np.maximum(np.asarray(v, np.float64), 1.0))).astype(np.int64) + 1  # noqa: E731
    return int(len(runs) * (len(name) + 4) + digits(runs["start"]).sum() + digits(depth_run_ends(runs, region_end)).sum()
               + digits(runs["depth"]).sum())


def write_ms(name, length, runs):
    from decodingustools_b200.callable_loci import BedGraphWriter
    if runs is None:
        return 0.0
    w = BedGraphWriter("/dev/null")
    t0 = time.perf_counter()
    w.add_contig(name, length, runs)
    t1 = time.perf_counter()
    w.close()
    return 1000.0 * (t1 - t0)


def run_workload(tag, c, opt, steps, warmup, info):
    from decodingustools_b200.callable_loci import CallableLociContext, admit_reads, compact_reads
    reads = compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0, threads=0))
    ctxs, first = [], []
    for _, raw, qc in VARIANTS:
        ctx = CallableLociContext(opt)
        ctx.set_depth_runs(raw)
        ctx.set_qc_depth_runs(qc)
        ctx.begin_contig(0, c.name, c.length, c.ref, c.length, max_ref_span=reads.max_ref_span())
        ctx.push_reads(reads)
        first.append(ctx.finish_contig(copy_intervals=True))
        ctxs.append(ctx)
    for _ in range(warmup):
        for ctx in ctxs:
            ctx.rerun_resident(fetch=False)
    times = [[] for _ in VARIANTS]
    last = [None] * len(VARIANTS)
    for _ in range(steps):
        for i, ctx in enumerate(ctxs):
            ms, res = ctx.rerun_resident(fetch=True, copy_intervals=False)
            times[i].append((ms, res.pileup_ms, res.fast_ms))
            last[i] = res
    identical = [same_result(first[i], first[0]) and last[i].state_counts.tolist() == first[0].state_counts.tolist()
                 for i in range(len(VARIANTS))]
    raw_same = bool(np.array_equal(first[1].depth_runs, first[3].depth_runs) and np.array_equal(last[3].depth_runs, first[1].depth_runs))
    qc_same = bool(np.array_equal(first[2].qc_depth_runs, first[3].qc_depth_runs) and np.array_equal(last[2].qc_depth_runs, first[2].qc_depth_runs))
    base = float(np.median([t[0] for t in times[0]]))
    for i, (name, raw, qc) in enumerate(VARIANTS):
        t = np.array(times[i])
        med = float(np.median(t[:, 0]))
        r = first[i]
        n_raw = len(r.depth_runs) if raw else 0
        n_qc = len(r.qc_depth_runs) if qc else 0
        n_bytes = 8 * (n_raw + n_qc)
        print(json.dumps({"workload": tag, "variant": name, "contig_bp": c.length, "reads_admitted": reads.n,
                          "cells": int(r.summed_coverage), "general_windows": int(last[i].general_windows), "steps": steps,
                          "step_ms_median": round(med, 4), "step_ms_min": round(float(t[:, 0].min()), 4),
                          "pileup_ms_median": round(float(np.median(t[:, 1])), 4), "fast_ms_median": round(float(np.median(t[:, 2])), 4),
                          "overhead_pct_vs_off": round(100.0 * (med / base - 1.0), 2),
                          "raw_runs": n_raw, "qc_runs": n_qc,
                          "raw_runs_per_1000": round(1000.0 * n_raw / c.length, 2), "qc_runs_per_1000": round(1000.0 * n_qc / c.length, 2),
                          "d2h_bytes": int(r.d2h_bytes), "runs_d2h_bytes": n_bytes, "runs_d2h_ms": round(d2h_ms(n_bytes), 3) if n_bytes else 0.0,
                          "raw_bedgraph_bytes": bedgraph_bytes(c.name, r.depth_runs, c.length) if raw else 0,
                          "qc_bedgraph_bytes": bedgraph_bytes(c.name, r.qc_depth_runs, c.length) if qc else 0,
                          "raw_bedgraph_write_ms": round(write_ms(c.name, c.length, r.depth_runs), 1) if raw else 0.0,
                          "qc_bedgraph_write_ms": round(write_ms(c.name, c.length, r.qc_depth_runs), 1) if qc else 0.0,
                          "results_identical_to_off": identical[i], "raw_runs_same_with_qc_runs": raw_same,
                          "qc_runs_same_with_raw_runs": qc_same, "qc_runs_hold": qc_runs_hold(last[i]) if qc else None, **info}), flush=True)
    assert all(identical) and raw_same and qc_same and qc_runs_hold(last[2]) and qc_runs_hold(last[3]), tag
    for ctx in ctxs:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="of the chr1-size workload")
    ap.add_argument("--only", choices=["chr1", "config4", "config5"], action="append")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("qc_depth_runs_cost.py needs a CUDA device")
    from decodingustools_b200 import synth
    from decodingustools_b200.options import CallableOptions
    info = card()
    dev = torch.device("cuda", 0)
    work = (("chr1", "chr1-size synthetic 30x 2x150 bp (bench.py workload)",
             lambda: synth.synth_short("chr1", max(100_000, int(synth.HG38["chr1"] * args.scale)), synth.SEED0 + 1, qual_device=dev),
             CallableOptions()),
            ("config4", "configs[3] at reduced scale: 2000x, 2.8 Mbp, --max-depth 500",
             lambda: synth.synth_short("chrY", 2_800_000, 4, depth=2000.0), CallableOptions()),
            ("config5", "configs[4] at reduced scale: 15 kb indel-heavy long reads, 25 Mbp, 30x",
             lambda: synth.synth_long("chr1", 25_000_000, 5), CallableOptions()))
    for key, tag, make, opt in work:
        if args.only and key not in args.only:
            continue
        run_workload(tag, make(), opt, args.steps, args.warmup, info)


if __name__ == "__main__":
    main()
