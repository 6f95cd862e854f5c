"""What the depth runs cost: HBM-resident steps (clb_rerun_resident) with the runs off and on, on the bench's chr1-size 30x
workload and on BASELINE configs 4 (2000x piles, default cap) and 5 (long reads) at the sizes bench.py's other_configs uses.

Each variant gets its own context with the contig resident; the steps of the two contexts alternate (off, on, off, ...) so
that drifts of the shared machine hit both alike.  The script checks on the same inputs that intervals, state counts, sums
and bins are identical with and without the runs, and on the last timed step that the runs are the first run's and hold
their invariants: they start at the region start, starts ascend, adjacent depths differ, sum (end - start) * depth is
summed_coverage and sum (end - start) over depth > 0 is n_covered_bases.  On the chr1 workload it also reports the run
count, the bytes and time of their device-to-host copy (a copy of the same size into pinned memory, CUDA events), and the
host time of clb_bedgraph_writer_add_contig writing them to a file.  One JSON line per workload and variant, with the card's
name and power limit read in the same run.  Needs a GPU; there is no CPU path.

    python scripts/depth_runs_cost.py [--steps 30] [--warmup 3] [--scale 1.0]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

VARIANTS = (False, True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().splitlines()[0].split(",")] + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def same_result(a, b):
    return bool(np.array_equal(a.intervals, b.intervals) and a.state_counts.tolist() == b.state_counts.tolist()
                and np.array_equal(a.bins, b.bins)
                and all(getattr(a, k) == getattr(b, k) for k in ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases")))


def runs_hold(r):
    from decodingustools_b200.callable_loci import depth_run_ends
    runs = r.depth_runs
    if runs is None or len(runs) == 0:
        return False
    starts = runs["start"].astype(np.int64)
    lens = depth_run_ends(runs, r.region_end) - starts
    depth = runs["depth"].astype(np.int64)
    return bool(starts[0] == r.region_start and (lens > 0).all() and (np.diff(depth) != 0).all()
                and int((lens * depth).sum()) == r.summed_coverage and int(lens[depth > 0].sum()) == r.n_covered_bases)


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


def run_workload(key, tag, c, opt, steps, warmup, info):
    from decodingustools_b200.callable_loci import BedGraphWriter, CallableLociContext, admit_reads, compact_reads
    reads = compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0, threads=0))
    ctxs, first = [], []
    for on in VARIANTS:
        ctx = CallableLociContext(opt)
        ctx.set_depth_runs(on)
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
    checks = [same_result(first[i], first[0]) and last[i].state_counts.tolist() == first[i].state_counts.tolist() for i in range(len(VARIANTS))]
    runs_ok = [True, runs_hold(last[1]) and np.array_equal(last[1].depth_runs, first[1].depth_runs)]
    base = float(np.median([t[0] for t in times[0]]))
    extra = {}
    if key == "chr1":
        n = len(first[1].depth_runs)
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "depth.bedgraph")
            w = BedGraphWriter(path)
            t0 = time.perf_counter()
            w.add_contig(c.name, c.length, first[1].depth_runs)
            t1 = time.perf_counter()
            w.close()
            size = os.path.getsize(path)
        extra = {"runs": n, "runs_per_admitted_read": round(n / reads.n, 3), "runs_d2h_bytes": 8 * n, "runs_d2h_ms": round(d2h_ms(8 * n), 3),
                 "d2h_bytes_off": int(first[0].d2h_bytes), "d2h_bytes_on": int(first[1].d2h_bytes),
                 "bedgraph_add_contig_s": round(t1 - t0, 3), "bedgraph_bytes": size}
    for i, on in enumerate(VARIANTS):
        t = np.array(times[i])
        med = float(np.median(t[:, 0]))
        print(json.dumps({"workload": tag, "variant": "on" if on else "off", "contig_bp": c.length, "reads_admitted": reads.n,
                          "cells": int(first[i].summed_coverage), "general_windows": int(last[i].general_windows), "steps": steps,
                          "step_ms_median": round(med, 4), "step_ms_min": round(float(t[:, 0].min()), 4),
                          "pileup_ms_median": round(float(np.median(t[:, 1])), 4), "fast_ms_median": round(float(np.median(t[:, 2])), 4),
                          "overhead_pct_vs_off": round(100.0 * (med / base - 1.0), 2),
                          "results_identical_to_off": checks[i], "runs_hold": runs_ok[i], **(extra if on else {}), **info}), flush=True)
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
        raise SystemExit("depth_runs_cost.py needs a CUDA device")
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
        run_workload(key, tag, make(), opt, args.steps, args.warmup, info)


if __name__ == "__main__":
    main()
