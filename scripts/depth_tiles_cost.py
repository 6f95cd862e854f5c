"""What the depth tiles cost: HBM-resident steps (clb_rerun_resident) with the tiles off, on with tiles of 256, 1000 (the
coverage command's default) and 100000 positions, and on with 1000-position tiles and 1001-bin depth histograms together,
on the bench's chr1-size 30x workload and on BASELINE configs 4 (2000x piles, default cap) and 5 (long reads) at the sizes
bench.py's other_configs uses.

Each variant gets its own context with the contig resident; the steps of the contexts alternate (off, 256, 1000, 100000,
1000 + histograms, off, ...) so that drifts of the shared machine hit all of them alike.  The script checks on the same
inputs that intervals, state counts, sums and bins are identical with and without the tiles, that the tiles add up (every
position that is not REF_N in one tile's territory, every CALLABLE one in one tile's callable count), that the last timed
step gives the tiles of the first run, and that the 1000-position tiles do not change when the histograms are on too.  One
JSON line per workload and variant, with the card's name and power limit read in the same run.  Needs a GPU; there is no
CPU path.

    python scripts/depth_tiles_cost.py [--steps 30] [--warmup 3] [--scale 1.0]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

VARIANTS = ((0, 0), (256, 0), (1000, 0), (100_000, 0), (1000, 1001))     # (tile length, histogram bins)
TILE_FIELDS = ("tile_territory", "tile_callable", "tile_raw_sum", "tile_qc_sum")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().splitlines()[0].split(",")] + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def same_result(a, b):
    return bool(np.array_equal(a.intervals, b.intervals) and a.state_counts.tolist() == b.state_counts.tolist()
                and np.array_equal(a.bins, b.bins)
                and all(getattr(a, k) == getattr(b, k) for k in ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases")))


def tiles_add_up(r, length):
    return bool(int(r.tile_territory.sum()) == length - int(r.state_counts[0]) and int(r.tile_callable.sum()) == int(r.state_counts[1]))


def same_tiles(a, b):
    return all(np.array_equal(getattr(a, k), getattr(b, k)) for k in TILE_FIELDS)


def run_workload(tag, c, opt, steps, warmup, info):
    from decodingustools_b200.callable_loci import CallableLociContext, admit_reads, compact_reads
    reads = compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0, threads=0))
    ctxs, first = [], []
    for tl, n in VARIANTS:
        ctx = CallableLociContext(opt)
        ctx.set_depth_tiles(tl)
        ctx.set_depth_histogram(n)
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
    # the same inputs, every variant: identical results; the last timed step of each variant: the same counters as its first run
    checks = [same_result(first[i], first[0]) and last[i].state_counts.tolist() == first[i].state_counts.tolist() for i in range(len(VARIANTS))]
    tiles_ok = [True] + [tiles_add_up(first[i], c.length) and same_tiles(last[i], first[i]) for i in range(1, len(VARIANTS))]
    tiles_ok[-1] = tiles_ok[-1] and same_tiles(first[-1], first[2])          # 1000 + histograms: the same tiles as 1000 alone
    base = float(np.median([t[0] for t in times[0]]))
    for i, (tl, n) in enumerate(VARIANTS):
        t = np.array(times[i])
        med = float(np.median(t[:, 0]))
        print(json.dumps({"workload": tag, "variant": "off" if tl == 0 else f"L={tl}" + (f" + hist n={n}" if n else ""), "contig_bp": c.length, "reads_admitted": reads.n,
                          "cells": int(first[i].summed_coverage), "general_windows": int(last[i].general_windows), "steps": steps,
                          "step_ms_median": round(med, 4), "step_ms_min": round(float(t[:, 0].min()), 4),
                          "pileup_ms_median": round(float(np.median(t[:, 1])), 4), "fast_ms_median": round(float(np.median(t[:, 2])), 4),
                          "overhead_pct_vs_off": round(100.0 * (med / base - 1.0), 2),
                          "results_identical_to_off": checks[i], "tiles_add_up": tiles_ok[i], **info}), flush=True)
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
        raise SystemExit("depth_tiles_cost.py needs a CUDA device")
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
