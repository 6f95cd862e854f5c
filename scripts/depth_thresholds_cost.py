"""What the depth thresholds cost: HBM-resident steps (clb_rerun_resident) with 1000-position depth tiles alone, with the
tiles and K = 4 thresholds (1, 10, 20, 30, mosdepth's usual list) and with the tiles and K = 8 thresholds, on the bench's
chr1-size 30x workload and on BASELINE configs 4 (2000x piles, default cap) and 5 (long reads) at the sizes bench.py's
other_configs uses.

Each variant gets its own context with the contig resident; the steps of the contexts alternate (tiles, K = 4, K = 8,
tiles, ...) so that drifts of the shared machine hit all of them alike.  The script checks on the same inputs that
intervals, state counts, sums, bins and the four tile arrays are identical across the variants, that the threshold counts
hold their invariants (raw_ge <= territory, qc_ge <= raw_ge, both non-increasing in the threshold), that K = 4's counts are
K = 8's at the same thresholds, and that the last timed step gives the counts of the first run.  One JSON line per workload
and variant, with the card's name, power limit and maximum SM clock read in the same run.  Needs a GPU; there is no CPU
path.

    python scripts/depth_thresholds_cost.py [--steps 30] [--warmup 3] [--scale 1.0]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.depth_tiles_cost import card, same_result, same_tiles  # noqa: E402

TILE_LEN = 1000
K4 = (1, 10, 20, 30)
K8 = (1, 5, 10, 15, 20, 30, 50, 100)
VARIANTS = ((), K4, K8)


def invariants_hold(r):
    raw, qc, ter = (np.asarray(x, np.int64) for x in (r.tile_raw_ge, r.tile_qc_ge, r.tile_territory))
    return bool(np.all(raw <= ter) and np.all(qc <= raw) and np.all(np.diff(raw, axis=0) <= 0) and np.all(np.diff(qc, axis=0) <= 0))


def same_counts(a, b):
    return bool(np.array_equal(a.tile_raw_ge, b.tile_raw_ge) and np.array_equal(a.tile_qc_ge, b.tile_qc_ge))


def run_workload(tag, c, opt, steps, warmup, info):
    from decodingustools_b200.callable_loci import CallableLociContext, admit_reads, compact_reads
    reads = compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0, threads=0))
    ctxs, first = [], []
    for ths in VARIANTS:
        ctx = CallableLociContext(opt)
        ctx.set_depth_tiles(TILE_LEN)
        ctx.set_depth_thresholds(ths)
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
    checks = [same_result(first[i], first[0]) and same_tiles(first[i], first[0]) and same_tiles(last[i], first[i])
              and last[i].state_counts.tolist() == first[i].state_counts.tolist() for i in range(len(VARIANTS))]
    counts_ok = [True] + [invariants_hold(first[i]) and same_counts(last[i], first[i]) for i in range(1, len(VARIANTS))]
    pick = [K8.index(t) for t in K4]                                     # K = 4's thresholds are among K = 8's
    counts_ok[1] = counts_ok[1] and np.array_equal(first[1].tile_raw_ge, first[2].tile_raw_ge[pick]) \
        and np.array_equal(first[1].tile_qc_ge, first[2].tile_qc_ge[pick])
    base = float(np.median([t[0] for t in times[0]]))
    for i, ths in enumerate(VARIANTS):
        t = np.array(times[i])
        med = float(np.median(t[:, 0]))
        print(json.dumps({"workload": tag, "variant": f"L={TILE_LEN}" + (f" + K={len(ths)} {list(ths)}" if ths else " tiles alone"),
                          "contig_bp": c.length, "reads_admitted": reads.n, "cells": int(first[i].summed_coverage),
                          "general_windows": int(last[i].general_windows), "steps": steps,
                          "step_ms_median": round(med, 4), "step_ms_min": round(float(t[:, 0].min()), 4),
                          "pileup_ms_median": round(float(np.median(t[:, 1])), 4), "fast_ms_median": round(float(np.median(t[:, 2])), 4),
                          "overhead_pct_vs_tiles": round(100.0 * (med / base - 1.0), 2),
                          "results_and_tiles_identical": checks[i], "threshold_counts_ok": counts_ok[i], **info}), flush=True)
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
        raise SystemExit("depth_thresholds_cost.py needs a CUDA device")
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
