#!/usr/bin/env python
"""bench.py -- aligned Gbases/s of the CallableLoci pileup + classify + BED-segmentation path on B200.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` (torchrun for N > 1) prints ONE JSON line.
A "step" is one pass of the hot path over one contig-sized batch of synthetic reads:
    workload : BASELINE.json configs[1] -- chr1-size contig (248.96 Mbp), synthetic 30x 2x150 bp.
    N = 1    : one B200.
    N > 1    : every rank runs the same chr1-size contig on its own GPU (weak scaling: per-GPU work fixed); the counters of
               the N replicas are summed with the library's own NCCL all-reduce (clb_allreduce_nccl) inside the step and
               checked (= N x the single-GPU counters).  The `strong` block cuts ONE chr1 into N region shards (halo
               reads, all-reduce of counters/bins, interval stitching on rank 0) and checks the stitched result against
               rank 0's single-GPU run of the whole contig.
`value`  : pileup cells (aligned bases = sum of raw depth) per second, inputs resident in HBM: window ranges + pileup
           kernels + interval compaction (+ all-reduce); the upload-time helper kernels are reported beside it.
`e2e`    : the same metric through the public C-ABI call sequence from HOST buffers, everything the CPU arm also pays
           inside the timed region: read admission (htslib depth cap, clb_admit_reads_mt), reference upload, column-batch
           H2D copies, kernels, D2H of intervals + counters, and the BED text written to a real file.
`--impl reference`: the CPU oracle (restatement of the reference's single-threaded loop; the Rust reference itself
           cannot be built in this image) timed on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "aligned Gbases/s CallableLoci pileup"
UNIT = "Gbases/s"
WORKLOAD = "chr1-size synthetic 30x 2x150bp PE, pileup+classify+BED on one B200 per rank (BASELINE configs[1])"
DUMP_INTERVAL_ROWS = 1 << 20       # 5 float64 columns of this many rows: 40 MiB, the rest of a dump is a few kB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the contig (1.0 = chr1, 248.96 Mbp)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-pipelined", type=int, default=6, help="contigs of the pipelined e2e leg (0: report the single-contig time as e2e)")
    ap.add_argument("--cpu-sample-mbp", type=float, default=48.0, help="oracle sample of the bounded CPU legs (Mbp of the contig)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip every CPU oracle leg (cpu_baseline, parity)")
    ap.add_argument("--no-parity-full", action="store_true", help="check parity on the bounded sample only, not on the whole contig")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the reduced-scale runs of BASELINE configs 4/4b/5")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the region-sharded strong-scaling leg")
    ap.add_argument("--no-e2e-bam", action="store_true", help="skip the BAM -> BED leg through the C++ coverage command")
    ap.add_argument("--bam-mbp", type=float, default=50.818468, help="contig size of the e2e_bam leg (default: chr22)")
    ap.add_argument("--batch-reads", type=int, default=4_000_000, help="column-batch size of the e2e leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the result of the GPU path (--impl b200)")
    return args


def load_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(scale, world):
    """dram__bytes_read + dram__bytes_write of ONE launch of the dominant kernel, from the ncu --set full capture of this
    workload summarised under profiles/ (never a literal in this file); None when no capture matches."""
    p = os.path.join(ROOT, "profiles", "r02_k_pileup_fast_traffic.json")
    if scale != 1.0 or world != 1 or not os.path.exists(p):
        return None, ("profiles/r02_k_pileup_fast_traffic.json" if os.path.exists(p) else None)
    try:
        d = json.load(open(p))
        return int(d["dram_bytes_read"]) + int(d["dram_bytes_write"]), "profiles/r02_k_pileup_fast_traffic.json"
    except Exception:
        return None, None


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML, the library behind nvidia-smi's
    clocks.sm / clocks_event_reasons.* query of B200_PROFILING.md; falls back to nvidia-smi itself)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int, period_s: float = 0.004):
        import threading
        self.idx, self.period = gpu_index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(physical_gpu_index(gpu_index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        import threading
        if self._h is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set(); self._thr.join(timeout=2)
            return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(self.samples), "source": "nvml"}
        try:   # one-shot fallback
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                 capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]),
                    "reasons": [n for n, v in zip(names, out[2:6]) if v.strip().lower().startswith("active")], "samples": 1,
                    "source": "nvidia-smi after the timed region"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"], "samples": 0}


def physical_gpu_index(local_index: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        parts = vis.split(",")
        if local_index < len(parts) and parts[local_index].strip().isdigit():
            return int(parts[local_index])
    return local_index


def bind_to_gpu_numa(local_rank: int):
    """Run this rank on the cores of its GPU's NUMA node, so that the column buffers it allocates (first touch) and
    page-locks live next to the GPU's PCIe root.  Returns what was done, for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(physical_gpu_index(local_rank))
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return share_cores(local_rank, {"numa_node": None, "note": "no NUMA information for this GPU"})
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return share_cores(local_rank, {"numa_node": node, "cores": len(cpus)})
    except Exception as e:      # binding is an optimisation, never a failure
        return share_cores(local_rank, {"numa_node": None, "note": f"not bound: {type(e).__name__}"})


def share_cores(local_rank: int, rec: dict):
    """Ranks that ended up on the same cores (one NUMA node for several GPUs, or no NUMA information) split them, so that the
    host-side stages (admission, BED formatting: one thread per core of the affinity mask) do not oversubscribe the box."""
    try:
        world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
        cpus = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cpus) >= world:
            per = len(cpus) // world
            mine = cpus[local_rank * per:(local_rank + 1) * per]
            os.sched_setaffinity(0, set(mine))
            rec["cores_of_rank"] = len(mine)
    except Exception as e:
        rec["share_note"] = f"cores not split: {type(e).__name__}"
    return rec


def make_workload(scale: float, device=None):
    """The chr1-size synthetic contig (same seed on every rank), unfiltered, as the decoder would hand it over."""
    from decodingustools_b200 import synth
    from decodingustools_b200.options import CallableOptions
    opt = CallableOptions()
    length = max(100_000, int(synth.HG38["chr1"] * scale))
    t0 = time.time()
    c = synth.synth_short("chr1", length, synth.SEED0 + 1, qual_device=device)     # the generator may fill the quality column on the GPU
    return opt, c, {"synth_s": round(time.time() - t0, 2)}


def oracle_run(c, reads, opt, length: int):
    """The CPU oracle over the first `length` bases of the contig (every read that starts inside)."""
    from oracle import oracle
    length = min(length, c.length)
    if length < c.length:
        hi = int(np.searchsorted(reads.pos, length - 200, side="left"))
        reads = reads.slice(0, hi)
    t0 = time.perf_counter()
    run = oracle.OracleRun(opt, length)
    oc = run.process_contig(c.name, 0, length, c.ref[:length], reads)
    dt = time.perf_counter() - t0
    return oc, run, dt, reads


def dump_outputs(out_dir: str, res) -> None:
    """What a caller of the resident step receives (a ContigDeviceResult) as out_dir/<name>.npy, float64: counters and bins
    whole; of the interval list the rows interval_row, a seeded sample of DUMP_INTERVAL_ROWS rows (every row of a shorter
    list), so that two builds computing the same intervals write the same files."""
    iv = res.intervals
    n = iv.shape[0]
    rows = np.arange(n) if n <= DUMP_INTERVAL_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_INTERVAL_ROWS, replace=False))
    arrays = {"state_counts": res.state_counts, "bins": res.bins, "stride": res.stride, "n_covered_bases": res.n_covered_bases,
              "summed_coverage": res.summed_coverage, "summed_baseq": res.summed_baseq, "summed_mapq": res.summed_mapq,
              "quality_bases": res.quality_bases, "n_intervals": n, "interval_row": rows, "interval_start": iv["start"][rows],
              "interval_end": iv["end"][rows], "interval_state": iv["state"][rows], "interval_soft_start": iv["soft_start"][rows]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_reference(args, rank, world):
    """--impl reference: the CPU restatement of the reference loop (single-threaded, like the reference)."""
    if rank != 0:
        return
    from decodingustools_b200 import synth
    from decodingustools_b200.options import CallableOptions
    opt = CallableOptions()
    sample_bp = int(args.cpu_sample_mbp * 1e6 * min(1.0, args.scale * 4))
    length = max(sample_bp, 100_000)
    c = synth.synth_short("chr1", length, synth.SEED0 + 1)
    times, cells = [], 0
    for i in range(args.warmup + args.steps):
        oc, _, dt, _ = oracle_run(c, c.reads, opt, sample_bp)
        if i >= args.warmup:
            times.append(dt)
        cells = oc.summed_coverage
    t = sum(times)
    val = cells * len(times) / t / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/u32 integer", "data": "synthetic",
        "config": {"workload": WORKLOAD + "; the CPU arm runs a bounded prefix of it (a rate, so comparable)",
                   "sample_bp": sample_bp, "sample_cells": int(cells)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": f"first {sample_bp} bp of the contig ({int(cells)} cells) per step; oracle/callable_oracle.c, "
                                   "single thread like the reference (src/api/coverage.rs:232-234), admission and BED text included; omits "
                                   "the reference's per-base faidx call and per-cell qname hashing, so it is faster than the real binary"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class Pinned:
    """A numpy array page-locked in place (the e2e leg streams from it; no second host copy)."""

    def __init__(self, rt, arr):
        self.arr, self._rt = arr, rt
        rc = rt.cudaHostRegister(arr.ctypes.data, arr.nbytes, 0)
        if int(rc) != 0:
            raise RuntimeError(f"cudaHostRegister failed: {rc}")

    def data_ptr(self):
        return self.arr.ctypes.data


class Nccl:
    """An ncclComm_t of our own over the ranks of the job, created through ctypes on the NCCL build torch loaded (the
    unique id travels through torch.distributed), so that the library's clb_allreduce_nccl is what reduces."""

    class _Uid(C.Structure):
        _fields_ = [("internal", C.c_char * 128)]

    def __init__(self, rank, world, dev):
        import torch
        import torch.distributed as dist
        path = None
        for ln in open("/proc/self/maps"):
            if "libnccl" in ln and ".so" in ln:
                path = ln.split()[-1]
                break
        self.lib = C.CDLL(path or "libnccl.so.2", mode=C.RTLD_GLOBAL)
        self.path = path or "libnccl.so.2"
        uid = Nccl._Uid()
        if rank == 0:
            self._ok(self.lib.ncclGetUniqueId(C.byref(uid)))
        t = torch.frombuffer(bytearray(bytes(uid)), dtype=torch.uint8).to(dev)
        dist.broadcast(t, 0)
        C.memmove(C.byref(uid), bytes(t.cpu().numpy().tobytes()), 128)
        self.comm = C.c_void_p(0)
        self.lib.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, Nccl._Uid, C.c_int]
        self._ok(self.lib.ncclCommInitRank(C.byref(self.comm), world, uid, rank))
        self.allreduce_fn = C.cast(self.lib.ncclAllReduce, C.c_void_p).value
        ver = C.c_int(0)
        self.lib.ncclGetVersion(C.byref(ver))
        self.version = ver.value

    @staticmethod
    def _ok(rc):
        if rc != 0:
            raise RuntimeError(f"NCCL call failed: {rc}")

    def close(self):
        try:
            self.lib.ncclCommDestroy.argtypes = [C.c_void_p]
            self.lib.ncclCommDestroy(self.comm)
        except Exception:
            pass


def kernel_config_run(tag, c, opt, peak, check=True):
    """One reduced-scale BASELINE config: admission, upload, then the HBM-resident kernel time (best of 4 re-runs); the
    result (BED text, counters, bins) is compared with the CPU oracle run on the same offered records."""
    from decodingustools_b200.callable_loci import CallableLociContext, CallableProfiler, admit_reads, compact_reads
    t0 = time.perf_counter()
    st = {}
    keep = admit_reads(c.reads, opt.pileup_max_depth, 0, threads=0, stats=st)
    reads = compact_reads(c.reads, keep)
    t_adm = time.perf_counter() - t0
    ctx = CallableLociContext(opt)
    ctx.begin_contig(0, c.name, c.length, c.ref, c.length, max_ref_span=reads.max_ref_span())
    ctx.push_reads(reads)
    r = ctx.finish_contig(copy_intervals=check)
    parity = None
    if check:
        prof = CallableProfiler(None, c.length)
        prof.add_contig(c.name, c.length, r.intervals, r.state_counts, r.bins.copy(), r.stride)
        gbed = prof.bed_bytes()
    runs = [ctx.rerun_resident(fetch=True) for _ in range(4)]
    best = min(runs, key=lambda x: x[1].pileup_ms)
    step_ms, res = best
    byts = reads.nbytes_device() + c.length // 8
    ctx.close()
    if check:
        oc, orun, dt, _ = oracle_run(c, c.reads, opt, c.length)
        parity = bool(orun.bed() == gbed and r.state_counts.tolist() == oc.counts and r.n_covered_bases == oc.n_covered_bases
                      and r.summed_coverage == oc.summed_coverage and r.summed_baseq == oc.summed_baseq and r.summed_mapq == oc.summed_mapq
                      and r.quality_bases == oc.quality_bases and oc.bins is not None and np.array_equal(r.bins, oc.bins))
    return {"config": tag, "parity": parity, "contig_bp": c.length, "reads_offered": c.reads.n, "reads_admitted": reads.n, "cigar_ops": reads.n_cigar,
            "cells": int(r.summed_coverage), "pileup_ms": round(res.pileup_ms, 4), "step_ms": round(step_ms, 4),
            "upload_kernels_ms": round(r.upload_ms, 4), "general_windows": int(res.general_windows),
            "Gbases_s": round(r.summed_coverage / res.pileup_ms / 1e6, 1), "frac": round(byts / res.pileup_ms / 1e6 / peak, 4),
            "host_admission_s": round(t_adm, 2), "admission_replayed": st.get("replayed")}


def e2e_bam_leg(args, opt, device_index: int):
    """BAM + FASTA files -> callable_regions.bed + summary.json through the C++ `coverage` command over the C ABI (what the
    reference's CLI does: BGZF inflate, record decode, admission, device, BED text, report), on a chr22-size synthetic
    BAM.  Wall time, host-decode time and device time are reported separately (north_star); the BED is checked against
    the CPU oracle run on the same records."""
    from decodingustools_b200 import synth
    from tests import bamio
    length = int(args.bam_mbp * 1e6)
    exe = os.path.join(ROOT, "decodingustools_b200", "decodingus-tools-b200")
    if not os.path.exists(exe) or not os.path.exists(os.path.join(ROOT, "decodingustools_b200", "clb-pack-bam")):
        return {"unavailable": "decodingus-tools-b200 / clb-pack-bam not built (python -c 'import __graft_entry__ as g; g.build()')"}
    work = tempfile.mkdtemp(prefix="clb_bam_")
    try:
        t0 = time.perf_counter()
        c = synth.synth_short("chr22", length, synth.SEED0)
        bam, fa = os.path.join(work, "in.bam"), os.path.join(work, "ref.fa")
        bamio.pack_bam_fast(bam, c.name, c.length, c.reads, os.path.join(work, "cols"))
        bamio.write_fasta(fa, [(c.name, c.ref.tobytes())])
        t_prep = time.perf_counter() - t0
        runs = []
        for _ in range(2):
            tj = os.path.join(work, "timing.json")
            t1 = time.perf_counter()
            p = subprocess.run([exe, "coverage", bam, "-r", fa, "-o", "callable_regions.bed", "--device", str(device_index), "--timing-json", tj],
                               cwd=work, capture_output=True, text=True, timeout=900)
            dt = time.perf_counter() - t1
            if p.returncode != 0:
                return {"unavailable": "coverage command failed: " + p.stderr[-300:]}
            tm = json.load(open(tj)); tm["process_wall_s"] = dt
            runs.append(tm)
        best = min(runs, key=lambda r: r["process_wall_s"])
        bed_sha = hashlib.sha256(open(os.path.join(work, "callable_regions.bed"), "rb").read()).hexdigest()
        out = {"workload": f"chr22-size synthetic 30x 2x150bp BAM ({os.path.getsize(bam) / 1e6:.0f} MB BGZF, {c.reads.n} records) + FASTA -> BED + summary.json + HTML + SVG",
               "value": best["aligned_bases"] / best["process_wall_s"] / 1e9, "unit": UNIT, "process_wall_s": round(best["process_wall_s"], 3),
               "pipeline_wall_s": round(best["wall_s"], 3), "host_decode_s": round(best["decode_s"], 3), "bgzf_inflate_s": round(best["inflate_s"], 3),
               "admission_s": round(best["admission_s"], 3), "decode_threads": best["threads"], "device_kernels_s": round(best["device_kernels_s"], 4),
               "h2d_s": round(best["h2d_s"], 4), "reference_load_s": round(best["reference_load_s"], 3), "unique_names_s": round(best["unique_names_s"], 3),
               "bed_and_plots_s": round(best["bed_and_plots_s"], 3), "device_thread_waited_for_decoder_s": round(best["device_thread_waited_s"], 3),
               "synth_and_pack_s": round(t_prep, 1),
               "note": "host decode (BGZF inflate on all cores + record scan + admission + packing) runs concurrently with the device thread; "
                       "the pipeline is decode-bound, the device is idle most of the wall time"}
        if not args.no_cpu_baseline:
            oc, orun, dt, _ = oracle_run(c, c.reads, opt, c.length)
            out["bed_equals_oracle"] = bool(hashlib.sha256(orun.bed()).hexdigest() == bed_sha)
            js = json.load(open(os.path.join(work, "summary.json")))["export"]["contigs"][0]
            out["summary_counts_equal_oracle"] = bool([js["state_distribution"][k] for k in ("ref_n", "callable", "no_coverage", "low_coverage", "excessive_coverage",
                                                                                              "poor_mapping_quality")] == oc.counts
                                                      and js["unique_reads"] == oc.n_reads and js["covered_bases"] == oc.n_covered_bases)
            out["cpu_oracle_same_records_s"] = round(dt, 1)
        return out
    finally:
        import shutil
        shutil.rmtree(work, ignore_errors=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    numa = bind_to_gpu_numa(local_rank) if world > 1 else None      # before any buffer of this rank is allocated

    import torch
    import torch.distributed as dist
    from decodingustools_b200 import _lib, sharding
    from decodingustools_b200.callable_loci import (INTERVAL_DTYPE, CallableLociContext, _result, admit_reads, compact_reads)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    peak, peak_src = load_peak()

    opt, c, prep = make_workload(args.scale, dev)
    reads = c.reads                                   # unfiltered: admission is part of the e2e step
    span = reads.max_ref_span()
    maxcnt = opt.pileup_max_depth
    alg_bytes = reads.nbytes_device() + c.length // 8          # packed columns + 1 bit per reference base

    rt = torch.cuda.cudart()
    cols = {k: Pinned(rt, getattr(reads, k)) for k in ("pos", "flag", "mapq", "cigar", "qual")}
    ref_pinned = Pinned(rt, c.ref)
    cig_off = reads.cigar_off.astype(np.int64); q_off = reads.qual_off.astype(np.int64)
    batches = []                                      # column batches as a decoder thread would emit them (batch-relative offsets)
    for lo in range(0, reads.n, args.batch_reads):
        hi = min(reads.n, lo + args.batch_reads)
        co = Pinned(rt, np.ascontiguousarray((cig_off[lo:hi + 1] - cig_off[lo]).astype(np.uint32)))
        qo = Pinned(rt, np.ascontiguousarray((q_off[lo:hi + 1] - q_off[lo]).astype(np.uint64)))
        batches.append((lo, hi, co, qo))

    ctx = CallableLociContext(opt, device=local_rank)
    stream = torch.cuda.Stream(device=dev)            # the context's kernels, the NCCL reduction and the timing events all go on this stream
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    bed_dir = tempfile.mkdtemp(prefix="clb_bench_")
    bed_path = os.path.join(bed_dir, f"callable_regions.rank{rank}.bed")
    mapped_only = None

    def e2e_pass(defer_bed=False):
        """What `coverage` does for one contig, from host buffers to the BED file.  defer_bed: return the BED step as a job
        for a writer thread (it gets its own copy of the interval list) instead of running it here."""
        nonlocal mapped_only
        t0 = time.perf_counter()
        st = {}
        verdict = {}

        def admission():
            ta = time.perf_counter()
            verdict["keep"] = admit_reads(reads, maxcnt, 0, threads=0, max_ref_span=span, stats=st)
            verdict["ms"] = 1e3 * (time.perf_counter() - ta)
        # Admission runs on host threads WHILE the column batches are being copied: the batches are pushed as they are
        # (the kernels skip placed-unmapped records themselves); should the depth cap refuse anything else, the contig
        # would have to be repacked and pushed again -- on 30x data it never does, and the verdict is checked before
        # the result is used.
        th = threading.Thread(target=admission)
        th.start()
        ctx._check(L.clb_begin_contig(ctx._h, 0, b"chr1", c.length, ref_pinned.data_ptr(), c.length, 0, c.length, 0, c.length, span))
        ctx.reserve(reads.n, reads.n_cigar, reads.n_qual)
        for lo, hi, co, qo in batches:
            ctx.push_raw(hi - lo, int(cig_off[hi] - cig_off[lo]), int(q_off[hi] - q_off[lo]),
                         cols["pos"].data_ptr() + 4 * lo, cols["flag"].data_ptr() + 2 * lo, cols["mapq"].data_ptr() + lo,
                         co.data_ptr(), cols["cigar"].data_ptr() + 4 * int(cig_off[lo]), qo.data_ptr(),
                         cols["qual"].data_ptr() + int(q_off[lo]))
        th.join()
        t1 = time.perf_counter()
        if mapped_only is None:
            mapped_only = (reads.flag & 4) == 0
        if not np.array_equal(verdict["keep"], mapped_only):
            raise SystemExit("the depth cap refused records of the 30x workload: this leg expects to stream the page-locked columns as they are")
        raw = ctx.finish_contig_raw()
        t2 = time.perf_counter()
        bins = np.ctypeslib.as_array(raw.bins, shape=(3 * int(raw.n_bins),)).copy()
        n_iv, n_bins, stride = int(raw.n_intervals), int(raw.n_bins), int(raw.stride)

        def write_bed(iv_ptr, keep=None):
            tb = time.perf_counter()
            w = L.clb_bed_writer_open(bed_path.encode(), c.length)
            has = C.c_int(0)
            rc = L.clb_bed_writer_add_contig(w, b"chr1", c.length, iv_ptr, n_iv, bins.ctypes.data_as(C.c_void_p), n_bins, stride, C.byref(has))
            rc2 = L.clb_bed_writer_close(w)
            if rc or rc2:
                raise SystemExit(f"BED writer failed: {rc} {rc2}")
            return 1e3 * (time.perf_counter() - tb)
        tm = {"admission_ms": verdict["ms"], "device_pipeline_ms": 1e3 * (t2 - t0), "admission_replayed": st.get("replayed")}
        if defer_bed:
            # the context's interval buffer is reused by the next contig: the writer thread works on its own copy
            iv_copy = np.ctypeslib.as_array(C.cast(raw.intervals, C.POINTER(C.c_uint8)), shape=(n_iv * INTERVAL_DTYPE.itemsize,)).copy()
            tm["total_ms"] = 1e3 * (time.perf_counter() - t0)
            return raw, tm, (lambda: write_bed(iv_copy.ctypes.data_as(C.c_void_p), iv_copy))
        tm["bed_write_ms"] = write_bed(raw.intervals)
        tm["total_ms"] = 1e3 * (time.perf_counter() - t0)
        return raw, tm

    raw_first, _ = e2e_pass()                # also leaves the contig resident for the HBM-resident leg
    first = _result(raw_first, True)
    cells = int(first.summed_coverage)
    upload_ms = float(first.upload_ms)
    # size-independent properties of the full-size result
    assert cells == int(reads.ref_len()[(reads.flag & 4) == 0].sum()), "summed coverage != aligned bases of the admitted reads"
    assert int(first.state_counts.sum()) == c.length
    iv = first.intervals
    assert iv["start"][0] == 0 and iv["end"][-1] == c.length and np.array_equal(iv["start"][1:], iv["end"][:-1])
    assert np.all(iv["state"][1:] != iv["state"][:-1])
    assert np.array_equal(np.bincount(iv["state"], weights=(iv["end"] - iv["start"]).astype(np.float64), minlength=6).astype(np.int64),
                          first.state_counts.astype(np.int64))
    assert int(first.bins.sum()) == int(first.state_counts[0] + first.state_counts[1] + first.state_counts[5])
    n_intervals = int(iv.shape[0])
    gpu_bed_sha = hashlib.sha256(open(bed_path, "rb").read()).hexdigest()

    nccl = None
    if world > 1:
        nccl = Nccl(rank, world, dev)
        L.clb_set_nccl_allreduce(C.c_void_p(nccl.allreduce_fn))

    def allreduce_counters():
        if nccl is not None:
            ctx.allreduce_nccl(nccl.comm.value)

    # ---------------- HBM-resident leg: W warm-up + K timed steps, barrier + sync on both sides
    for _ in range(args.warmup):
        ctx.rerun_resident(fetch=False)
        allreduce_counters()
    sampler = ClockSampler(local_rank); sampler.start()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):                          # K steps queued back to back (clb_rerun_resident(ctx, NULL, NULL) only enqueues)
        ctx.rerun_resident(fetch=False, sync=False)
        allreduce_counters()
    ev1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    total_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.refresh_counters())     # the last timed step's result, before anything runs again
    step_ms = []                                         # per-step device times of three more steps, outside the timed region
    for _ in range(3):
        ms, _ = ctx.rerun_resident(fetch=False)
        allreduce_counters()
        step_ms.append(ms)
    allreduce_ok = None
    if world > 1:
        summed = ctx.refresh_counters()          # the last step's counters, all-reduced: N identical replicas
        allreduce_ok = bool(np.array_equal(summed.state_counts, first.state_counts * np.uint64(world))
                            and summed.summed_coverage == world * first.summed_coverage and summed.summed_baseq == world * first.summed_baseq
                            and np.array_equal(summed.bins.astype(np.uint64), first.bins.astype(np.uint64) * np.uint64(world)))
    _, res = ctx.rerun_resident(fetch=True, copy_intervals=True)
    pileup_ms, fast_ms, general_windows = res.pileup_ms, res.fast_ms, res.general_windows
    # what the resident steps compute is what the e2e pass (checked against the oracle below) computed
    resident_ok = bool(np.array_equal(res.intervals, first.intervals) and np.array_equal(res.state_counts, first.state_counts)
                       and np.array_equal(res.bins, first.bins) and res.summed_coverage == first.summed_coverage
                       and res.summed_baseq == first.summed_baseq and res.summed_mapq == first.summed_mapq
                       and res.quality_bases == first.quality_bases and res.n_covered_bases == first.n_covered_bases)
    if not resident_ok:
        raise SystemExit("the HBM-resident step does not reproduce the result of the e2e pass")
    launches_per_step = res.gpu_launches

    # ---------------- end-to-end leg through the public API with host buffers (admission and BED text inside)
    e2e_runs = []
    raw = raw_first
    for i in range(args.e2e_steps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        raw, tm = e2e_pass()
        allreduce_counters()
        torch.cuda.synchronize()
        e2e_runs.append(tm)
    e2e_best = min(e2e_runs, key=lambda t: t["total_ms"]) if e2e_runs else {"total_ms": float("nan")}
    # The same steps as consecutive contigs of a genome: contig i's BED text is formatted and written by a writer thread while
    # contig i + 1 is admitted and uploaded (what a host does between two process_single_contig calls).  Wall time of the
    # whole sequence, last BED file included, divided by the number of contigs.
    e2e_pipe_ms, pipe_n = float("nan"), max(0, args.e2e_pipelined)
    if pipe_n:
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        tp0 = time.perf_counter()
        writer, bed_ms = None, []
        for i in range(pipe_n):
            raw, _, job = e2e_pass(defer_bed=True)
            allreduce_counters()
            if writer is not None:
                writer.join()
            writer = threading.Thread(target=lambda j=job: bed_ms.append(j()))
            writer.start()
        writer.join()
        torch.cuda.synchronize()
        e2e_pipe_ms = 1e3 * (time.perf_counter() - tp0) / pipe_n
        if hashlib.sha256(open(bed_path, "rb").read()).hexdigest() != gpu_bed_sha:
            raise SystemExit("the BED file of the pipelined e2e leg differs from the first pass")
    # the ceiling the e2e leg runs against: a plain page-locked -> device copy of 1 GiB, all ranks at the same time
    copy_gbs = None
    if args.e2e_steps:
        nb = 1 << 30
        hsrc = torch.empty(nb, dtype=torch.uint8, pin_memory=True); hsrc.zero_()
        ddst = torch.empty(nb, dtype=torch.uint8, device=dev)
        ddst.copy_(hsrc, non_blocking=True); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(3):
            ddst.copy_(hsrc, non_blocking=True)
        c1.record(stream); torch.cuda.synchronize()
        copy_gbs = 3 * nb / (c0.elapsed_time(c1) * 1e-3) / 1e9
        del hsrc, ddst
    h2d_bytes, d2h_bytes, h2d_dev_ms = int(raw.h2d_bytes), int(raw.d2h_bytes), float(raw.h2d_ms)
    e2e_single_ms = e2e_best["total_ms"]
    e2e_best_ms = e2e_pipe_ms if pipe_n else e2e_single_ms

    # ---------------- strong scaling: ONE chr1 cut into N region shards (halo reads, all-reduce, stitching, parity)
    strong = None
    if world > 1 and not args.no_strong:
        window = int(L.clb_window_positions())
        plan = sharding.plan_regions([c.length], world, window)[rank]
        assert len(plan) == 1, plan                        # one contig: one window-aligned region per rank
        sh = plan[0]
        lo, hi = sharding.reads_for_region(reads, sh.start, sh.end, span)
        sub = reads.slice(lo, hi)
        # admission was decided for the whole contig above (nothing but placed-unmapped records refused; the kernels skip those)
        ctx2 = CallableLociContext(opt, device=local_rank)
        ctx2.set_stream(stream.cuda_stream)
        ctx2.begin_contig(0, "chr1", c.length, c.ref, c.length, region=(sh.start, sh.end), max_ref_span=span)
        ctx2.push_reads(sub)
        part = ctx2.finish_contig()
        for _ in range(args.warmup):
            ctx2.rerun_resident(fetch=False); ctx2.allreduce_nccl(nccl.comm.value)
        torch.cuda.synchronize(); dist.barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(args.steps):
            ctx2.rerun_resident(fetch=False, sync=False); ctx2.allreduce_nccl(nccl.comm.value)
        s1.record(stream)
        torch.cuda.synchronize(); dist.barrier()
        strong_ms = s0.elapsed_time(s1) / args.steps
        tot = ctx2.refresh_counters()
        stitched = sharding.gather_and_stitch(part.intervals, sh.start, dst=0)
        t_strong = torch.tensor([strong_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t_strong, op=dist.ReduceOp.MAX)
        ok, detail = None, None
        if rank == 0:
            detail = {"intervals": bool(stitched.shape == first.intervals.shape and np.array_equal(stitched["start"], first.intervals["start"])
                                        and np.array_equal(stitched["end"], first.intervals["end"]) and np.array_equal(stitched["state"], first.intervals["state"])),
                      "state_counts": bool(np.array_equal(tot.state_counts, first.state_counts)),
                      "sums": bool(tot.summed_coverage == first.summed_coverage and tot.summed_baseq == first.summed_baseq
                                   and tot.summed_mapq == first.summed_mapq and tot.quality_bases == first.quality_bases
                                   and tot.n_covered_bases == first.n_covered_bases),
                      "bins": bool(np.array_equal(tot.bins, first.bins))}
            ok = all(detail.values())
        strong = {"workload": f"the same chr1-size contig cut into {world} region shards (window-aligned), one per GPU",
                  "ms_per_step": float(t_strong[0]), "value": cells / (float(t_strong[0]) * 1e-3) / 1e9, "unit": UNIT,
                  "shard_reads": int(sub.n), "shard_bp": int(sh.end - sh.start), "sharded_parity": ok, "sharded_parity_detail": detail,
                  "exchange": "clb_allreduce_nccl (ncclAllReduce sum of 12 counters + 3 x n_bins bins, uint64) inside the step; interval "
                              "lists gathered and stitched on rank 0 outside it"}
        ctx2.close()

    # ---------------- max over ranks
    t_total = torch.tensor([total_ms, e2e_best_ms, float(cells), h2d_bytes / max(h2d_dev_ms, 1e-9) / 1e6, copy_gbs or 0.0, e2e_single_ms],
                           dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t_total.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t_total.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        tmin = t_total.clone(); dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        total_ms, e2e_best_ms, cells_all, e2e_single_ms = float(tmax[0]), float(tmax[1]), float(tsum[2]), float(tmax[5])
        h2d_rank_gbs = {"min": float(tmin[3]), "max": float(tmax[3])}
        copy_rank_gbs = {"min": float(tmin[4]), "max": float(tmax[4])}
    else:
        cells_all = float(cells)
        h2d_rank_gbs = {"min": float(t_total[3]), "max": float(t_total[3])}
        copy_rank_gbs = {"min": float(t_total[4]), "max": float(t_total[4])}

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = cells_all / (ms_per_step * 1e-3) / 1e9
        achieved = alg_bytes / (pileup_ms * 1e-3) / 1e9
        traffic, traffic_src = load_traffic(args.scale, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u32 integer", "data": "synthetic",
            "config": {"workload": WORKLOAD, "contig_bp": c.length, "reads": reads.n, "cells_per_rank": cells, "bed_intervals": n_intervals,
                       "scale": args.scale,
                       "l2_policy": f"inputs ({alg_bytes / 1e9:.2f} GB per step) are far larger than the 126 MB L2; no flush needed",
                       "parallelism": (f"{world} replicas of the contig, one per GPU, counters summed by clb_allreduce_nccl; see `strong` for the region-sharded run"
                                       if world > 1 else "single GPU"), **prep},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "k_pileup_fast (+ k_pileup_general for the windows it hands over)", "kernel_ms": pileup_ms,
                         "k_pileup_fast_ms": fast_ms, "general_windows": int(general_windows),
                         "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_cell": alg_bytes / cells, "peak_source": peak_src},
            "upload_kernels_ms": round(upload_ms, 3),
            "upload_kernels_note": "k_validate_batch + k_rebase_batch per column batch and k_nmask_from_ascii per contig run once at upload, "
                                   "outside the resident step `value` times (inside `e2e`)",
            "e2e": {"value": cells_all / (e2e_best_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_best_ms,
                    "steps": pipe_n if pipe_n else args.e2e_steps,
                    "pipelining": (f"{pipe_n} contigs back to back; contig i's BED text is written by a writer thread while contig i + 1 is admitted and "
                                   "uploaded; wall time of the whole sequence (last BED file included) / contigs" if pipe_n else "none: best single contig"),
                    "single_contig_ms": e2e_single_ms,
                    "single_contig_note": "one contig alone, nothing overlapped across contigs: admission || upload, kernels, D2H, then the BED file "
                                          "(best of --e2e-steps passes); the three *_ms fields below are this pass",
                    "admission_ms": round(e2e_best.get("admission_ms", float("nan")), 2),
                    "admission_note": "host threads, concurrent with the H2D copies (inside device_pipeline_ms, not added to it)",
                    "device_pipeline_ms": round(e2e_best.get("device_pipeline_ms", float("nan")), 2),
                    "bed_write_ms": round(e2e_best.get("bed_write_ms", float("nan")), 2),
                    "admission_replayed_reads": e2e_best.get("admission_replayed"),
                    "h2d_device_ms": round(h2d_dev_ms, 2), "h2d_GBps_per_rank": h2d_rank_gbs,
                    "h2d_ceiling_GBps_per_rank": copy_rank_gbs,
                    "h2d_ceiling_note": "plain cudaMemcpyAsync of 1 GiB page-locked -> device, all ranks at the same time: what the host's PCIe / memory "
                                        "system gives each rank; the e2e leg's copies run at h2d_GBps_per_rank",
                    "bed_bytes": os.path.getsize(bed_path),
                    "note": "per contig: clb_admit_reads_mt (htslib depth cap) + clb_begin_contig + clb_push_reads batches from page-locked host "
                            "columns + clb_finish_contig (D2H) + clb_bed_writer_* to a real file; the device part is PCIe-bound"},
            "resident_equals_e2e": resident_ok,
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
            "kernel_step_ms": {"min": min(step_ms), "median": statistics.median(step_ms), "max": max(step_ms)},
        }
        if world > 1:
            line["allreduce_verified"] = allreduce_ok
            line["nccl"] = {"library": nccl.path, "version": nccl.version}
            line["numa"] = numa
            if strong is not None:
                line["strong"] = strong
        if not args.no_cpu_baseline and world == 1:
            full = not args.no_parity_full
            sample_bp = c.length if full else int(min(args.cpu_sample_mbp * 1e6, c.length))
            oc, orun, dt, sub = oracle_run(c, reads, opt, sample_bp)
            line["cpu_baseline"] = {
                "value": oc.summed_coverage / dt / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": (f"the whole workload ({oc.summed_coverage} cells, {dt:.1f} s)" if full else
                           f"first {sample_bp} bp of the same contig ({oc.summed_coverage} cells, {dt:.1f} s)")
                          + f"; oracle/callable_oracle.c single-threaded like the reference, admission and BED text included; host has {os.cpu_count()} cores"}
            obed = orun.bed()
            if full:
                ok = (hashlib.sha256(obed).hexdigest() == gpu_bed_sha and first.state_counts.tolist() == oc.counts
                      and first.n_covered_bases == oc.n_covered_bases and first.summed_coverage == oc.summed_coverage
                      and first.summed_baseq == oc.summed_baseq and first.summed_mapq == oc.summed_mapq and first.quality_bases == oc.quality_bases
                      and oc.bins is not None and np.array_equal(first.bins, oc.bins))
                line["parity_full"] = bool(ok)
                line["parity_full_note"] = (f"whole contig: sha256 of the BED file written by the e2e leg ({len(obed)} bytes) == sha256 of the oracle's BED; "
                                            "6 state counts, 5 sums and 3 x n_bins bins equal")
            else:
                gctx = CallableLociContext(opt, device=local_rank)
                gctx.begin_contig(0, "chr1", sample_bp, c.ref[:sample_bp], sample_bp, max_ref_span=span)
                gctx.push_reads(compact_reads(sub, admit_reads(sub, maxcnt, 0)))
                g = gctx.finish_contig()
                from decodingustools_b200.callable_loci import CallableProfiler
                prof = CallableProfiler(None, sample_bp)
                gb = g.bins.copy()
                prof.add_contig("chr1", sample_bp, g.intervals, g.state_counts, gb, g.stride)
                ok = (prof.bed_bytes() == obed and g.state_counts.tolist() == oc.counts and g.summed_coverage == oc.summed_coverage
                      and g.summed_baseq == oc.summed_baseq and g.summed_mapq == oc.summed_mapq and g.quality_bases == oc.quality_bases
                      and g.n_covered_bases == oc.n_covered_bases and oc.bins is not None and np.array_equal(g.bins, oc.bins))
                line["parity_on_cpu_sample"] = bool(ok)
                gctx.close()
            del obed
        if not args.no_e2e_bam and world == 1:
            if ctx is not None:
                ctx.close(); ctx = None                  # free the resident contig: the command opens its own context
            line["e2e_bam"] = e2e_bam_leg(args, opt, local_rank)
        if not args.no_other_configs and world == 1:
            from decodingustools_b200 import synth
            from decodingustools_b200.options import CallableOptions
            if ctx is not None:
                ctx.close(); ctx = None                  # free the resident contig before the other configs
            others = []
            for tag, mk, o in (("configs[3] at reduced scale: 2000x, chrY-size/20, --max-depth 500 (cap active)",
                                lambda: synth.synth_short("chrY", 2_800_000, 4, depth=2000.0), CallableOptions()),
                               ("configs[3] variant: 2000x, 1 Mbp, --max-depth 4000 (no cap: true 2000x piles)",
                                lambda: synth.synth_short("chrY", 1_000_000, 4, depth=2000.0), CallableOptions(max_depth=4000)),
                               ("configs[4] at reduced scale: 15 kb indel-heavy long reads, 25 Mbp, 30x",
                                lambda: synth.synth_long("chr1", 25_000_000, 5), CallableOptions())):
                others.append(kernel_config_run(tag, mk(), o, peak))
            line["other_configs"] = others
        print(json.dumps(line), flush=True)
    if ctx is not None:
        ctx.close()
    try:
        os.remove(bed_path); os.rmdir(bed_dir)
    except OSError:
        pass
    if nccl is not None:
        nccl.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
