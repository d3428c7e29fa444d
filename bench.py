#!/usr/bin/env python
"""bench.py -- the reference's headline metric on the reference's headline workload (BASELINE.json):
aligned reads/s for `snap single`, 150 bp synthetic reads vs a 3 Gbp hg-sized synthetic reference, seed 20,
maxDist 14 (configs[1]), read-sharded over N GPUs -- and, in the same line, the other configs to the same bar.

A "step" is one pass of the hot path (seed lookup + LV / affine-gap scoring, BaseAligner::AlignRead semantics) over
one batch of synthetic reads.  `value` = reads of all ranks per second with the inputs already resident in HBM,
timed with CUDA events around exactly K steps (max over ranks).  `e2e` = the same metric through the C ABI call a
SNAP extension makes (snapgpu_align_single) with HOST buffers: host->device copies of the reads and device->host
copy of the results inside the timed region (aligner only: no FASTQ parsing, no SAM formatting).  `roofline` is for the
step's alignment launches taken together, timed with CUDA events on their stream.
`paired_phase` = BASELINE configs[2] (stock `snap paired`; at N > 1 this is configs[4]'s read-sharded shape),
`ag_forced_phase` = configs[3] (`-G -d 20` and `-ne -d 20`): each with its own value / e2e / roofline and, at N = 1, a
`cpu_baseline` whose `parity_vs_reference` compares the engine's records with the UNMODIFIED reference's on ~1 M reads
(0.5 M pairs) at the full 3 Gbp size.  Any `differing != 0`, and any exception in those legs, makes the run exit 3
after the line is printed.
`seed_phase` is the seed-lookup kernel run in isolation over every seed of the batch (BASELINE's second metric).
`cpu_baseline` / `--impl reference` time the UNMODIFIED reference (oracle/_ref, compiled from /root/reference) on the
host cores, on a bounded sample of the same workload, against the same index written out in the reference's own
directory format into tmpfs with its pages interleaved over the NUMA nodes (the protocol of BASELINE.md 3: threads started
before the clock, >= 5 s timed, stock flags and -march=x86-64-v3, 1-thread and all-thread rates, a stock-CLI cross-check).
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the tree may be read-only: nothing is written there, not even __pycache__
sys.path.insert(0, ROOT)

READ_LEN = 150
SEED_LEN = 20
MAX_DIST = 14
ALG_BYTES_PER_CANDIDATE = READ_LEN - SEED_LEN + 2 * (MAX_DIST + 1)     # SURVEY 8d: (readLen - seedLen + 2*k_used) reference bytes
ALG_BYTES_PER_READ_IO = 2 * READ_LEN + 88                              # bases + qualities in, result record out
# stock `snap paired` (BASELINE configs[2] names no options): -d 27, -n 8, -H 4000, -s 0 1000, soft clipping on
PAIRED_MAX_DIST = 27
PAIRED_KW = dict(maxDist=PAIRED_MAX_DIST, numSeedsFromCommandLine=8)
PAIRED_PKW = dict()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--genome-mbp", type=int, default=int(os.environ.get("SNAPGPU_BENCH_GENOME_MBP", "3000")),
                    help="total reference size in Mbp (24 contigs); 3000 = BASELINE configs[1]")
    ap.add_argument("--batch-reads", type=int, default=int(os.environ.get("SNAPGPU_BENCH_BATCH", str(1 << 20))),
                    help="reads per step per GPU")
    ap.add_argument("--cpu-sample-reads", type=int, default=1000000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-seed-phase", action="store_true")
    ap.add_argument("--workload", default=os.environ.get("SNAPGPU_BENCH_WORKLOAD", "single"), choices=["single", "paired", "ag_d20", "ne_d20"],
                    help="the HEADLINE workload (timed over exactly --steps): single = BASELINE configs[1] (default); paired = configs[2]; "
                         "ag_d20 / ne_d20 = configs[3].  The others still run, as paired_phase / ag_forced_phase, unless --only-headline")
    ap.add_argument("--only-headline", action="store_true", help="skip the other configs' phases (profiling runs)")
    ap.add_argument("--no-sam-phase", action="store_true")
    ap.add_argument("--no-stress-phase", action="store_true")
    ap.add_argument("--no-cli-crosscheck", action="store_true")
    ap.add_argument("--repeat-frac", type=float, default=float(os.environ.get("SNAPGPU_BENCH_REPEAT_FRAC", "0")),
                    help="SURVEY 8d stress variant: this fraction of the reference is drawn from a 10 kbp repeat library at 0-5 %% divergence")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the headline's result records of the last timed step (rank 0) as DIR/<field>.npy")
    return ap.parse_args()


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [l.strip().split(",") for l in open(self.path) if l.strip()]
            sm = [float(r[0]) for r in rows if r[0].strip().replace(".", "").isdigit()]
            if sm:
                out["sm_mhz"] = float(np.median(sm))
                out["sm_max_mhz"] = float(rows[0][1])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for k, nme in enumerate(names):
                if any(len(r) > 4 + k and "Active" in r[4 + k] and "Not" not in r[4 + k] for r in rows):
                    out["reasons"].append(nme)
            out["samples"] = len(rows)
        except Exception:
            pass
        finally:
            try:
                os.unlink(self.path)
            except Exception:
                pass
        return out



# ---- the workloads of BASELINE.json's configs (SURVEY 8d command lines) ----
WORKLOADS = {
    # configs[1]: `snap single idx r150.fq -d 14` -- the headline
    "single": dict(kind="single", kw=dict(maxDist=MAX_DIST), pkw=None, max_dist=MAX_DIST, config="BASELINE configs[1]",
                   cli="snap-aligner single idx3G r150.fq -d 14"),
    # configs[2] (and, sharded, configs[4]): stock `snap paired`
    "paired": dict(kind="paired", kw=PAIRED_KW, pkw=PAIRED_PKW, max_dist=PAIRED_MAX_DIST, config="BASELINE configs[2] (configs[4] when sharded over N GPUs)",
                   cli="snap-aligner paired idx3G r1.fq r2.fq   (stock options: -d 27 -n 8 -H 4000 -s 0 1000, soft clipping on)"),
    # configs[3]: the same reads, maxDist 20, affine gap "forced": -G re-asserts the default (AlignerOptions.cpp:696-701) ...
    "ag_d20": dict(kind="single", kw=dict(maxDist=20, useAffineGap=1), pkw=None, max_dist=20, config="BASELINE configs[3], -G",
                   cli="snap-aligner single idx3G r150.fq -d 20 -G"),
    # ... and -ne is what rescores EVERY candidate with affine gap (AlignerOptions.cpp:964-967; it also clears useAffineGap)
    "ne_d20": dict(kind="single", kw=dict(maxDist=20, noEditDistance=1, useAffineGap=0), pkw=None, max_dist=20, config="BASELINE configs[3], -ne",
                   cli="snap-aligner single idx3G r150.fq -d 20 -ne"),
}


sys.path.insert(0, os.path.join(ROOT, "profiles"))
from kernel_stamp import csrc_sha16, sass_sha16_for       # noqa: E402  profiles/traffic.json records both stamps of the kernels its ncu capture
                                                          # was taken of; the line only quotes `traffic` / `issue_slots` from a capture of THESE kernels


def traffic_entry(workload, batch_reads, genome_mbp):
    """(entry or None, why-not).  The entry is ONE step's alignment launches from `ncu --set full` (profiles/refresh_traffic.sh)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None, "profiles/traffic.json unreadable"
    key = "%s_%dreads_%dmbp" % (workload, batch_reads, genome_mbp)
    if key not in t:
        return None, "no capture of this workload"
    e = dict(t[key])
    if e.get("csrc_sha16") == csrc_sha16():
        e["stamp"] = "csrc_sha16 %s" % e["csrc_sha16"] + ("; captured at csrc_sha16 %s, %s" % (e.get("csrc_sha16_at_capture"), e["restamped"]) if e.get("restamped") else "")
        return e, None
    now = sass_sha16_for(key)
    if e.get("sass_sha16") and now and e["sass_sha16"] == now:
        e["stamp"] = "sass_sha16 %s (the SASS of these kernels is what was captured; other sources of the library changed since)" % now
        return e, None
    return None, "capture is of other kernels (csrc_sha16 %s, now %s; sass_sha16 %s, now %s): refresh with profiles/refresh_traffic.sh" % (
        e.get("csrc_sha16"), csrc_sha16(), e.get("sass_sha16"), now)


class Ctx:
    """Everything the workloads share on one rank: device, the genome and index in HBM, the reads, rank / world."""
    pass


def build_context(args, repeat_frac=None, like=None):
    """like: an existing context whose rank / device / process group this one shares (the stress genome's context)."""
    import torch
    import torch.distributed as dist
    from snap_b200 import engine, synth_device
    c = Ctx()
    if repeat_frac is None:
        repeat_frac = args.repeat_frac
    c.rank = int(os.environ.get("RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if c.world != args.gpus and c.world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, c.world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    c.device = torch.device("cuda", c.local_rank)
    torch.cuda.set_device(c.device)
    if c.world > 1 and like is None:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=c.device)
    n_contigs = 24
    c.contig_len = args.genome_mbp * 1_000_000 // n_contigs
    t0 = time.time()
    c.bases, c.starts = synth_device.make_genome(n_contigs, c.contig_len, seed=20260924, device=c.device)
    if repeat_frac > 0:
        synth_device.plant_repeats(c.bases, c.starts, c.contig_len, repeat_frac, seed=77)
    torch.cuda.synchronize()
    t1 = time.time()
    c.idx = engine.Index.build_device(c.bases.data_ptr(), c.bases.numel(), c.starts, seed_len=SEED_LEN, chromosome_padding=2000, device=c.device.index or 0)
    torch.cuda.synchronize()
    t2 = time.time()
    info = c.idx.info()
    c.setup = {"genome_s": round(t1 - t0, 2), "index_build_s": round(t2 - t1, 2), "index_hbm_gb": round(info.hbmBytes / 1e9, 2),
               "overflow_words": int(info.overflowTableSize)}
    c.peak, c.peak_src = measured_peaks()
    c.ref = None
    c.repeat_frac = repeat_frac
    return c


def make_batches(c, args, kind, n):
    """n batches of this rank's shard: every (rank, step) has its own reads; the global batch of a step is the concatenation over ranks."""
    from snap_b200 import synth_device
    out = []
    for b in range(n):
        seed = 1000 + b * 64 + c.rank
        if kind == "paired":
            out.append(synth_device.make_pairs(c.bases, c.starts, c.contig_len, args.batch_reads // 2, READ_LEN, seed=seed))
        else:
            out.append(synth_device.make_reads(c.bases, c.starts, c.contig_len, args.batch_reads, READ_LEN, seed=seed))
    return out


def to_host_batch(dev_batch, pinned=True):
    from snap_b200 import synth
    rb, rq, ro, rl = dev_batch[:4]
    if pinned:
        return synth.ReadBatch(rb.cpu().pin_memory().numpy(), rq.cpu().pin_memory().numpy(), ro.cpu().numpy().astype(np.uint64), rl.cpu().numpy().astype(np.uint32))
    return synth.ReadBatch(rb.cpu().numpy(), rq.cpu().numpy(), ro.cpu().numpy().astype(np.uint64), rl.cpu().numpy().astype(np.uint32))


DUMP_LIMIT = 64 * 10**6                 # bytes of all the .npy files --dump-outputs writes


def dump_outputs(d, records):
    """The result records a caller of the timed path receives, one float64 array per field (paired fields are [pairs, 2]), as d/<field>.npy.
    When all rows would not fit in DUMP_LIMIT bytes, a fixed sample of rows (seed 0, ascending) is written, with its row numbers as
    d/rows.npy; the inputs are seeded, so two builds run with the same arguments can be compared array for array."""
    names = [f for f in records.dtype.names if f != "reserved"]
    row_bytes = 8 + sum(8 * int(np.prod(records.dtype[f].shape)) for f in names)
    n = len(records)
    m = min(n, (DUMP_LIMIT - (1 << 16)) // row_bytes)           # 64 KiB left for the .npy headers
    rows = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "rows.npy"), rows.astype(np.float64))
    for f in names:
        np.save(os.path.join(d, f + ".npy"), records[f][rows].astype(np.float64))


def run_workload(c, args, name, batches, W, K, sample_clocks=False, dump_dir=None):
    """One workload on this rank (all ranks call it together): device-resident timing over exactly K steps after W warm-ups, then the
    same through the C ABI with host buffers.  Returns the workload's object; ["_records"] holds the engine's records for batches[0]
    (rank 0, for the parity leg), ["_host0"] those reads on the host.  dump_dir: where rank 0 writes the records of the last timed step."""
    import torch
    import torch.distributed as dist
    from snap_b200 import engine, shard
    wl = WORKLOADS[name]
    paired = wl["kind"] == "paired"
    B = (args.batch_reads // 2) * 2 if paired else args.batch_reads
    n_units = B // 2 if paired else B
    device, world, rank = c.device, c.world, c.rank
    if paired:
        al = engine.PairedAligner(c.idx, engine.default_params(**wl["kw"]), engine.default_paired_params(**wl["pkw"]), max_batch_pairs=n_units)
        res_dtype = engine.PAIRED_RESULT_DTYPE
    else:
        al = engine.SingleAligner(c.idx, engine.default_params(**wl["kw"]), max_batch_reads=B)
        res_dtype = engine.RESULT_DTYPE
    result_bytes_per_read = res_dtype.itemsize // (2 if paired else 1)
    # a dedicated (non-default) stream: the kernels are launched on it through the C ABI and the CUDA events that time
    # them are recorded on the same stream (a NULL stream argument would mean "the aligner's own stream")
    stream = torch.cuda.Stream(device)
    assert stream.cuda_stream != 0
    res = torch.zeros((n_units, res_dtype.itemsize), dtype=torch.uint8, device=device)
    d_ctr = torch.zeros((engine.N_COUNTERS,), dtype=torch.int64, device=device)

    def step(b):
        rb, rq, ro, rl = batches[b][:4]
        al.align_device(n_units, rb.data_ptr(), rq.data_ptr(), ro.data_ptr(), rl.data_ptr(), res.data_ptr(), d_ctr.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ----
    for b in range(W):
        step(b)
    barrier()
    d_ctr.zero_()
    sampler = ClockSampler(c.local_rank)
    if sample_clocks and rank == 0:
        sampler.start()
    launches0 = al.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    barrier()
    ev[0].record(stream)
    for k in range(K):
        step(W + k)
        ev[k + 1].record(stream)
    barrier()
    clocks = sampler.stop() if (sample_clocks and rank == 0) else {}
    ms_total = ev[0].elapsed_time(ev[K])
    kernel_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(K)]
    launches = al.launch_count() - launches0
    if paired:
        al.check(stream.cuda_stream)        # raises if a kernel latched an error (pool overflow)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, res.cpu().numpy().view(res_dtype).reshape(-1))
    ctr = d_ctr.cpu().numpy()
    ms_max = shard.max_over_ranks(ms_total, device) if world > 1 else ms_total
    ctr_all = shard.allreduce_counters(ctr, device) if world > 1 else ctr
    cd = engine.counters_dict(ctr_all)
    value = B * K * world / (ms_max / 1e3)

    # ---- end to end through the C ABI: reads in pinned HOST memory, records back in pinned host memory, copies inside the clock ----
    host_batches = [to_host_batch(batches[b]) for b in range(min(3, W + K))]
    res_host = torch.empty((n_units * res_dtype.itemsize,), dtype=torch.uint8).pin_memory().numpy().view(res_dtype)
    for b in range(2):
        al.align(host_batches[b % len(host_batches)], out=res_host)         # warm-ups
    barrier()
    e2e_steps = max(3, min(K, 10))
    t0 = time.perf_counter()
    n_e2e = 0
    for k in range(e2e_steps):
        r, _ = al.align(host_batches[k % len(host_batches)], out=res_host)
        n_e2e += len(r) * (2 if paired else 1)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_s = shard.max_over_ranks(e2e_s, device) if world > 1 else e2e_s
    e2e_value = n_e2e * world / e2e_s
    records0 = None
    if rank == 0 and world == 1:
        records0, _ = al.align(host_batches[0])
        records0 = records0.copy()

    # ---- roofline of the step's alignment launches taken together (algorithmic bytes of the step / its duration) ----
    per_step = 1.0 / (K * world)
    alg_cand = READ_LEN - SEED_LEN + 2 * (wl["max_dist"] + 1)
    alg_bytes = (cd["nHashEntriesProbed"] * 8 + cd["nOverflowWordsRead"] * 4 + (cd["lvCalls"] + cd["affineGapCalls"]) * alg_cand
                 + cd["totalReads"] * (2 * READ_LEN + result_bytes_per_read)) * per_step
    kernel_ms_avg = float(np.mean(kernel_ms))
    achieved = alg_bytes / (kernel_ms_avg / 1e3) / 1e9
    entry, why = traffic_entry(name, B, args.genome_mbp)
    roofline = {"kernel": ("sg_align_paired_kernel<.,1..3> (staged launch: seed/LV, affine gap, single-end fallback) + retry pass" if paired else
                           "sg_align_kernel<.,1> + <.,2> (two-pass launch)" if not wl["kw"].get("noEditDistance") else "sg_align_kernel<.,0> (one launch: every candidate is rescored)"),
                "launches_per_step": round(launches / K, 2), "bound": "hbm", "achieved": round(achieved, 3), "peak": c.peak, "unit": "GB/s",
                "frac": round(achieved / c.peak, 6), "traffic": int(entry["dram_bytes_per_launch"]) if entry else None, "peak_source": c.peak_src,
                "algorithmic_bytes_per_step": int(alg_bytes), "avg_step_ms": round(kernel_ms_avg, 3),
                "note": "latency/issue-bound integer state machine: ~%.0f B of index+reference+read traffic per read" % (alg_bytes / B)}
    if entry:
        roofline["traffic_over_algorithmic"] = round(entry["dram_bytes_per_launch"] / max(1.0, alg_bytes), 2)
        roofline["traffic_source"] = "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one step's launches of these kernels (%s), captured with `%s`" % (entry["stamp"], str(entry.get("captured_with", "ncu"))[:160])
        n_inst = entry.get("warp_instructions_per_step")
        sm_mhz = clocks.get("sm_mhz") or c.__dict__.get("sm_mhz")
        if n_inst and sm_mhz:
            sms = torch.cuda.get_device_properties(device).multi_processor_count
            issue_peak = sms * 4 * float(sm_mhz) * 1e6
            issue_ach = n_inst / (kernel_ms_avg / 1e3)
            roofline["issue_slots"] = {"warp_instructions_per_step": int(n_inst), "achieved_per_s": round(issue_ach, 1), "peak_per_s": round(issue_peak, 1),
                                       "frac": round(issue_ach / issue_peak, 4)}
    else:
        roofline["traffic_note"] = why
    if clocks.get("sm_mhz"):
        c.sm_mhz = clocks["sm_mhz"]

    out = {"workload": wl["cli"], "config": wl["config"], "value": round(value, 1), "unit": "reads/s", "steps": K, "warmup": W,
           "ms_per_step": round(ms_max / K, 3), "reads_per_step": B * world,
           "e2e": {"value": round(e2e_value, 1), "unit": "reads/s", "h2d_bytes_per_step": int(B * (2 * READ_LEN + 12)),
                   "d2h_bytes_per_step": int(B * result_bytes_per_read + engine.N_COUNTERS * 8), "steps": e2e_steps,
                   "scope": "aligner only, through snapgpu_align_%s with host buffers (reads already parsed, no SAM formatting)" % ("paired" if paired else "single")},
           "gpu_launches": int(launches), "roofline": roofline,
           "per_read": {"lookups": round(cd["nHashTableLookups"] / max(1, cd["totalReads"]), 3),
                        "hash_entries_per_lookup": round(cd["nHashEntriesProbed"] / max(1, cd["nHashTableLookups"]), 3),
                        "overflow_words": round(cd["nOverflowWordsRead"] / max(1, cd["totalReads"]), 3),
                        "lv_locations": round(cd["lvCalls"] / max(1, cd["totalReads"]), 3),
                        "ag_locations": round(cd["affineGapCalls"] / max(1, cd["totalReads"]), 3),
                        "aligned_frac": round((cd["singleHits"] + cd["multiHits"]) / max(1, cd["totalReads"]), 5)},
           "_clocks": clocks, "_records": records0, "_host0": host_batches[0], "_host_batches": host_batches}
    al.close()
    del res, res_host
    torch.cuda.empty_cache()
    return out


class RefContext:
    """The unmodified reference (oracle/_ref) over the same index, written out once in SNAP's own directory format into tmpfs with its
    pages interleaved over the NUMA nodes, and mapped (GenomeIndex::loadFromDirectory(map = true), what stock `-map` does)."""

    def __init__(self, idx):
        from oracle import reflib
        self.reflib = reflib
        self.nodes = reflib.numa_interleave()
        t0 = time.time()
        self.dir = export_index_for_reference(idx)
        self.export_s = time.time() - t0
        t0 = time.time()
        self.ridx = {"stock": reflib.RefIndex(self.dir, "stock", map_files=True, prefetch=False)}
        self.load_s = time.time() - t0
        if reflib.available_v3():
            self.ridx["v3"] = reflib.RefIndex(self.dir, "v3", map_files=True, prefetch=False)
        self.cores = os.cpu_count() or 1

    def host(self):
        sockets = set()
        model = ""
        try:
            for l in open("/proc/cpuinfo"):
                if l.startswith("physical id"):
                    sockets.add(l.split(":")[1].strip())
                elif l.startswith("model name") and not model:
                    model = l.split(":")[1].strip()
        except Exception:
            pass
        return {"cpu": model, "hw_threads": self.cores, "sockets": max(1, len(sockets)), "numa_nodes_interleaved": self.nodes,
                "threads_used": getattr(self, "threads", self.cores), "thread_sweep_reads_per_s": getattr(self, "thread_sweep", None),
                "thread_sweep_note": "fastest (thread count, pinning) of the sweep is used: the reference adds to one process-wide counter per probe chain (HashTable.h:109-110), which stops it scaling across sockets",
                "pinning": ("thread t pinned to logical CPU t (stock -b)" if getattr(self, "pinned", False) else "threads unpinned") + "; index pages interleaved over the memory nodes with MPOL_INTERLEAVE (= numactl --interleave=all)",
                "index": "ours, exported to SNAP's directory format in tmpfs (%.0f s), mapped like stock -map (%.1f s)" % (self.export_s, self.load_s)}

    def run(self, name, batch, threads, build="stock", reps=1):
        """(records, counters, seconds for `reps` passes)"""
        wl = WORKLOADS[name]
        rl = self.reflib
        if wl["kind"] == "paired":
            p, pp = rl.default_params(**wl["kw"]), rl.default_paired_params(**wl["pkw"])
            return rl.paired_align_mt(self.ridx[build], p, pp, batch, threads, reps)
        return rl.align_mt(self.ridx[build], rl.default_params(**wl["kw"]), batch, threads, reps)

    def pick_threads(self, name, batch):
        """The reference does not scale to every hardware thread of a two-socket box: GetFirstValueForKey adds to a process-wide counter
        on every probe chain (`nProbesInGetEntryForKey += nProbes`, HashTable.h:109-110), one cache line all threads write.  So the
        thread count (stock -t) is swept on a small sample and the FASTEST is what the baseline is quoted at."""
        if getattr(self, "threads", None):
            return self.threads
        m = min(batch.n, 500000) // 2 * 2
        sample = batch.slice(0, m)
        sweep = {}
        cands = sorted(set(t for t in (self.cores // 8, self.cores // 4, self.cores // 2, self.cores) if t >= 1))
        self.run(name, sample, self.cores)
        best = (0.0, self.cores, False)
        for pin in (False, True):
            self.reflib.set_thread_pinning(pin, builds=tuple(self.ridx))
            for t in cands:
                rate = round(m / self.run(name, sample, t)[2], 1)
                sweep["%d%s" % (t, " pinned" if pin else "")] = rate
                if rate > best[0]:
                    best = (rate, t, pin)
        self.thread_sweep = sweep
        self.threads, self.pinned = best[1], best[2]
        self.reflib.set_thread_pinning(self.pinned, builds=tuple(self.ridx))
        return self.threads

    def close(self):
        shutil.rmtree(self.dir, ignore_errors=True)


def cpu_leg(ref, args, name, host_batch, records, min_seconds=3.0, builds=("stock",), one_thread=False):
    """The reference on all host threads over a bounded sample of the step's reads: its rate, and its records against the engine's
    for the same reads (full-size parity: 3 Gbp index, ~1 M reads / 0.5 M pairs)."""
    wl = WORKLOADS[name]
    paired = wl["kind"] == "paired"
    n = min(args.cpu_sample_reads, host_batch.n)
    n -= n % 2
    sample = host_batch.slice(0, n)
    units = n // 2 if paired else n
    T = ref.pick_threads(name, sample)
    ref.run(name, sample.slice(0, min(n, 20000)), T)               # warm the page cache / TLB
    want, ctr, secs1 = ref.run(name, sample, T)
    reps = int(max(1, min(40, np.ceil(min_seconds / max(secs1, 1e-3)))))
    _, _, secs = ref.run(name, sample, T, reps=reps) if reps > 1 else (None, None, secs1)
    out = {"value": round(n * reps / secs, 1), "unit": "reads/s", "cores": T, "kind": "reference",
           "sample": "%d of the step's %d %s x %d passes = %.1f s, %d threads started before the clock, oracle/_ref %s (aligner only, no SAM output)"
                     % (units, host_batch.n // (2 if paired else 1), "pairs" if paired else "reads", reps, secs, T,
                        "ChimericPairedEndAligner(IntersectingPairedEndAligner)::align" if paired else "BaseAligner::AlignRead"),
           "seconds": round(secs, 3), "build": "-O3 -std=c++98 -msse (the reference Makefile's flags)",
           "lv_per_read": round(ctr["lvCalls"] / n, 3), "ag_per_read": round(ctr["affineGapCalls"] / n, 3)}
    if "v3" in builds and "v3" in ref.ridx:
        ref.run(name, sample.slice(0, min(n, 20000)), T, build="v3")
        _, _, s3 = ref.run(name, sample, T, build="v3", reps=reps)
        out["value_march_x86_64_v3"] = round(n * reps / s3, 1)
        out["build_v3"] = "-O3 -march=x86-64-v3 (stands in for -march=native: the build host is not the bench host)"
    if one_thread:
        m = min(n, 20000)
        _, _, s1 = ref.run(name, sample.slice(0, m), 1)
        out["value_1thread"] = round(m / s1, 1)
    if paired:
        out["aligned_as_pair_frac"] = round(float(want["alignedAsPair"].mean()), 5)
    parity = None
    if records is not None:
        differing, skipped = count_differing(want, records[:units], paired)
        parity = {("pairs_compared" if paired else "reads_compared"): units, "differing": differing, "n_skipped": skipped,
                  "skip_rule": ("none; mapq / scorePriorToClipping of ends reported NotFound are zeroed on both sides (uninitialised in the reference)" if paired else
                                "records BOTH sides report NotFound (the reference leaves their other fields uninitialised)")}
    out["parity_vs_reference"] = parity
    return out


def seed_phase(args, idx, batches, device, peak, peak_src):
    """The seed-lookup kernel alone over the 7 non-overlapping seeds of every read of one batch (BASELINE's second metric), against two
    measured ceilings: the streaming copy peak, and the device's random 32-byte-sector read rate over a table of the index's size (a
    hash probe IS a random sector read, so that rate / sectors per lookup bounds lookups/s).
    Algorithmic bytes per lookup = the bytes the lookup has to examine: slots examined x 8 B (whole 32-byte buckets on the sector-bucket
    layout, entries of both probe chains on the reference's layout) + overflow words x 4 B + the seed's own 20 bytes."""
    import torch
    from snap_b200 import engine
    B = args.batch_reads
    rb = batches[0][0].reshape(B, READ_LEN)
    offs = [0, 20, 40, 60, 80, 100, 120]
    seeds = torch.stack([rb[:, o:o + SEED_LEN] for o in offs], dim=1).contiguous()       # [B, 7, 20]
    n = B * len(offs)
    nh = torch.empty((n * 2,), dtype=torch.int64, device=device)
    probes = torch.empty((n,), dtype=torch.int32, device=device)
    st = torch.cuda.Stream(device)
    torch.cuda.synchronize()
    for _ in range(3):
        idx.lookup_seeds_device(seeds.data_ptr(), n, nh.data_ptr(), 0, probes.data_ptr(), 0, st.cuda_stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record(st)
    for _ in range(reps):
        idx.lookup_seeds_device(seeds.data_ptr(), n, nh.data_ptr(), 0, probes.data_ptr(), 0, st.cuda_stream)
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    entries = int(probes.to(torch.int64).sum().item())
    multi = nh[nh > 1]
    overflow_words = int((multi + 1).sum().item())
    info = idx.info()
    bucket = int(info.reserved) == 1
    alg = entries * 8 + overflow_words * 4 + n * SEED_LEN
    index_bytes = entries * 8 + overflow_words * 4
    table_bytes = int(info.hashTableSlots) * 8
    sector_rate = engine.measure_random_sector_rate(table_bytes, 1 << 26, device.index or 0)
    sectors = entries / 4 if bucket else entries           # reference layout: every entry examined sits in a sector of its own (quadratic / far-apart probes)
    achieved = alg / (ms / 1e3) / 1e9
    lookups_per_s = n / (ms / 1e3)
    out = {"kernel": "sg_lookup_bucket_kernel (one thread per seed, 32-byte sector buckets keyed by the canonical seed)" if bucket else "sg_lookup_kernel (one warp per seed, the reference's table layout)",
           "layout": "sector buckets (sg_bucket.h)" if bucket else "reference tables", "seeds": n, "ms": round(ms, 3), "lookups_per_s": round(lookups_per_s, 1),
           "slots_examined_per_lookup": round(entries / n, 3), "sectors_per_lookup": round(sectors / n, 3),
           "algorithmic_bytes_per_lookup": round(alg / n, 2), "index_bytes_per_lookup": round(index_bytes / n, 2),
           "achieved_algorithmic_gbs": round(achieved, 2), "peak_stream_gbs": peak, "peak_source": peak_src, "frac_of_stream_peak": round(achieved / peak, 5),
           "random_sector_peak": {"sectors_per_s": round(sector_rate, 1), "gbs": round(sector_rate * 32 / 1e9, 1), "table_gb": round(table_bytes / 1e9, 1),
                                  "how": "snapgpu_measure_random_sector_rate: random aligned 32 B reads over a table of the index's size, one per thread in flight, best of 3"},
           "achieved_sectors_per_s": round(sectors / (ms / 1e3), 1),
           "frac_of_random_sector_peak": round(sectors / (ms / 1e3) / sector_rate, 4),
           "index_gbs_as_sectors": round(sectors * 32 / (ms / 1e3) / 1e9, 1)}
    entry, why = traffic_entry("lookup", B, args.genome_mbp)
    if entry:
        out["dram_bytes_per_lookup"] = round(entry["dram_bytes_per_launch"] / n, 1)
        out["dram_over_algorithmic"] = round(entry["dram_bytes_per_launch"] / alg, 2)
        out["dram_source"] = "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel (%s), captured with `%s`" % (entry["stamp"], str(entry.get("captured_with", "ncu"))[:160])
    else:
        out["dram_bytes_per_lookup"] = None
        out["dram_note"] = why
    return out


def ingest_phase(args, host_batch, device, peak, peak_src):
    """FASTQ ingest (SURVEY 8f N2): snapgpu_fastq_parse_device over the FASTQ text of one batch, text resident in HBM.
    Algorithmic bytes = text read once + clipped bases and qualities + offsets/lengths/id table written once."""
    import torch
    from snap_b200 import engine
    n = host_batch.n
    L = READ_LEN
    rec = 2 + 8 + 1 + L + 3 + L + 1
    txt = np.empty((n, rec), dtype=np.uint8)
    txt[:, 0] = ord("@"); txt[:, 1] = ord("r")
    ids = np.arange(n, dtype=np.int64)
    for d in range(8):
        txt[:, 2 + 7 - d] = (ids // 10 ** d % 10 + 48).astype(np.uint8)
    txt[:, 10] = 10
    txt[:, 11:11 + L] = host_batch.bases.reshape(n, L)
    txt[:, 11 + L] = 10; txt[:, 12 + L] = ord("+"); txt[:, 13 + L] = 10
    q = host_batch.quals.reshape(n, L).copy()
    q[::7, L - 9:] = ord("#")                       # every 7th read carries a '#' tail the reader clips
    txt[:, 14 + L:14 + 2 * L] = q
    txt[:, 14 + 2 * L] = 10
    text = txt.reshape(-1)
    d_text = torch.from_numpy(text).to(device)
    fq = engine.FastqParser(max_bytes=int(text.size) + 64, max_reads=n + 8, device=device.index or 0)
    d_b = torch.empty((text.size // 2 + 64,), dtype=torch.uint8, device=device); d_q = torch.empty_like(d_b)
    d_off = torch.empty((n + 8,), dtype=torch.int64, device=device); d_len = torch.empty((n + 8,), dtype=torch.int32, device=device)
    d_ido = torch.empty((n + 8,), dtype=torch.int64, device=device); d_idl = torch.empty((n + 8,), dtype=torch.int32, device=device)
    d_fc = torch.empty((n + 8,), dtype=torch.int32, device=device)
    st = torch.cuda.Stream(device)

    def run():
        return fq.parse_device(d_text.data_ptr(), int(text.size), 2, d_b.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_ido.data_ptr(),
                               d_idl.data_ptr(), d_fc.data_ptr(), st.cuda_stream)
    for _ in range(3):
        nr, used = run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record(st)
    for _ in range(reps):
        run()
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    kept = int(d_len[:nr].to(torch.int64).sum().item())
    alg = int(text.size) + 2 * kept + nr * (8 + 4 + 8 + 4 + 4)
    out = {"kernels": "sg_fastq_count/positions/records/copy + 2 cub scans", "reads": int(nr), "text_bytes": int(text.size), "ms": round(ms, 3),
           "text_gbs": round(text.size / (ms / 1e3) / 1e9, 2), "reads_per_s": round(nr / (ms / 1e3), 1),
           "achieved_algorithmic_gbs": round(alg / (ms / 1e3) / 1e9, 2), "peak_gbs": peak, "peak_source": peak_src,
           "frac": round(alg / (ms / 1e3) / 1e9 / peak, 4), "bytes_consumed_ok": bool(used == text.size)}
    try:
        from oracle import reflib
        if reflib.available():
            m = min(n, 200000)
            t0 = time.perf_counter()
            reflib.fastq_parse(text[:m * rec], 2)
            dt = time.perf_counter() - t0
            out["cpu_reference_1thread_text_gbs"] = round(m * rec / dt / 1e9, 3)
    except Exception as e:  # pragma: no cover
        out["cpu_reference_error"] = str(e)[:100]
    fq.close()
    return out


def sam_phase(args, c, host_batch, paired):
    """Output stage (SURVEY 8f N1) on the headline's first batch, single-end: (1) the formatter alone with everything resident in HBM
    (snapgpu_sam_format_single_device: reads as parsed on the device, the engine's own records, packed SAM text left in HBM; CUDA events);
    (2) the same through the host-buffer ABI; (3) `e2e_with_output`: FASTQ text in pinned host memory -> H2D -> parse (device) -> align
    (device) -> SAM records (device) -> D2H of the text, one batch after the other, wall clock."""
    import torch
    from snap_b200 import engine, synth
    device = c.device
    if paired:
        return {"note": "measured for the single-end headline only"}
    n = host_batch.n
    L = READ_LEN
    text = fastq_text(host_batch)
    h_text = torch.from_numpy(text).pin_memory()
    p = engine.default_params(maxDist=MAX_DIST)
    al = engine.SingleAligner(c.idx, p, max_batch_reads=n)
    fq = engine.FastqParser(max_bytes=int(text.size) + 64, max_reads=n + 8, device=device.index or 0)
    fmt = engine.SamFormatter(c.idx, p, n, use_m=True)
    st = torch.cuda.Stream(device)
    d_text = torch.empty((text.size + 64,), dtype=torch.uint8, device=device)
    d_b = torch.empty((text.size // 2 + 64,), dtype=torch.uint8, device=device); d_q = torch.empty_like(d_b)
    d_off = torch.empty((n + 8,), dtype=torch.int64, device=device); d_len = torch.empty((n + 8,), dtype=torch.int32, device=device)
    d_ido = torch.empty((n + 8,), dtype=torch.int64, device=device); d_idl = torch.empty((n + 8,), dtype=torch.int32, device=device)
    d_fc = torch.empty((n + 8,), dtype=torch.int32, device=device)
    d_res = torch.empty((n, engine.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=device)
    cap = n * (2 * L + 256)
    d_sam = torch.empty((cap,), dtype=torch.uint8, device=device)
    h_sam = torch.empty((cap,), dtype=torch.uint8).pin_memory()

    def pipeline(copy_back=True):
        with torch.cuda.stream(st):
            d_text[:text.size].copy_(h_text, non_blocking=True)
        nr, used = fq.parse_device(d_text.data_ptr(), int(text.size), 2, d_b.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_ido.data_ptr(),
                                   d_idl.data_ptr(), d_fc.data_ptr(), st.cuda_stream)
        al.align_device(nr, d_b.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_res.data_ptr(), 0, st.cuda_stream)
        nbytes = fmt.format_device(nr, L, d_b.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_text.data_ptr(), d_ido.data_ptr(), d_idl.data_ptr(),
                                   d_res.data_ptr(), d_sam.data_ptr(), cap, stream=st.cuda_stream)
        if copy_back:
            with torch.cuda.stream(st):
                h_sam[:nbytes].copy_(d_sam[:nbytes], non_blocking=True)
            st.synchronize()
        return nr, nbytes

    try:
        nr, nbytes = pipeline()                                   # warm-up: sizes the formatter's scratch
        torch.cuda.synchronize()
        ok = bool(nr == n and int((h_sam[:nbytes] == 10).sum().item()) == n)
        # (1) the formatter alone, device-resident
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        e0.record(st)
        for _ in range(reps):
            fmt.format_device(n, L, d_b.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_text.data_ptr(), d_ido.data_ptr(), d_idl.data_ptr(),
                              d_res.data_ptr(), d_sam.data_ptr(), cap, stream=st.cuda_stream)
        e1.record(st)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        # (1b) row N4: the coordinate sort of that batch's records on the device (keys, stable radix sort, scan, move)
        d_sorted = torch.empty((cap,), dtype=torch.uint8, device=device)
        d_keys = torch.empty((n,), dtype=torch.int64, device=device)
        sorted_bytes = fmt.sort_device(d_sam.data_ptr(), d_sorted.data_ptr(), cap, d_keys.data_ptr(), 0, st.cuda_stream)
        e0.record(st)
        for _ in range(reps):
            fmt.sort_device(d_sam.data_ptr(), d_sorted.data_ptr(), cap, d_keys.data_ptr(), 0, st.cuda_stream)
        e1.record(st)
        torch.cuda.synchronize()
        sort_ms = e0.elapsed_time(e1) / reps
        k = d_keys.cpu().numpy().view(np.uint64)
        sort_ok = bool(sorted_bytes == nbytes and (k[1:] >= k[:-1]).all() and int((d_sorted[:sorted_bytes] == 10).sum().item()) == n)
        del d_keys
        # (1c) row N4 after the sort, on BAM records: format as BAM, sort, mark duplicates, wrap into BGZF members, build the .bai
        bam = {}
        try:
            fmt.set_format(bam=True)
            nb = fmt.format_device(n, L, d_b.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_text.data_ptr(), d_ido.data_ptr(), d_idl.data_ptr(),
                                   d_res.data_ptr(), d_sam.data_ptr(), cap, stream=st.cuda_stream)
            d_roffs = torch.empty((n,), dtype=torch.int64, device=device)
            sb = fmt.sort_device(d_sam.data_ptr(), d_sorted.data_ptr(), cap, 0, d_roffs.data_ptr(), st.cuda_stream)
            fmt.markdup_device(d_sorted.data_ptr(), d_roffs.data_ptr(), n, st.cuda_stream)         # warm-up: sizes the work buffer
            t0 = time.perf_counter()
            marked = fmt.markdup_device(d_sorted.data_ptr(), d_roffs.data_ptr(), n, st.cuda_stream)
            torch.cuda.synchronize()
            dup_ms = (time.perf_counter() - t0) * 1e3
            n_members = (sb + 0xff00 - 1) // 0xff00
            d_bgzf = torch.empty((sb + 31 * n_members,), dtype=torch.uint8, device=device)
            torch.cuda.synchronize()
            e0.record(st)
            out_bytes = engine.bgzf_device(d_sorted.data_ptr(), sb, d_bgzf.data_ptr(), d_bgzf.numel(), st.cuda_stream)
            e1.record(st)
            torch.cuda.synchronize()
            bgzf_ms = e0.elapsed_time(e1)
            fmt.index_device(d_sorted.data_ptr(), d_roffs.data_ptr(), n, sb, 0, st.cuda_stream)
            t0 = time.perf_counter()
            bai = fmt.index_device(d_sorted.data_ptr(), d_roffs.data_ptr(), n, sb, 0, st.cuda_stream)
            idx_ms = (time.perf_counter() - t0) * 1e3
            n_ref = int(np.frombuffer(bai[4:8], dtype=np.int32)[0])
            bam = {"what": "the batch as BAM records: snapgpu_sam_sort_device, then snapgpu_bam_markdup_device (BAMDupMarkFilter: runs by pointer jumping, 5 radix sorts of "
                           "the keys, one thread per key), snapgpu_bgzf_device, snapgpu_bam_index_device (BAMIndexSupplier; the file composed on the host)",
                   "records": int(n), "record_bytes": int(sb), "markdup_ms": round(dup_ms, 3), "markdup_records_per_s": round(n / (dup_ms / 1e3), 1),
                   "duplicates_marked": int(marked), "second_pass_marks_nothing": bool(marked == 0 or fmt.markdup_device(d_sorted.data_ptr(), d_roffs.data_ptr(), n, st.cuda_stream) == 0),
                   "bgzf_ms": round(bgzf_ms, 3), "bgzf_gbs": round(sb / (bgzf_ms / 1e3) / 1e9, 1), "bgzf_bytes": int(out_bytes),
                   "index_ms": round(idx_ms, 3), "bai_bytes": len(bai), "bai_references": n_ref,
                   "note": "uniform random reads over 3 Gbp hold next to no duplicates: the timing is of the machinery; parity with the reference's marked stream "
                           "and .bai is in tests/test_gpu_sorted_output.py"}
            # the same stream through the compressor on the device (snapgpu_bgzf_deflate_device: one thread block per member) and the .bai of that file
            try:
                fmt.bgzf_deflate_device(d_sorted.data_ptr(), sb, d_bgzf.data_ptr(), d_bgzf.numel(), st.cuda_stream)      # warm-up: sizes the work buffer
                torch.cuda.synchronize()
                e0.record(st)
                z_bytes, member_offsets = fmt.bgzf_deflate_device(d_sorted.data_ptr(), sb, d_bgzf.data_ptr(), d_bgzf.numel(), st.cuda_stream)
                e1.record(st)
                torch.cuda.synchronize()
                z_ms = e0.elapsed_time(e1)
                import zlib
                k = int(member_offsets.size // 2)
                probe = d_bgzf[int(member_offsets[k]):int(member_offsets[k + 1])].cpu().numpy().tobytes()
                want = d_sorted[k * 0xff00:min(sb, (k + 1) * 0xff00)].cpu().numpy().tobytes()
                zbai = fmt.index_device(d_sorted.data_ptr(), d_roffs.data_ptr(), n, sb, 0, st.cuda_stream, member_offsets=member_offsets)
                bam["deflate"] = {"what": "snapgpu_bgzf_deflate_device: LZ77 + dynamic Huffman per 65280-byte member, one block of 1024 threads each (sg_deflate.h)",
                                  "ms": round(z_ms, 3), "gbs_in": round(sb / (z_ms / 1e3) / 1e9, 2), "bytes": int(z_bytes), "ratio": round(z_bytes / max(1, sb), 4),
                                  "zlib6_ratio_of_one_member": round(len(zlib.compress(want, 6)) / max(1, len(want)), 4),
                                  "member_inflates_to_its_payload": bool(zlib.decompress(probe, 31) == want), "bai_bytes": len(zbai)}
            except Exception as e:      # pragma: no cover
                bam["deflate"] = {"error": str(e)[:200]}
            del d_bgzf, d_roffs
        except Exception as e:      # pragma: no cover
            bam = {"error": str(e)[:200]}
        finally:
            fmt.set_format(bam=False)
            fmt.format_device(n, L, d_b.data_ptr(), d_q.data_ptr(), d_off.data_ptr(), d_len.data_ptr(), d_text.data_ptr(), d_ido.data_ptr(), d_idl.data_ptr(),
                              d_res.data_ptr(), d_sam.data_ptr(), cap, stream=st.cuda_stream)
        del d_sorted
        # (3) FASTQ text on the host -> SAM text on the host
        t0 = time.perf_counter()
        for _ in range(reps):
            pipeline()
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / reps
        # (2) host-buffer ABI
        res_host = np.ascontiguousarray(d_res.cpu().numpy().view(engine.RESULT_DTYPE).reshape(-1))
        ids = [b"r%08d" % i for i in range(n)]
        id_buf, id_offs, id_lens = fmt.pack_ids(ids)
        sb = synth.ReadBatch(np.ascontiguousarray(host_batch.bases), np.ascontiguousarray(host_batch.quals), np.ascontiguousarray(host_batch.offsets), np.ascontiguousarray(host_batch.lens))
        buf, used = fmt.format_arrays(sb, id_buf, id_offs, id_lens, res_host, False)
        t0 = time.perf_counter()
        buf, used = fmt.format_arrays(sb, id_buf, id_offs, id_lens, res_host, False, text=buf)
        host_s = time.perf_counter() - t0
        same = bool(used == nbytes and np.array_equal(buf[:used], h_sam[:nbytes].numpy()))
    finally:
        fmt.close(); fq.close(); al.close()
    alg = nbytes + n * (2 * L + engine.RESULT_DTYPE.itemsize + 10)          # the text written + the reads, ids and records read
    return {"kernel": "sg_sam_kernel (one octet of threads per read: the 8 SSE lanes of the CIGAR DP) + scan + sg_sam_pack_kernel", "reads": int(n),
            "ms": round(ms, 3), "reads_per_s": round(n / (ms / 1e3), 1), "text_bytes": int(nbytes), "text_gbs": round(nbytes / (ms / 1e3) / 1e9, 3),
            "roofline": {"bound": "hbm", "achieved": round(alg / (ms / 1e3) / 1e9, 2), "peak": c.peak, "unit": "GB/s", "frac": round(alg / (ms / 1e3) / 1e9 / c.peak, 5),
                         "note": "algorithmic bytes = SAM text written + reads, ids and result records read; the kernel is latency / issue bound (integer DP per read), not bandwidth bound"},
            "host_buffer_abi_reads_per_s": round(n / host_s, 1), "records_ok": ok, "device_and_host_paths_agree": same,
            "sort": {"what": "snapgpu_sam_sort_device: SortedDataFilter's stable coordinate sort of the batch's records (SURVEY 8f N4), keys + cub radix sort + "
                             "scan + one warp per record", "records": int(n), "ms": round(sort_ms, 3), "records_per_s": round(n / (sort_ms / 1e3), 1),
                     "gbs": round(2 * nbytes / (sort_ms / 1e3) / 1e9, 1), "frac_of_hbm_peak": round(2 * nbytes / (sort_ms / 1e3) / 1e9 / c.peak, 4),
                     "keys_ascending_and_all_records_present": sort_ok},
            "sorted_bam": bam,
            "e2e_with_output": {"value": round(n / e2e_s, 1), "unit": "reads/s", "scope": "FASTQ text in pinned host memory -> H2D -> snapgpu_fastq_parse_device -> snapgpu_align_single_device -> "
                                "snapgpu_sam_format_single_device -> D2H of the SAM text; batches one after the other (no overlap between batches)",
                                "h2d_bytes_per_step": int(text.size), "d2h_bytes_per_step": int(nbytes), "ms_per_batch": round(e2e_s * 1e3, 2)},
            "cpu_reference_note": "SAMFormat::computeCigarString on one host thread: 0.107-0.112 M reads/s (round 1, test genome)"}


def sam_cpu_reference(idx, sample, res, paired, n_cpu=20000):
    """reads/s of the reference's SAMFormat::computeCigarString (both overloads; the dominant cost of its writer) on one host thread."""
    from oracle import reflib
    from snap_b200 import synth
    if not reflib.available():
        return None
    d = export_index_for_reference(idx)
    try:
        ridx = reflib.RefIndex(d)
        m = min(n_cpu, sample.n)
        data = []; qual = []; jl = []; ja = []; off = 0
        for i in range(m):
            if paired:
                r = res[i // 2]; w = i % 2
                status, loc, direction, used_ag, score, cb, ca = (int(r["status"][w]), int(r["location"][w]), int(r["direction"][w]), int(r["usedAffineGapScoring"][w]),
                                                                   int(r["score"][w]), int(r["basesClippedBefore"][w]), int(r["basesClippedAfter"][w]))
            else:
                r = res[i]
                status, loc, direction, used_ag, score, cb, ca = (int(r["status"]), int(r["location"]), int(r["direction"]), int(r["usedAffineGapScoring"]), int(r["score"]),
                                                                   int(r["basesClippedBefore"]), int(r["basesClippedAfter"]))
            if status == 0:
                continue
            b, q = sample.read(i)
            x = np.frombuffer(b, dtype=np.uint8); y = np.frombuffer(q, dtype=np.uint8)
            if direction == 1:
                x = synth.revcomp(x); y = y[::-1]
            data.append(x); data.append(np.zeros(16, dtype=np.uint8)); qual.append(y); qual.append(np.zeros(16, dtype=np.uint8))
            if used_ag or score > 0:
                ja.append((off + cb, loc, len(b) - cb - ca, cb, 0, ca, 0, 0, direction, 1, score, 0))
            else:
                jl.append((off, loc, len(b), 0, 0, 0, 0, 0, direction, 1))
            off += len(b) + 16
        data = np.concatenate(data); qual = np.concatenate(qual)
        jl = np.array(jl, dtype=reflib.CIGAR_JOB_DTYPE); ja = np.array(ja, dtype=reflib.CIGAR_AG_JOB_DTYPE)
        t0 = time.perf_counter()
        if jl.size:
            reflib.cigar_lv_batch(ridx, data, jl)
        if ja.size:
            reflib.cigar_ag_batch(ridx, data, qual, ja)
        dt = time.perf_counter() - t0
        return round((jl.size + ja.size) / dt, 1)
    finally:
        shutil.rmtree(d, ignore_errors=True)



def export_index_for_reference(idx):
    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    d = tempfile.mkdtemp(prefix="snapidx_", dir=base)
    idx.save(d)
    return d


def count_differing(want, got, paired):
    """(differing, skipped): result records of the engine vs the reference's for the same reads, bytewise (doubles bit for bit),
    vectorised.  Same exclusions as tests/conftest.py: single-end records BOTH sides report NotFound are skipped (the reference leaves
    the rest uninitialised on its early returns) and counted; mapq / scorePriorToClipping of a paired end reported NotFound are zeroed
    on both sides (copied from an unwritten stack object by ChimericPairedEndAligner), nothing is skipped."""
    w, g = want.copy(), np.asarray(got).view(want.dtype).copy()
    if paired:
        for arr in (w, g):
            nf = arr["status"] == 0
            arr["mapq"][nf] = 0
            arr["scorePriorToClipping"][nf] = 0
        skip = np.zeros(len(w), dtype=bool)
    else:
        skip = (w["status"] == 0) & (g["status"] == 0)
    wb = w.view(np.uint8).reshape(len(w), -1)
    gb = g.view(np.uint8).reshape(len(g), -1)
    return int(((wb != gb).any(axis=1) & ~skip).sum()), int(skip.sum())


def fastq_text(host_batch, prefix=b"r"):
    """FASTQ text of a batch of fixed-length reads, vectorised (ids r00000000 ...)."""
    n = host_batch.n
    L = READ_LEN
    rec = 2 + 8 + 1 + L + 3 + L + 1
    txt = np.empty((n, rec), dtype=np.uint8)
    txt[:, 0] = ord("@"); txt[:, 1] = prefix[0]
    ids = np.arange(n, dtype=np.int64)
    for d in range(8):
        txt[:, 2 + 7 - d] = (ids // 10 ** d % 10 + 48).astype(np.uint8)
    txt[:, 10] = 10
    txt[:, 11:11 + L] = host_batch.bases.reshape(n, L)
    txt[:, 11 + L] = 10; txt[:, 12 + L] = ord("+"); txt[:, 13 + L] = 10
    txt[:, 14 + L:14 + 2 * L] = host_batch.quals.reshape(n, L)
    txt[:, 14 + 2 * L] = 10
    return txt.reshape(-1)


def cli_crosscheck(ref, host_batches, max_dist, threads):
    """Stock `oracle/_ref/snap-aligner single <index> reads.fq -t N -d D` (no -o) over the same reads as a FASTQ file in tmpfs:
    the reference's own "Reads/s" (AlignerContext::printStats, AlignerContext.cpp:491-540; excludes the index load, :420)."""
    import re
    from oracle import reflib
    fq = os.path.join(ref.dir, "reads.fq")
    with open(fq, "wb") as f:
        for hb in host_batches:
            f.write(fastq_text(hb).tobytes())
    n = sum(hb.n for hb in host_batches)
    cmd = [reflib.SNAP_ALIGNER, "single", ref.dir, fq, "-t", str(threads), "-d", str(max_dist)]
    t0 = time.time()
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    wall = time.time() - t0
    os.unlink(fq)
    if r.returncode != 0:
        return {"error": "snap-aligner exited %d: %s" % (r.returncode, (r.stdout + r.stderr)[-300:])}
    lines = [l for l in r.stdout.split("\n") if l.strip()]
    k = [i for i, l in enumerate(lines) if "Reads/s" in l]
    if not k or k[-1] + 1 >= len(lines):
        return {"error": "no stats line in snap-aligner's output", "tail": r.stdout[-300:]}
    toks = [t for t in re.sub(r"\([^)]*\)", " ", lines[k[-1] + 1]).split() if re.fullmatch(r"[0-9,]+", t)]
    return {"command": " ".join(["snap-aligner"] + cmd[1:]).replace(ref.dir, "<index>"), "reads": n, "reads_per_s": int(toks[-2].replace(",", "")),
            "time_in_aligner_s": int(toks[-1].replace(",", "")), "total_reads_reported": int(toks[0].replace(",", "")), "wall_s_incl_index_load": round(wall, 1),
            "note": "includes FASTQ reading by the reference's own supplier threads; harness rate above is aligner only"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl reference: the workload's index is generated on the GPU; no CUDA device")
    W, K = args.warmup, args.steps
    n = args.cpu_sample_reads
    saved = args.batch_reads
    args.batch_reads = n
    os.environ.pop("WORLD_SIZE", None); os.environ["RANK"] = "0"; os.environ["LOCAL_RANK"] = "0"      # rank 0 alone: no process group
    c = build_context(args)
    name = args.workload
    wl = WORKLOADS[name]
    paired = wl["kind"] == "paired"
    dev_batches = make_batches(c, args, wl["kind"], W + K)
    hb = [to_host_batch(b, pinned=False) for b in dev_batches]
    del dev_batches
    args.batch_reads = saved
    ref = RefContext(c.idx)
    c.idx.close()
    del c.bases
    torch.cuda.empty_cache()
    try:
        cores = ref.pick_threads(name, hb[0])
        for b in range(W):
            ref.run(name, hb[b], cores)
        total_s = 0.0
        aligned = 0
        for k in range(K):
            res, ctr, secs = ref.run(name, hb[W + k], cores)
            total_s += secs
            aligned += int((res["status"] != 0).sum())
        value = n * K / total_s
        extra = {}
        if "v3" in ref.ridx:
            ref.run(name, hb[0], cores, build="v3")
            s3 = sum(ref.run(name, hb[W + k], cores, build="v3")[2] for k in range(min(K, 5)))
            extra["value_march_x86_64_v3"] = round(n * min(K, 5) / s3, 1)
        m = min(n, 20000)
        extra["value_1thread"] = round(m / ref.run(name, hb[0].slice(0, m), 1)[2], 1)
        if not paired and not args.no_cli_crosscheck:
            try:
                extra["cli_crosscheck"] = cli_crosscheck(ref, hb[W:W + min(K, 4)], wl["max_dist"], cores)
                if cores != ref.cores:
                    extra["cli_crosscheck_all_hw_threads"] = cli_crosscheck(ref, hb[W:W + min(K, 4)], wl["max_dist"], ref.cores)
            except Exception as e:
                extra["cli_crosscheck"] = {"error": str(e)[:200]}
        sample = ("%d %s per step (bounded sample of the %d-read step), %d threads (the fastest -t of a sweep) started before the clock, stock build (-O3 -msse)"
                  % (n // 2 if paired else n, "pairs" if paired else "reads", saved, cores))
        out = {"impl": "reference", "metric": "aligned reads/s", "value": round(value, 1), "unit": "reads/s", "n_gpus": args.gpus, "steps": K,
               "warmup": W, "ms_per_step": round(total_s / K * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "u8/int32 (+f64 match probabilities)", "data": "synthetic",
               "config": {"workload": ("snap paired (stock options), 2 x %d x %d bp synthetic FR pairs per step vs %d Mbp synthetic reference (24 contigs), seed %d, maxDist %d"
                                       % (n // 2, READ_LEN, args.genome_mbp, SEED_LEN, PAIRED_MAX_DIST)) if paired else
                                      ("snap single, %d x %d bp synthetic reads per step vs %d Mbp synthetic reference (24 contigs), seed %d, maxDist %d"
                                       % (n, READ_LEN, args.genome_mbp, SEED_LEN, wl["max_dist"])), "read_len": READ_LEN, "genome_mbp": args.genome_mbp,
                          "seed_len": SEED_LEN, "max_dist": wl["max_dist"]},
               "cpu_baseline": dict({"value": round(value, 1), "unit": "reads/s", "cores": cores, "kind": "reference", "sample": sample, "host": ref.host()}, **extra),
               "e2e": {"value": round(value, 1), "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "aligned_frac": round(aligned / (n * K), 5),
               "note": "unmodified amplab/snap aligner (BaseAligner::AlignRead / ChimericPairedEndAligner::align) via oracle/_ref on host cores; index = GPU-built, exported to SNAP's format"}
        emit(json.dumps(out))
    finally:
        ref.close()


def stress_phase(args, c_main, failures):
    import torch
    c = build_context(args, repeat_frac=0.05, like=c_main)
    W, K = 2, 3
    batches = make_batches(c, args, "single", W + K)
    res = run_workload(c, args, "single", batches, W, K)
    res.pop("_clocks")
    out = {"reference_genome": "%d Mbp, 5 %% of the bases overwritten with copies of 32 repeat units of 10 kbp at 0-5 %% divergence (a tenth of them tandem arrays of a 2-50 bp motif)" % args.genome_mbp,
           "index_overflow_words": c.setup["overflow_words"], "index_build_s": c.setup["index_build_s"]}
    for k in ("workload", "value", "unit", "steps", "warmup", "ms_per_step", "e2e", "gpu_launches", "per_read"):
        out[k] = res[k]
    if not args.no_cpu_baseline:
        ref = RefContext(c.idx)
        try:
            ref.threads, ref.pinned = getattr(c_main, "ref_threads", (ref.cores, False))
            ref.reflib.set_thread_pinning(ref.pinned, builds=tuple(ref.ridx))
            saved = args.cpu_sample_reads
            args.cpu_sample_reads = min(saved, 250000)
            out["cpu_baseline"] = cpu_leg(ref, args, "single", res["_host0"], res["_records"], min_seconds=1.0)
            args.cpu_sample_reads = saved
            par = out["cpu_baseline"].get("parity_vs_reference")
            if not par or par["differing"] != 0:
                failures.append("parity: stress genome: %s" % par)
        finally:
            ref.close()
    c.idx.close()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    c = build_context(args)
    rank, world = c.rank, c.world
    W, K = args.warmup, args.steps
    headline = args.workload
    failures = []

    # ---- the headline workload: exactly K timed steps after W warm-ups ----
    kind = WORKLOADS[headline]["kind"]
    t0 = time.time()
    batches = {kind: make_batches(c, args, kind, W + K)}
    torch.cuda.synchronize()
    c.setup["reads_s"] = round(time.time() - t0, 2)
    head = run_workload(c, args, headline, batches[kind], W, K, sample_clocks=True, dump_dir=args.dump_outputs)
    clocks = head.pop("_clocks")

    # ---- the other BASELINE configs, each to the same bar (device-resident + e2e + roofline; parity below): configs[2] / [4] paired,
    #      configs[3] -G -d 20 and -ne -d 20.  Bounded step counts of their own so the default run stays within minutes. ----
    phases = {}
    if not args.only_headline:
        Wp, Kp = 3, max(3, min(K, 5))
        for name in ("paired", "ag_d20", "ne_d20", "single"):
            if name == headline:
                continue
            k2 = WORKLOADS[name]["kind"]
            if k2 not in batches:
                batches[k2] = make_batches(c, args, k2, Wp + Kp)
            elif len(batches[k2]) < Wp + Kp:
                batches[k2] += make_batches(c, args, k2, Wp + Kp)[len(batches[k2]):]
            phases[name] = run_workload(c, args, name, batches[k2], Wp, Kp)
            phases[name].pop("_clocks")
    batch0 = {k: v[0] for k, v in batches.items()}
    del batches
    torch.cuda.empty_cache()

    paired = kind == "paired"
    B = args.batch_reads
    out = {
        "metric": "aligned reads/s", "value": head["value"], "unit": "reads/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/int32 (+f64 match probabilities)", "data": "synthetic",
        "config": {"workload": ("snap paired (stock options), 2 x %d x %d bp synthetic FR pairs (insert N(400,40)) per step per GPU vs %d Mbp "
                                "synthetic reference (24 contigs), seed %d, maxDist %d, IntersectingPairedEndAligner + chimeric single-end fallback "
                                "(BASELINE configs[2] shape)" % (B // 2, READ_LEN, args.genome_mbp, SEED_LEN, PAIRED_MAX_DIST)) if paired else
                               ("snap single, %d x %d bp synthetic reads per step per GPU vs %d Mbp synthetic reference (24 contigs), "
                                "seed %d, maxDist %d, affine gap on (BASELINE configs[1] shape)" % (B, READ_LEN, args.genome_mbp, SEED_LEN, WORKLOADS[headline]["max_dist"])),
                   "reads_per_step": B * world, "read_len": READ_LEN, "genome_mbp": args.genome_mbp, "seed_len": SEED_LEN,
                   "max_dist": WORKLOADS[headline]["max_dist"], "repeat_frac": args.repeat_frac,
                   "parallelism": "read-sharded x%d, index replicated per GPU" % world,
                   "l2": "each step uses fresh reads (%.0f MB/step > L2) against a %.1f GB index" % (B * 2 * READ_LEN / 1e6, c.setup["index_hbm_gb"])},
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": clocks, "roofline": head["roofline"], "per_read": head["per_read"],
        "setup": c.setup, "csrc_sha16": csrc_sha16(),
    }
    for name, ph in phases.items():
        key = {"paired": "paired_phase", "single": "single_phase"}.get(name)
        if key:
            out[key] = ph
        else:
            out.setdefault("ag_forced_phase", {})[name] = ph

    # ---- seed-lookup phase and FASTQ ingest in isolation (rank 0) ----
    if rank == 0 and not args.no_seed_phase:
        single_batch = batch0.get("single")
        if single_batch is not None:
            try:
                out["seed_phase"] = seed_phase(args, c.idx, [single_batch], c.device, c.peak, c.peak_src)
            except Exception as e:
                out["seed_phase"] = {"error": str(e)[:300]}
                failures.append("seed_phase: " + str(e)[:200])
            try:
                out["ingest_phase"] = ingest_phase(args, to_host_batch(single_batch, pinned=False), c.device, c.peak, c.peak_src)
            except Exception as e:
                out["ingest_phase"] = {"error": str(e)[:300]}
                failures.append("ingest_phase: " + str(e)[:200])

    # ---- CPU reference: rate on the host cores AND full-size parity of every workload above (rank 0, N=1 only).  A mismatch or an
    #      exception here fails the run (exit code 3 after the line is printed). ----
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = None
        try:
            ref = RefContext(c.idx)
            out["cpu_baseline"] = cpu_leg(ref, args, headline, head["_host0"], head["_records"], min_seconds=5.0, builds=("stock", "v3"), one_thread=True)
            out["cpu_baseline"]["host"] = ref.host()
            c.ref_threads = (ref.threads, ref.pinned)
            for name, ph in phases.items():
                ph["cpu_baseline"] = cpu_leg(ref, args, name, ph["_host0"], ph["_records"], min_seconds=2.0)
            for name, leg in [(headline, out["cpu_baseline"])] + [(n2, p2["cpu_baseline"]) for n2, p2 in phases.items()]:
                par = leg.get("parity_vs_reference")
                if not par or par["differing"] != 0:
                    failures.append("parity: workload %s: %s" % (name, par))
            if "paired" in phases:
                phases["paired"]["per_read"]["aligned_as_pair_frac"] = phases["paired"]["cpu_baseline"].pop("aligned_as_pair_frac", None)
        except Exception as e:
            import traceback
            traceback.print_exc()
            out.setdefault("cpu_baseline", {})["error"] = str(e)[:300]
            failures.append("cpu_baseline: " + str(e)[:200])
        finally:
            if ref is not None:
                ref.close()
    # ---- output stage in isolation (rank 0, N=1; SURVEY 8f N1): the headline's first batch and the engine's own records for it ----
    if rank == 0 and world == 1 and not args.no_seed_phase and not args.no_sam_phase and head.get("_records") is not None:
        try:
            out["sam_phase"] = sam_phase(args, c, head["_host0"], paired)
            if not out["sam_phase"].get("records_ok", True) or not out["sam_phase"].get("device_and_host_paths_agree", True):
                failures.append("sam_phase: records malformed or the device-resident and host-buffer paths disagree")
            if not out["sam_phase"].get("sort", {}).get("keys_ascending_and_all_records_present", True):
                failures.append("sam_phase.sort: sorted records not in key order or not all there")
            if "error" in out["sam_phase"].get("sorted_bam", {}):
                failures.append("sam_phase.sorted_bam: " + out["sam_phase"]["sorted_bam"]["error"])
        except Exception as e:
            import traceback
            traceback.print_exc()
            out["sam_phase"] = {"error": str(e)[:300]}
            failures.append("sam_phase: " + str(e)[:200])

    for ph in [head] + list(phases.values()):
        for k in ("_records", "_host0", "_host_batches"):
            ph.pop(k, None)

    # ---- SURVEY 8d's stress variant (rank 0, N=1): the same shape on a repeat-bearing reference (5 % of the bases from a 10 kbp repeat
    #      library at 0-5 % divergence + tandem arrays), where overflow lists, maxHits skips and the merge logic actually run ----
    if rank == 0 and world == 1 and not args.no_stress_phase and not args.only_headline and args.repeat_frac == 0:
        try:
            c.idx.close(); c.idx = None
            del c.bases
            torch.cuda.empty_cache()
            out["stress_phase"] = stress_phase(args, c, failures)
        except Exception as e:
            import traceback
            traceback.print_exc()
            out["stress_phase"] = {"error": str(e)[:300]}
            failures.append("stress_phase: " + str(e)[:200])
    if failures:
        out["failures"] = failures
    if rank == 0:
        emit(json.dumps(out))
    try:
        if c.idx is not None:
            c.idx.close()
    except Exception:  # pragma: no cover
        pass
    if world > 1:
        dist.destroy_process_group()
    if failures:
        sys.stderr.write("bench.py: FAILED: %s\n" % "; ".join(failures))
        sys.exit(3)


_REAL_STDOUT = None


def emit(line: str) -> None:
    """The one JSON line goes to the process's real stdout; everything else any library prints (NCCL's version banner, for one,
    goes to fd 1 at communicator creation whatever NCCL_DEBUG says short of unset) has been routed to stderr by main()."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)                      # C-level stdout of this process (and its children) -> stderr
    sys.stdout = sys.stderr
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs writes the engine's records; it does not apply to --impl reference")
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
