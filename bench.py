#!/usr/bin/env python
"""bench.py -- the coverage hot path on synthetic reads of BASELINE.json's shapes.

  python bench.py --gpus N --steps K --warmup W            (one rank per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py ... --dump-outputs DIR                    (also write the last timed step's outputs, see dump_outputs)

A "step" = one pass of the hot path over one batch: mapped reads (SoA) -> per-base depth of every
contig -> per-contig statistics (the work of reference metacov/pileup.py:9-26 driven by the loop at
metacov/cli.py:85-95).  Workload at N=1: config C2 of BASELINE.json (10 M x 150 bp reads over 1 000
contigs of 50 kb); for N>1 every rank gets its own C2-sized contig range (weak scaling, no
data-path collective, one NCCL all-gather of the 64-byte per-contig statistics records).

Prints ONE JSON line (rank 0).  `value` is timed with the SoA already resident in HBM; `e2e` is the
same metric through the public API with HOST buffers (H2D + D2H inside the timed region).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "aligned bases/sec -> per-base coverage + per-contig stats"
UNIT = "aligned_bases/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled during the timed region (NVML)."""

    def __init__(self, index, period=0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def make_workload(name, scale, n_ranks):
    """Global workload = n_ranks copies of the named shape, split into contiguous contig ranges."""
    from metacov_b200 import synth
    w = synth.WORKLOADS[name](scale * n_ranks)
    return w


def workload_label(name, n_ranks, w):
    """config.workload: the same string in both arms (the driver compares it)."""
    return "%s x%d ranks: %s" % (name, n_ranks, w.describe())


def pin_rank_to_cores(local, world):
    """One rank per GPU: give every rank its own slice of the host cores (and thereby of the memory controllers its
    pinned buffers are first touched from) instead of letting all ranks share the default affinity mask -- the GPU's own
    NUMA-local cores when NVML knows them."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        near = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(cpus) // 64) + 1)
            near = [c for c in cpus if (words[c // 64] >> (c % 64)) & 1]
        except Exception:
            near = None
        pool = near if near and len(near) >= world else cpus
        per = max(1, len(pool) // world)
        mine = pool[(local * per) % len(pool):(local * per) % len(pool) + per]
        if mine:
            os.sched_setaffinity(0, mine)
        return {"cores": len(mine), "first": mine[0] if mine else None, "numa_local": bool(near and pool is near)}
    except Exception as e:                       # affinity is an optimisation, never a requirement
        return {"error": str(e)}


def cpu_port_time(batch, lengths, regions, threads, reps=2):
    """The C restatement (oracle/coverage.c), contig-parallel: depth + per-contig statistics."""
    from oracle import cport
    tid, st, en = regions
    best = None
    aligned = 0
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        d, off, info = cport.depth(batch, lengths, mode="par", threads=threads)
        cport.region_stats(d, off, lengths, tid, st, en, threads=threads)
        dt = time.perf_counter() - t0
        aligned = info["aligned_bases"]
        best = dt if best is None else min(best, dt)
    return aligned, best


def python_port_rate(batch, lengths, max_contigs=1):
    """The reference's own structure: one Python object per pileup column and numpy/sorted()
    reductions per region (metacov/pileup.py:13-26), over the restated htslib engine.  Tiny sample."""
    from oracle import bamio, classic as oc
    from oracle.pysam_boundary import FakeAlignmentFile
    sel = np.asarray(batch.tid) < max_contigs
    n = int(sel.sum())
    r = bamio.BamRecords()
    o = np.asarray(batch.cig_off).astype(np.int64)
    r.tid, r.pos = np.asarray(batch.tid)[:n], np.asarray(batch.pos)[:n]
    r.flag, r.mapq = np.asarray(batch.flag)[:n], np.asarray(batch.mapq)[:n]
    r.cig_off, r.cig = o[:n + 1], np.asarray(batch.cig)[:o[n]]
    r.names, r.seqs = [""] * n, [None] * n
    r.reflen = bamio.cigar_reflen(r.cig_off, r.cig)
    names = tuple("c%d" % c for c in range(max_contigs))
    bam = FakeAlignmentFile(bamio.BamHeader("", names, tuple(int(x) for x in lengths[:max_contigs])), r)
    t0 = time.perf_counter()
    total = 0
    for c in range(max_contigs):
        total += oc.classic(bam, names[c], 0, int(lengths[c]))["sum"]
    return total / (time.perf_counter() - t0), n


def run_reference(args):
    """--impl reference: the CPU implementation of the path on the host cores (the reference itself needs
    pysam/htslib, absent from this image, so this is the C port of oracle/, kind 'port').  Same workload as the GPU
    arm at the same N (N x the named shape); built with the oracle-side generator, so this process never loads the
    product library.  A step = the whole workload; --warmup untimed steps, then exactly --steps timed ones."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cport, synthgen
    cport.build()
    w = synthgen.WORKLOADS[args.workload](args.scale * args.gpus)
    cores = os.cpu_count() or 1
    batch, _ = synthgen.generate(w, threads=cores)
    tid = np.arange(w.n_contigs, dtype=np.int32)
    regions = (tid, np.zeros_like(tid), w.contig_len)
    times = []
    aligned = 0
    for k in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        d, off, info = cport.depth(batch, w.contig_len, mode="par", threads=cores)
        st = cport.region_stats(d, off, w.contig_len, *regions, threads=cores)
        dt = time.perf_counter() - t0
        aligned = info["aligned_bases"]
        if k >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, st, w.contig_len, lambda c: d[off[c]:off[c] + w.contig_len[c]])
    ms = 1e3 * float(np.mean(times))
    value = aligned / (ms / 1e3)
    py_rate, py_n = python_port_rate(batch, w.contig_len, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": workload_label(args.workload, args.gpus, w), "scale": args.scale},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "the whole %s workload per step (C port oracle/coverage.c, contig-parallel pthreads), %d timed "
                                   "steps" % (args.workload, args.steps),
                         "python_port_value": py_rate,
                         "python_port_sample": "first contig (%d reads) through the reference-structured Python loop, 1 core" % py_n},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(args.real_stdout, line)


DUMP_STATS_FIELDS = ("sum", "sumsq", "iq_sum", "n_ge1", "n_geN", "min", "max", "med_lo", "med_hi", "flags")
DUMP_MAX_REGIONS = 100_000           # 10 float64 fields: at most 8 MB of statistics
DUMP_MAX_DEPTH = 12 * 2 ** 20        # float32 depth values: at most 48 MB


def dump_outputs(out_dir, records, lengths, depth_of, tid_base=0):
    """--dump-outputs: what the timed path handed its caller in the last step, as DIR/<name>.npy.
    `records` are the statistics records, `depth_of(c)` the depth of local contig c (length lengths[c]).

    stats_<field>.npy   per-region statistics records (float64), one entry per region in region order; above
                        DUMP_MAX_REGIONS regions a seeded sample, whose region indices are in stats_index.npy
    depth.npy           per-base depth (float32) of a seeded sample of whole contigs, concatenated
    depth_contigs.npy   the global contig ids of that sample, in the order their depth is concatenated (float64)
    With the same arguments the workload is the same, so two builds give files that compare entry by entry.
    With --gpus N > 1 rank 0 writes the file: the records are the gathered ones of all regions, the depth sample is
    drawn from rank 0's own contig range only (the reference arm draws from all contigs), so depth samples of the two
    arms at N > 1 are matched through depth_contigs.npy."""
    os.makedirs(out_dir, exist_ok=True)
    g = len(records)
    idx = np.arange(g) if g <= DUMP_MAX_REGIONS else np.sort(np.random.default_rng(0).choice(g, DUMP_MAX_REGIONS, replace=False))
    if g > DUMP_MAX_REGIONS:
        np.save(os.path.join(out_dir, "stats_index.npy"), idx.astype(np.float64))
    for f in DUMP_STATS_FIELDS:
        np.save(os.path.join(out_dir, "stats_%s.npy" % f), records[f][idx].astype(np.float64))
    contigs, room = [], DUMP_MAX_DEPTH
    for c in np.random.default_rng(1).permutation(len(lengths)):
        if lengths[c] <= room:
            contigs.append(int(c))
            room -= int(lengths[c])
    depth = [depth_of(c) for c in contigs]
    np.save(os.path.join(out_dir, "depth.npy"), np.concatenate(depth).astype(np.float32) if depth else np.zeros(0, np.float32))
    np.save(os.path.join(out_dir, "depth_contigs.npy"), np.asarray(contigs, dtype=np.float64) + tid_base)


def batch_bytes(b):
    tot = 0
    for a in b:
        tot += a.numel() * a.element_size() if hasattr(a, "numel") else a.nbytes
    return int(tot)


def strong_scaling_c4(args, sharding, synth, dist, torch, world, rank, local, dev, barrier):
    """BASELINE config 4 (1 B x 150 bp reads, 100 k contigs), the SAME total work at every N: contiguous contig ranges
    balanced on cost, each rank generates and processes its range, one all-gather of the 64-byte records per pass.
    Reported beside the weak-scaling `value` so that N = 1 keeps agreeing with the single-GPU bench line."""
    from metacov_b200 import CoverageEngine
    torch.cuda.empty_cache()
    w = synth.WORKLOADS["c4"](args.strong_scale)
    rpc = np.diff(w.read_start)
    bounds = sharding.partition_contigs(w.contig_len, rpc, world)
    c0, c1 = int(bounds[rank]), int(bounds[rank + 1])
    r0, r1 = sharding.shard_read_range(w.read_start, bounds, rank)
    lengths = w.contig_len[c0:c1]
    dbatch, _ = synth.generate_device(w, local, i0=r0, n=r1 - r0, tid_base=c0)
    g = c1 - c0
    reg_tid = np.arange(g, dtype=np.int32)
    reg_start, reg_end = np.zeros(g, dtype=np.int32), lengths.astype(np.int32)
    stream = torch.cuda.current_stream(dev)
    eng = CoverageEngine(lengths, device=local, stream=stream.cuda_stream)
    owner = sharding.assign_regions(np.arange(w.n_contigs), bounds)
    dg = sharding.DeviceGather(owner, world, dev) if world > 1 else None

    def run(k):
        prev = None
        for i in range(k):
            eng.depth_sorted(dbatch, wait=False)
            if world > 1:
                eng.region_stats_enqueue(reg_tid, reg_start, reg_end, dg.local[i & 1])
                dg.submit(i & 1, want_host=(rank == 0))
                if prev is not None:
                    dg.collect(prev, want_host=(rank == 0))
                prev = i & 1
            else:
                t = eng.region_stats_submit(reg_tid, reg_start, reg_end, slot=i & 1)
                if prev is not None:
                    eng.region_stats_collect(prev, copy=False)
                prev = t
        return dg.collect(prev, want_host=(rank == 0)) if world > 1 else eng.region_stats_collect(prev, copy=False)

    run(3)
    info = eng.pass_info()
    al = torch.tensor([info["aligned_bases"]], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(al)
    steps = args.steps
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = run(steps)
    e1.record()
    barrier()
    mine = e0.elapsed_time(e1) / steps
    t_all = torch.zeros(world, dtype=torch.float64, device=dev)
    t_all[rank] = mine
    if world > 1:
        dist.all_reduce(t_all)
    per_rank = [float(x) for x in t_all.tolist()]
    ms = max(per_rank)
    # gather cost alone (the one collective of the path)
    gather_ms = None
    if world > 1:
        barrier()
        t0 = time.perf_counter()
        for i in range(10):
            dg.submit(i & 1, want_host=(rank == 0))
            dg.collect(i & 1, want_host=(rank == 0))
        torch.cuda.synchronize()
        gather_ms = 1e3 * (time.perf_counter() - t0) / 10
    if rank == 0 and out is not None and world == 1:
        assert int(np.asarray(out["sum"], dtype=np.int64).sum()) == int(al.item()), "strong-scaling block: mass conservation violated"
    res = {"workload": "c4 (strong): %s, contig-range sharded over %d rank(s)" % (w.describe(), world),
           "ms_per_pass": ms, "value": int(al.item()) / (ms / 1e3), "unit": UNIT, "steps": steps,
           "per_rank_ms": per_rank, "imbalance": (max(per_rank) / (sum(per_rank) / len(per_rank))) if per_rank else None,
           "gather_ms": gather_ms, "reads_total": int(w.n_reads), "reads_per_rank": int(r1 - r0),
           "timing": "CUDA events around the pipelined passes on each rank, max over ranks"}
    eng.close()
    del dbatch
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    from metacov_b200 import CoverageEngine, ReadBatch, sharding, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = pin_rank_to_cores(local, world) if world > 1 else None      # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- workload: contiguous contig range of this rank --------------------------------------
    w = make_workload(args.workload, args.scale, world)
    rpc = np.diff(w.read_start)
    bounds = sharding.partition_contigs(w.contig_len, rpc, world)
    c0, c1 = int(bounds[rank]), int(bounds[rank + 1])
    r0, r1 = sharding.shard_read_range(w.read_start, bounds, rank)
    lengths = w.contig_len[c0:c1]
    dbatch, _ = synth.generate_device(w, local, i0=r0, n=r1 - r0, tid_base=c0)
    n_reads = r1 - r0
    g = c1 - c0
    reg_tid = np.arange(g, dtype=np.int32)
    reg_start = np.zeros(g, dtype=np.int32)
    reg_end = lengths.astype(np.int32)
    owner = sharding.assign_regions(np.arange(w.n_contigs), bounds)

    # One explicit (non-default) torch stream carries everything: the engine's kernels, the NCCL
    # gather (which orders itself against torch's *current* stream) and the timing events.  The
    # legacy default stream has handle 0, which mcov_create would take as "make your own stream".
    work_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(work_stream)
    eng = CoverageEngine(lengths, device=local, stream=work_stream.cuda_stream)
    assert work_stream.cuda_stream != 0

    if world > 1:
        dg = sharding.DeviceGather(owner, world, dev)
        local_dev, out_dev = dg.local_dev, dg.out_dev

    def depth_dev(batch):
        """Per-base depth of the rank's contigs from a device-resident batch."""
        if args.path == "push":                   # any-order formulation: clear + k_expand (red.global) + look-back scan
            eng.begin()
            eng.push(batch)
            eng.finalize()
        else:                                     # default for sorted input: k_fused_prep + k_fused_tile
            eng.depth_sorted(batch, wait=False)   # verdict delivered by the next synchronising call

    def step(batch):
        depth_dev(batch)
        if world == 1:
            return eng.region_stats(reg_tid, reg_start, reg_end)          # one sync per step
        # N>1: records stay on the device, ONE all-gather over NCCL, one D2H of all records
        eng.region_stats_enqueue(reg_tid, reg_start, reg_end, local_dev)
        return dg.gather(want_host=(rank == 0))

    # the first statistics call builds the region plan (chunk / slice tables, sorted tasks: host work + small copies),
    # cached for every later call with the same regions; its cost is reported, not hidden in the warm-up
    torch.cuda.synchronize()
    t_first = time.perf_counter()
    stats = step(dbatch)
    torch.cuda.synchronize()
    first_call_ms = 1e3 * (time.perf_counter() - t_first)
    for _ in range(max(args.warmup, 3)):
        stats = step(dbatch)
    if args.breakdown:
        def tt(fn, n=30):
            barrier(); t0 = time.perf_counter()
            for _ in range(n):
                fn()
            torch.cuda.synchronize(); return (time.perf_counter() - t0) / n * 1e6
        parts = {"depth_only": tt(lambda: depth_dev(dbatch))}
        if world > 1:
            parts["stats_enqueue"] = tt(lambda: eng.region_stats_enqueue(reg_tid, reg_start, reg_end, local_dev))
            parts["all_gather"] = tt(lambda: dist.all_gather_into_tensor(out_dev, local_dev))
            parts["gather+d2h+merge"] = tt(lambda: dg.gather())
        else:
            parts["stats"] = tt(lambda: eng.region_stats(reg_tid, reg_start, reg_end))
        parts["step"] = tt(lambda: step(dbatch))
        print("rank %d breakdown us: %s" % (rank, {k: round(v, 1) for k, v in parts.items()}), file=sys.stderr)
    info = eng.pass_info()
    aligned_local = info["aligned_bases"]
    aligned_t = torch.tensor([aligned_local], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(aligned_t)
    aligned_total = int(aligned_t.item())
    # sanity of what is being timed (size-independent property, any workload size): no synthetic read is
    # clipped at a contig end, so the per-contig `sum` records must add up to the aligned bases
    if rank == 0 or world == 1:
        got_sum = int(np.asarray(stats["sum"], dtype=np.int64).sum())
        assert got_sum == aligned_total, "mass conservation violated: sum(records.sum)=%d, aligned bases=%d" % (got_sum, aligned_total)

    # ---- timed region: device-resident inputs ---------------------------------------------------
    # NVML is a shared, lock-protected service: only rank 0 samples (its GPU runs the same kernels)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    # The K steps are pipelined the way a caller with batch after batch would run them --
    # the statistics of step k are collected from a pinned slot after step k+1 has been enqueued
    # (mcov_region_stats_submit / collect), so the GPU never waits for the host between steps.
    # Every step's records still reach the host inside the timed region.
    def run_steps(k, depth_call):
        if world > 1:
            # same pipelining with the collective in it: records of step k+1, their all-gather and the
            # copy-back are enqueued before step k's are waited for (two DeviceGather slots)
            prev, out = None, None
            for i in range(k):
                depth_call()
                eng.region_stats_enqueue(reg_tid, reg_start, reg_end, dg.local[i & 1])
                dg.submit(i & 1, want_host=(rank == 0))
                if prev is not None:
                    out = dg.collect(prev, want_host=(rank == 0))
                prev = i & 1
            return dg.collect(prev, want_host=(rank == 0))
        prev = None
        for i in range(k):
            depth_call()
            t = eng.region_stats_submit(reg_tid, reg_start, reg_end, slot=i & 1)
            if prev is not None:
                eng.region_stats_collect(prev, copy=False)     # records: a view of the pinned slot
            prev = t
        return eng.region_stats_collect(prev, copy=False)

    piped = run_steps(3, lambda: depth_dev(dbatch))
    if world == 1:
        ref_stats = step(dbatch)
        assert piped.tobytes() == ref_stats.tobytes(), "pipelined statistics differ from the synchronous call"
    barrier()
    l0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    last = run_steps(args.steps, lambda: depth_dev(dbatch))
    ev1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, np.array(last), lengths, eng.copy_depth, c0)
    ms_total = ev0.elapsed_time(ev1)
    t_t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_t, op=dist.ReduceOp.MAX)
    ms_step = float(t_t.item()) / args.steps
    launches = eng.launch_count() - l0
    # the same K steps with one synchronising call per step (no pipelining), for comparison
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        step(dbatch)
    e3.record()
    barrier()
    t_s = torch.tensor([e2.elapsed_time(e3)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_s, op=dist.ReduceOp.MAX)
    ms_sync = float(t_s.item()) / args.steps
    # per-kernel durations: the same K steps once more with a CUDA-event pair around every launch
    # (the events cost ~8 % of a 0.4 ms step, so they stay out of the pass that produces `value`)
    eng.profile(True)
    for _ in range(args.steps):
        step(dbatch)
    kt = eng.profile_read()
    eng.profile(False)

    # ---- e2e: host (pinned) buffers through the public API, H2D + D2H inside the timed region ------
    # The host side hands over what the product's decoder produces for a sorted file: the TRANSPORT BLOCK
    # (mcov_bam_stream_next_block -> mcov_pack_block: one contiguous pinned buffer per batch, one host-to-device
    # copy).  The block is packed here once, outside the timed region, by that same native packer (its time is
    # reported as pack_ms); `plain_soa` is the same step from the plain pinned SoA columns, `from_bam` the whole
    # way from the compressed file.
    e2e = None
    hbatch = None
    # a batch of 2^32 or more CIGAR ops (config C5 at full size: 56 GB of ops) has no host-side leg here: it would have to sit
    # in pinned host memory as plain 64-bit-offset columns
    wide_ops = dbatch.cig_off.dtype == torch.int64 and int(dbatch.cig_off[-1].item()) > 0xFFFFFFFF
    if wide_ops and not args.no_e2e:
        e2e = {"skipped": "the batch holds 2^32 or more CIGAR ops (64-bit offsets): no narrow host transport; device-resident leg only"}
    if not args.no_e2e and not wide_ops:
        from metacov_b200.engine import pack_batch, pack_block, packed_bytes
        hbatch = ReadBatch(*[t.cpu() for t in dbatch])
        t_pack = time.perf_counter()
        try:
            blk = pack_block(hbatch, g, with_mapq=False, pinned=True)
            pack_ms = 1e3 * (time.perf_counter() - t_pack)
            transport = ("transport block of the product decoder (mcov_pack_block v4: contig prefix, one byte per read = position "
                         "difference | (flag, CIGAR class) index as nibbles with u8 side lists, exceptions / escapes, CIGAR dictionary + "
                         "u16 explicit ops, chunk table, no mapq): ONE pinned buffer, ONE H2D copy, ONE unpack kernel")
            depth_packed = lambda wait=False: eng.depth_sorted_block(blk, wait=wait)
            h2d_bytes = int(blk[1])
        except ValueError:
            # long reads (config C5: thousands of ops per CIGAR) do not qualify: compact columns instead
            packed = pack_batch(hbatch, g, with_mapq=False, pinned=True)
            pack_ms = 1e3 * (time.perf_counter() - t_pack)
            transport = "compact columns (contig prefix, u16 op counts, no mapq)"
            depth_packed = lambda wait=False: eng.depth_sorted_packed(packed, wait=wait)
            h2d_bytes = packed_bytes(packed)

        def e2e_step():
            depth_packed(False)
            if world == 1:
                return eng.region_stats(reg_tid, reg_start, reg_end)
            eng.region_stats_enqueue(reg_tid, reg_start, reg_end, local_dev)
            return dg.gather(want_host=(rank == 0))

        def timed(fn, k):
            barrier()
            t0 = time.perf_counter()
            for _ in range(k):
                fn()
            barrier()
            dt = (time.perf_counter() - t0) / k
            d_t = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(d_t, op=dist.ReduceOp.MAX)
            return float(d_t.item())

        for _ in range(2):
            st_e2e = e2e_step()
        if world == 1:
            assert int(np.asarray(st_e2e["sum"], dtype=np.int64).sum()) == aligned_total, "e2e path: mass conservation violated"
        # pipelined like the device-resident run: the copy of batch k+1 overlaps the kernels of batch k
        # The host is inside this loop (it waits for the previous copy, enqueues the next one, collects the records), so
        # one window of K steps = 15 ms catches whatever the host does besides (first run of a process on a fresh box:
        # 0.50 ms/step, the next ones 0.29 - 0.33): five windows of K steps, the best one reported, all of them listed.
        # (the host-only phase in front of this leg -- copying the batch back, packing the block: seconds -- lets the GPU and
        #  the PCIe link fall into their idle states; 0.25 s of untimed steps bring both back before anything is timed)
        t_w = time.perf_counter()
        while time.perf_counter() - t_w < 0.25:
            run_steps(20, lambda: depth_packed(False))
        e2e_windows = [timed(lambda: run_steps(args.e2e_steps, lambda: depth_packed(False)), 1) / args.e2e_steps for _ in range(5)]
        dt = min(e2e_windows)
        dt_sync = timed(e2e_step, args.e2e_steps)
        # for comparison: the plain SoA columns (tid[], u32 offsets, mapq) from pinned memory
        pbatch = ReadBatch(*[t.pin_memory() for t in hbatch])

        def soa_step():
            eng.depth_sorted(pbatch, wait=False)
            if world == 1:
                return eng.region_stats(reg_tid, reg_start, reg_end)
            eng.region_stats_enqueue(reg_tid, reg_start, reg_end, local_dev)
            return dg.gather(want_host=(rank == 0))

        for _ in range(5):
            soa_step()
        dt_soa = timed(soa_step, args.e2e_steps)
        # the block's copy alone (same pinned buffer, same size): what the link allows per step
        h2d_only_ms = None
        try:
            src = blk[0][:h2d_bytes]
            dst = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
            for _ in range(3):
                dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(20):
                dst.copy_(src, non_blocking=True)
            c1.record(); torch.cuda.synchronize()
            h2d_only_ms = c0.elapsed_time(c1) / 20
            del dst
        except Exception:
            pass
        e2e = {"value": aligned_total / dt, "unit": UNIT, "h2d_only_ms": h2d_only_ms,
               "h2d_bytes_per_step": h2d_bytes + g * 16, "d2h_bytes_per_step": g * 64 + 64,
               "ms_per_step": 1e3 * dt, "windows_ms_per_step": [round(1e3 * x, 4) for x in e2e_windows],
               "unpipelined_ms_per_step": 1e3 * dt_sync,
               "bytes_scope": "per rank (every rank copies its own shard; multiply by n_gpus for the whole job)" if world > 1 else "whole job",
               "transport": transport, "pack_ms": pack_ms,
               "plain_soa": {"value": aligned_total / dt_soa, "h2d_bytes_per_step": batch_bytes(pbatch) + g * 16,
                             "ms_per_step": 1e3 * dt_soa}}
        # ---- the whole way from the compressed FILE (rank 0 at N = 1): BGZF inflate + record parsing on the host cores in
        # batches (mcov_bam_stream_*), transport blocks, streamed fused pass (mcov_stream_push_block), statistics.
        if world == 1 and not args.no_bam:
            import tempfile
            n_bam = int(min(n_reads, args.bam_reads))
            wb = synth.WORKLOADS[args.workload](args.scale * n_bam / max(n_reads, 1))
            hb, isz = synth.generate_host(wb)
            if len(hb.tid) and int(np.diff(hb.cig_off.astype(np.int64)).max()) < 65536:
                tmp = tempfile.mkdtemp(prefix="mcov_bench_")
                path = os.path.join(tmp, "bench.bam")
                synth.write_bam(path, wb, hb, isz)
                from metacov_b200 import AlignmentFile
                rt_ = np.arange(wb.n_contigs, dtype=np.int32)
                best, batches, al_b = None, 0, 0
                for _ in range(3):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    with AlignmentFile(path, device=local, batch_reads=args.bam_batch) as af:
                        e2 = af.coverage_engine()
                        sb = e2.region_stats(rt_, np.zeros_like(rt_), wb.contig_len)
                        al_b = e2.pass_info()["aligned_bases"]
                        batches = af.stream_batches
                    dtb = time.perf_counter() - t0
                    best = dtb if best is None else min(best, dtb)
                assert int(np.asarray(sb["sum"], dtype=np.int64).sum()) == al_b
                e2e["from_bam"] = {"value": al_b / best, "unit": UNIT, "reads": int(len(hb.tid)), "bam_bytes": os.path.getsize(path),
                                   "ms_total": 1e3 * best, "batches": int(batches), "batch_reads": int(args.bam_batch),
                                   "host_cores": os.cpu_count(),
                                   "what": "open + BGZF inflate + record parsing on the host cores, batch by batch into pinned buffers, "
                                           "transport blocks, streamed fused pass, per-contig statistics; best of 3 (page cache warm)"}
                # the same file decoded ON THE GPU (mcov_bam_decode_gpu: the compressed image over PCIe, inflate + record
                # parsing on the device); file read and the copy of the image included, like for like with the host leg
                try:
                    bestg = None
                    for _ in range(3):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        with AlignmentFile(path, device=local, decode="gpu") as af:
                            e2 = af.coverage_engine()
                            sg = e2.region_stats(rt_, np.zeros_like(rt_), wb.contig_len)
                            al_g = e2.pass_info()["aligned_bases"]
                        dtg = time.perf_counter() - t0
                        bestg = dtg if bestg is None else min(bestg, dtg)
                    assert sg.tobytes() == sb.tobytes() and al_g == al_b, "GPU-decoded file gives other records than the host-decoded one"
                    e2e["from_bam"]["gpu_decode"] = {"value": al_b / bestg, "ms_total": 1e3 * bestg,
                                                     "what": "file read + image H2D (pageable) + BGZF inflate and record parsing on the "
                                                             "GPU + fused pass + statistics; records identical to the host-decoded leg"}
                except Exception as e:                       # (reported, not fatal: the headline legs stand without it)
                    e2e["from_bam"]["gpu_decode"] = {"error": str(e)[:200]}
                # the same file through the STREAMED GPU decoder (mcov_bam_gpu_stream_depth): chunks of the file into pinned
                # memory by a host thread, each inflated / parsed / pushed into the streamed pass on the device -- what a
                # file larger than the device takes; here the chunk is a quarter of the file
                try:
                    chunk = max(1 << 20, os.path.getsize(path) // 4)
                    bests, chunks = None, 0
                    for _ in range(3):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        with AlignmentFile(path, device=local, decode="gpu-stream", gpu_chunk_bytes=chunk) as af:
                            e2 = af.coverage_engine()
                            ss = e2.region_stats(rt_, np.zeros_like(rt_), wb.contig_len)
                            al_s = e2.pass_info()["aligned_bases"]
                            chunks = af.stream_batches
                        dts = time.perf_counter() - t0
                        bests = dts if bests is None else min(bests, dts)
                    assert ss.tobytes() == sb.tobytes() and al_s == al_b, "streamed GPU decode gives other records than the host-decoded file"
                    e2e["from_bam"]["gpu_stream"] = {"value": al_b / bests, "ms_total": 1e3 * bests, "chunks": int(chunks), "chunk_bytes": int(chunk),
                                                     "what": "file read in chunks into pinned memory (host thread) + per chunk: H2D, BGZF inflate, "
                                                             "record chain and columns on the GPU, streamed fused pass; + statistics"}
                except Exception as e:
                    e2e["from_bam"]["gpu_stream"] = {"error": str(e)[:200]}
                try:
                    os.remove(path); os.remove(path + ".bai"); os.rmdir(tmp)
                except OSError:
                    pass

    # ---- strong scaling on the 1 B-read config C4, contig-range sharded over the N ranks (north_star) -----------------
    strong = None
    if not args.no_strong:
        strong = strong_scaling_c4(args, sharding, synth, dist, torch, world, rank, local, dev, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (CUDA events around every launch, timed region) ------------
    peak, peak_src = peaks()
    flag = dbatch.flag.to(torch.int32) & 0xFFFF
    passing = ((flag & 0x704) == 0) & ~(((flag & 1) != 0) & ((flag & 2) == 0)) & ((flag & 4) == 0)
    if dbatch.cig_off.dtype == torch.int64:                       # 64-bit offsets (a batch of 2^32 or more ops)
        ncig = dbatch.cig_off[1:] - dbatch.cig_off[:-1]
    else:
        ncig = (dbatch.cig_off[1:].to(torch.int64) & 0xFFFFFFFF) - (dbatch.cig_off[:-1].to(torch.int64) & 0xFFFFFFFF)
    cig_pass = int((ncig * passing).sum().item())
    n_pass = int(passing.sum().item())
    slots = eng.n_slots
    L_regions = int(lengths.astype(np.int64).sum())
    alg_bytes = {
        "k_fused_prep": 15 * n_reads + 4 * cig_pass + 4 * n_reads,      # SoA + CIGAR ops in, 4-byte records out
        "k_fused_tile": 4 * n_reads + 4 * slots,                        # records in, depth out
        "k_fused_prep_tma": 15 * n_reads + 4 * cig_pass + 4 * n_reads,  # (the TMA-staged kernels move the same bytes)
        "k_fused_tile_tma": 4 * n_reads + 4 * slots,
        "k_region_stats": 4 * int(lengths[lengths > 8192].astype(np.int64).sum()) + 64 * int((lengths > 8192).sum()),
        "k_stats_stream": 4 * int(lengths[lengths > 8192].astype(np.int64).sum()) + 64 * int((lengths > 8192).sum()),
        "k_region_stats_warp": 4 * int(lengths[lengths <= 8192].astype(np.int64).sum()) + 64 * int((lengths <= 8192).sum()),
        "k_expand": 15 * n_reads + 4 * cig_pass + 8 * n_pass,
        "k_scan_inplace": 8 * slots,
        "memset_depth": 4 * slots,
    }
    kernels = {}
    for name, (n_l, tot) in kt.items():
        per = tot / max(n_l, 1)
        ent = {"launches": int(n_l), "ms_per_launch": per, "share_of_step": per * (n_l / args.steps) / ms_step}
        if name in alg_bytes and per > 0:
            ent["algorithmic_bytes"] = alg_bytes[name]
            ent["gbs"] = alg_bytes[name] / per / 1e6
            ent["frac"] = ent["gbs"] / peak
        kernels[name] = ent
    dom = max((k for k in kernels if "gbs" in kernels[k]), key=lambda k: kernels[k]["ms_per_launch"] * kernels[k]["launches"])
    # measured DRAM traffic of the dominant kernel (dram__bytes_read+write from the committed ncu capture);
    # only quoted for the workload it was captured on
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic_c2.json")
    if args.workload == "c2" and args.scale == 1.0 and os.path.exists(tpath):
        with open(tpath) as fh:
            traffic = json.load(fh)["dram_bytes_per_launch"].get(dom)
    roof = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
            "frac": kernels[dom]["frac"], "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": kernels[dom]["algorithmic_bytes"], "kernels": kernels,
            "timing": "CUDA-event pair around every launch on the launching stream, K steps run right after the timed region"}
    if args.path == "push":
        whole_bytes = alg_bytes["memset_depth"] + alg_bytes["k_expand"] + alg_bytes["k_scan_inplace"] + 4 * L_regions + 64 * g
    else:
        whole_bytes = alg_bytes["k_fused_prep"] + alg_bytes["k_fused_tile"] + 4 * L_regions + 64 * g
    roof["whole_step"] = {"algorithmic_bytes": whole_bytes, "gbs": whole_bytes / ms_step / 1e6,
                          "frac": whole_bytes / ms_step / 1e6 / peak}

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only) --------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        from oracle import cport
        cport.build()
        if hbatch is None:
            hbatch = ReadBatch(*[t.cpu() for t in dbatch])
        nb = ReadBatch(*[t.numpy().view({"torch.int16": np.uint16, "torch.int32": np.int32, "torch.uint8": np.uint8}[str(t.dtype)])
                         for t in hbatch])
        nb = ReadBatch(nb.tid, nb.pos, nb.flag, nb.mapq, nb.cig_off.view(np.uint32), nb.cig.view(np.uint32))
        cores = os.cpu_count() or 1
        al, dt = cpu_port_time(nb, lengths, (reg_tid, reg_start, reg_end), cores)
        al1, dt1 = cpu_port_time(nb, lengths, (reg_tid, reg_start, reg_end), 1, reps=0)
        py_rate, py_n = python_port_rate(nb, lengths, 1)
        cpu = {"value": al / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "full %s shard (%d reads) per step, C port oracle/coverage.c contig-parallel, best of 3" % (args.workload, n_reads),
               "one_core_value": al1 / dt1,
               "python_port_value": py_rate,
               "python_port_sample": "first contig (%d reads), reference-structured Python loop (one object per column), 1 core" % py_n}

    line = {
        "metric": METRIC, "value": aligned_total / (ms_step / 1e3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": workload_label(args.workload, world, w), "scale": args.scale,
                   "path": ("fused sorted path (k_fused_prep_tma, k_fused_tile_tma, k_stats_stream)" if args.path == "fused" else
                            "push path (memset, k_expand, k_scan_inplace): the any-order formulation"),
                   "per_gpu": {"reads": n_reads, "contigs": g, "slots": int(slots)},
                   "regions": "one whole-contig region per contig (reference util.py:64-69)",
                   "l2": "inputs+depth (%d MB per GPU) exceed the 126 MB L2; no explicit flush" %
                         ((batch_bytes(dbatch) + 4 * slots) // 2 ** 20),
                   "parallelism": "contig-range shards, 1 all-gather of 64 B/region" if world > 1 else "single GPU",
                   "pipelining": ("steps overlap on the host side only: step k's records are collected from a pinned slot "
                                  "after step k+1 is enqueued (mcov_region_stats_submit/collect); unpipelined_ms_per_step = "
                                  "one synchronising call per step") if world == 1 else
                                  "as N=1, with the NCCL all-gather of the records inside the pipeline (two DeviceGather slots)"},
        "unpipelined_ms_per_step": ms_sync,
        "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "aligned_bases_per_step": aligned_total, "strong_scaling": strong,
        "region_plan_first_call_ms": first_call_ms, "rank_affinity": affinity,
    }
    emit(args.real_stdout, line)
    if world > 1:
        dist.destroy_process_group()


def main():
    # stdout carries exactly ONE JSON line: everything else (NCCL's version banner, library chatter)
    # goes to stderr until the line is printed
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        _main(real_stdout)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)


def emit(real_stdout, line):
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())


def _main(real_stdout):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--path", default="fused", choices=["fused", "push"],
                    help="depth formulation of the device-resident step: fused sorted path (default, what sorted BAM input takes) "
                         "or the any-order push path (clear + atomics + decoupled look-back scan)")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the named workload per GPU")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the e2e legs (0: as many as --steps)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-bam", action="store_true", help="skip the from-the-BAM-file leg of e2e")
    ap.add_argument("--bam-reads", type=int, default=2_000_000, help="reads written to the synthetic BAM of the from-file leg")
    ap.add_argument("--bam-batch", type=int, default=1 << 19, help="records per batch of the streamed from-file pass")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block (config C4 sharded over the ranks)")
    ap.add_argument("--strong-scale", type=float, default=1.0, help="fraction of config C4 (1 B reads) used by the strong-scaling block")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--breakdown", action="store_true", help="print a host-side time breakdown of one step to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the statistics records and a sample of the depth of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    args.real_stdout = real_stdout
    if args.e2e_steps <= 0:
        args.e2e_steps = args.steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
