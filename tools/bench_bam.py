#!/usr/bin/env python
"""From the BAM FILE to per-base depth, three ways, each timed from the closed file on disk to the finished depth:
  host_decode   whole-file host reader (mcov_bam_open/load: zlib on all host cores + serial record walk), H2D of the SoA;
  host_stream   the streaming reader (mcov_bam_stream_*: batches decoded into pinned sets and pushed while the next one
                is decoded) -- what AlignmentFile does by default;
  gpu_decode    the file is read into a pinned staging buffer (allocated once, like the engine's own staging; the READ is
                inside the timed region), the compressed image goes over PCIe, inflate + record chain + SoA on the device.
  gpu_stream    mcov_bam_gpu_stream_depth: the file read chunk by chunk into pinned memory by a host thread, each chunk
                inflated / chained / parsed on the device and pushed into the streamed pass (any file size).
  sam (--sam)   the same reads as SAM text (QUAL of full length, two optional fields): the file is read into a pinned
                staging buffer (inside the timed region, like gpu_decode), parsed on the device (bamgpu.decode_sam) and
                the depth computed; against it, a plain host-to-device copy of the same bytes from the same staging buffer,
                the runs of the two alternated.
SURVEY.md 8(f) row 3.  Prints one JSON line.

  python tools/bench_bam.py [--scale 0.2] [--reps 3] [--sam]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=0.2, help="fraction of config C2 (10 M reads) written to the BAM")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--bam", default=None, help="reuse / create the synthetic BAM at this path")
    ap.add_argument("--sam", action="store_true", help="also time the SAM text leg")
    args = ap.parse_args()
    import torch
    from metacov_b200 import AlignmentFile, CoverageEngine, bamgpu, synth
    from oracle import bamio
    w = synth.c2(args.scale)
    hb, isz = synth.generate_host(w)
    d = tempfile.mkdtemp()
    path = args.bam or os.path.join(d, "c2.bam")
    t0 = time.perf_counter()
    if args.bam and os.path.exists(path):
        return _measure(args, path, w, hb, 0.0)
    # random bases (nt16 codes of A C G T) so that the file compresses like sequence data, not like padding;
    # l_seq follows the CIGAR-independent read length of the generator (150)
    rng = np.random.Generator(np.random.PCG64(11))
    big = np.array([1, 2, 4, 8], dtype=np.uint8)[rng.integers(0, 4, len(hb.tid) * 150, dtype=np.uint8)]
    seqs = [big[i * 150:(i + 1) * 150] for i in range(len(hb.tid))]
    bamio.write_bam(path, ["c%d" % c for c in range(w.n_contigs)], [int(x) for x in w.contig_len], hb.tid, hb.pos, hb.flag,
                    hb.mapq, hb.cig_off, hb.cig, isize=isz, seqs=seqs)
    t_write = time.perf_counter() - t0
    if args.sam:
        # the same records as SAM text, with the lines an aligner writes: QUAL of full length, two optional fields
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import samio                                            # (the SAM writer of the tests)
        letters = np.frombuffer(bamio.NT16.encode(), np.uint8)[big].tobytes().decode()
        n = len(hb.tid)
        args.sam_path = os.path.join(d, "c2.sam")
        samio.write_sam(args.sam_path, ["c%d" % c for c in range(w.n_contigs)], [int(x) for x in w.contig_len], hb.tid, hb.pos,
                        hb.flag, hb.mapq, hb.cig_off, hb.cig, isize=isz, seqs=[letters[i * 150:(i + 1) * 150] for i in range(n)],
                        quals=["F" * 150] * n, aux=["NM:i:%d\tAS:i:%d" % (i % 4, 150 - i % 4) for i in range(n)])
        del letters
    del seqs, big
    return _measure(args, path, w, hb, t_write)


def _measure(args, path, w, hb, t_write):
    import torch
    from metacov_b200 import AlignmentFile, CoverageEngine, bamgpu
    size = os.path.getsize(path)
    n = len(hb.tid)
    eng = CoverageEngine(w.contig_len)

    def host_path():
        t0 = time.perf_counter()
        with AlignmentFile(path) as bam:
            t1 = time.perf_counter()                 # file read + inflate (all host cores) + header
            s = bam.soa()
            t2 = time.perf_counter()                 # serial record walk -> SoA
            from metacov_b200 import ReadBatch
            eng.depth_sorted(ReadBatch(s["tid"], s["pos"], s["flag"], s["mapq"], s["cig_off"], s["cig"]))
            t3 = time.perf_counter()                 # H2D of the SoA + kernels
        return t1 - t0, t2 - t1, t3 - t2

    def stream_path():
        from metacov_b200.alignmentfile import BamStream, stream_depth
        t0 = time.perf_counter()
        with BamStream(path) as st:
            stream_depth(eng, st)
        return time.perf_counter() - t0

    t0 = time.perf_counter()
    staging = torch.empty(size, dtype=torch.uint8).pin_memory()      # persistent staging buffer: allocated once, reported
    t_pin = time.perf_counter() - t0
    staging_np = staging.numpy()

    def gpu_path(crc=True):
        t0 = time.perf_counter()
        with open(path, "rb", buffering=0) as fh:
            got = fh.readinto(memoryview(staging_np))
        assert got == size
        t1 = time.perf_counter()                     # file -> pinned staging
        soa = bamgpu.decode(eng, staging, verify_crc=crc)
        t2 = time.perf_counter()                     # H2D of the compressed image + inflate + record chain + SoA
        bamgpu.depth_sorted(eng, soa)
        t3 = time.perf_counter()
        return t1 - t0, t2 - t1, t3 - t2, soa

    def gpu_stream_path(chunk):
        t0 = time.perf_counter()
        info = bamgpu.stream_depth(eng, path, chunk_bytes=chunk)
        eng.sync()
        return time.perf_counter() - t0, info

    host = [host_path() for _ in range(args.reps)]
    stream = [stream_path() for _ in range(args.reps)]
    gpu_path()
    eng.profile(True)
    gpu = [gpu_path()[:3] for _ in range(args.reps)]
    kt = eng.profile_read()
    eng.profile(False)
    soa = gpu_path()[3]
    nocrc = min((gpu_path(crc=False)[:3] for _ in range(args.reps)), key=sum)
    gs = {}
    for chunk in (max(1 << 20, size // 4), 256 << 20):
        gpu_stream_path(chunk)
        runs = [gpu_stream_path(chunk) for _ in range(args.reps)]
        bt, info = min(runs, key=lambda r: r[0])
        gs["chunk_%d" % chunk] = {"total_s": bt, "reads_per_s": n / bt, "chunks": int(info["n_chunks"]), "max_carry": int(info["max_carry"])}
    sam = _measure_sam(args, eng, size, n, sum(min(gpu, key=sum)[1:])) if getattr(args, "sam_path", None) else None
    best_h = min(host, key=sum)
    best_g = min(gpu, key=sum)
    best_s = min(stream)
    kern = {k: v[1] / max(v[0], 1) for k, v in kt.items() if k.startswith("k_b")}
    line = {
        "what": "BAM file -> per-base depth", "reads": n, "bam_bytes": size, "inflated_bytes": int(soa.inflated_bytes),
        "segments": int(soa.n_segments), "host_cores": os.cpu_count(),
        "host_decode": {"open_inflate_s": best_h[0], "record_walk_s": best_h[1], "h2d_and_depth_s": best_h[2], "total_s": sum(best_h),
                        "reads_per_s": n / sum(best_h)},
        "host_stream": {"total_s": best_s, "reads_per_s": n / best_s},
        "gpu_decode": {"file_read_s": best_g[0], "decode_s": best_g[1], "depth_s": best_g[2], "total_s": sum(best_g),
                       "reads_per_s": n / sum(best_g), "decode_s_without_crc_check": nocrc[1],
                       "staging_alloc_once_s": t_pin, "kernel_ms": kern,
                       "inflate_gbs_out": soa.inflated_bytes / (kern.get("k_bgzf_inflate", 0) or float("nan")) / 1e6},
        "gpu_stream": gs,
        "timed": "every arm: closed file on disk (page cache warm) -> depth ready",
        "speedup_total": sum(best_h) / sum(best_g), "speedup_vs_stream": best_s / sum(best_g), "bam_write_s": t_write,
    }
    if sam is not None:
        line["sam"] = sam
    print(json.dumps(line))
    eng.close()


def _measure_sam(args, eng, bam_size, n, bam_decode_depth_s):
    """SAM file -> depth through decode_sam, against a plain copy of the same bytes from the same pinned buffer."""
    import subprocess
    import torch
    from metacov_b200 import bamgpu
    path = args.sam_path
    size = os.path.getsize(path)
    staging = torch.empty(size, dtype=torch.uint8).pin_memory()
    staging_np = staging.numpy()
    dst = torch.empty(size, dtype=torch.uint8, device="cuda:%d" % eng.device)

    def read():
        with open(path, "rb", buffering=0) as fh:
            assert fh.readinto(memoryview(staging_np)) == size

    def sam_path():
        t0 = time.perf_counter()
        read()
        t1 = time.perf_counter()
        soa = bamgpu.decode_sam(eng, staging)                   # (synchronises)
        t2 = time.perf_counter()
        bamgpu.depth_sorted(eng, soa)
        t3 = time.perf_counter()
        return t1 - t0, t2 - t1, t3 - t2, soa

    def copy_path():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dst.copy_(staging, non_blocking=True)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    soa = sam_path()[3]                                         # warm-up of every shape
    copy_path()
    runs, copies = [], []
    for _ in range(max(args.reps, 3)):                          # alternated
        runs.append(sam_path()[:3])
        copies.append(copy_path())
    eng.profile(True)
    sam_path()
    kt = eng.profile_read()
    eng.profile(False)
    kern = {k: v[1] / max(v[0], 1) for k, v in kt.items() if k.startswith("k_sam")}
    best = min(runs, key=lambda r: r[1] + r[2])
    best_copy = min(copies)
    parse_ms = sum(kern.values())
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(eng.device)],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        card = torch.cuda.get_device_name(eng.device)
    return {"sam_bytes": size, "records": int(soa.n_records), "sam_over_bam_bytes": size / bam_size, "bytes_per_line": size / n,
            "file_read_s": best[0], "decode_s": best[1], "depth_s": best[2], "decode_and_depth_s": best[1] + best[2],
            "plain_copy_s": best_copy, "copy_gbs": size / best_copy / 1e9,
            "decode_and_depth_over_copy": (best[1] + best[2]) / best_copy, "kernel_ms": kern,
            "parse_kernels_gbs": size / parse_ms / 1e6 if parse_ms else float("nan"),
            "bam_gpu_decode_and_depth_s": bam_decode_depth_s, "runs": [list(r) for r in runs], "copies": copies, "card": card}


if __name__ == "__main__":
    main()
