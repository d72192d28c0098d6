#!/usr/bin/env python
"""SAM text through a pipe to per-base depth, the way an aligner's output reaches ``metacov pileup -b -``.

The 2 M-read C2 SAM of ``tools/bench_bam.py --sam`` (QUAL of full length, two optional fields) is held in memory and
written into an ``os.pipe`` (capacity set to 1 MiB with F_SETPIPE_SZ) by a writer thread, in 1 MiB writes.  Timed, each
from the first byte written to the last result:
  drain          a reader that only empties the pipe into a buffer of the chunk size (``readinto``): what the pipe allows;
  reader         ``samstream.ChunkReader`` with a decoder that does nothing: the host side of the piped path alone (reader
                 thread, two buffers, the cut at the last LF, the carried tail);
  pileup         ``AlignmentFile(pipe)`` + the depth of every contig (chunked GPU decode, any-order pass with the exact
                 cap verdict) + ``mapped``, with pageable host buffers (the default);
  pileup_pinned  the same with page-locked buffers (``pinned_buffers=True``);
  scan           ``AlignmentFile(pipe)`` + ``scan_reads`` with ``ByFlag([IsizeHist, KmerHist])``.
The arms alternate, and the best of ``--reps`` rounds of each is reported.  A last, separate pileup run with per-kernel
event timing gives the device time of the piped pass by kernel.  Prints one JSON line with the card's name and power
limit.

  python tools/bench_pipe.py [--scale 0.2] [--reps 3] [--chunk-mb 64] [--out FILE]
"""
import argparse
import fcntl
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _c2_sam(scale):
    from metacov_b200 import synth
    from oracle import bamio
    import samio                                                # (the SAM writer of the tests, as in bench_bam.py --sam)
    w = synth.c2(scale)
    hb, isz = synth.generate_host(w)
    rng = np.random.Generator(np.random.PCG64(11))
    big = np.array([1, 2, 4, 8], dtype=np.uint8)[rng.integers(0, 4, len(hb.tid) * 150, dtype=np.uint8)]
    letters = np.frombuffer(bamio.NT16.encode(), np.uint8)[big].tobytes().decode()
    n = len(hb.tid)
    path = os.path.join(tempfile.mkdtemp(), "c2.sam")
    samio.write_sam(path, ["c%d" % c for c in range(w.n_contigs)], [int(x) for x in w.contig_len], hb.tid, hb.pos, hb.flag,
                    hb.mapq, hb.cig_off, hb.cig, isize=isz, seqs=[letters[i * 150:(i + 1) * 150] for i in range(n)],
                    quals=["F" * 150] * n, aux=["NM:i:%d\tAS:i:%d" % (i % 4, 150 - i % 4) for i in range(n)])
    with open(path, "rb") as f:
        data = f.read()
    os.unlink(path)
    return data, n


def _pipe(data):
    """The read end of a pipe that a writer thread fills with `data` in 1 MiB writes."""
    r, w = os.pipe()
    fcntl.fcntl(w, fcntl.F_SETPIPE_SZ, 1 << 20)
    mv = memoryview(data)

    def writer():
        try:
            p = 0
            while p < len(mv):
                p += os.write(w, mv[p:p + (1 << 20)])
        except OSError:
            pass
        finally:
            os.close(w)

    t = threading.Thread(target=writer, daemon=True)
    t.start()
    return os.fdopen(r, "rb", buffering=0), t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=0.2, help="fraction of config C2 (10 M reads)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--chunk-mb", type=int, default=64)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    from metacov_b200 import AlignmentFile
    from metacov_b200 import scan as mscan
    if not torch.cuda.is_available():
        raise SystemExit("bench_pipe.py needs a GPU")
    data, n = _c2_sam(args.scale)
    chunk = args.chunk_mb << 20

    def drain():
        f, t = _pipe(data)
        t0 = time.perf_counter()
        buf = bytearray(chunk)
        mv = memoryview(buf)
        got = 0
        while True:
            k = f.readinto(mv)
            if not k:
                break
            got += k
        dt = time.perf_counter() - t0
        mv.release()
        f.close()
        t.join()
        assert got == len(data)
        return dt

    def reader():
        from metacov_b200 import samstream
        f, t = _pipe(data)
        t0 = time.perf_counter()
        rd = samstream.ChunkReader(samstream._Source(f), b"", chunk)
        rd.run(lambda view, last: True)
        dt = time.perf_counter() - t0
        f.close()
        t.join()
        assert rd.bytes == len(data)
        return dt

    def pileup(pinned=False, profile=False):
        f, t = _pipe(data)
        t0 = time.perf_counter()
        with AlignmentFile(f, gpu_chunk_bytes=chunk, pinned_buffers=pinned) as s:
            if profile:
                s._pipe_eng.profile(True)
            eng = s.coverage_engine()
            eng.sync()
            m = s.mapped
            dt = time.perf_counter() - t0
            info = dict(s.pipe_info, mapped=m, n_pass=eng.pass_info()["n_pass"], cap_metric=eng.pass_info()["cap_metric"])
            if profile:
                info = {k: v[1] for k, v in eng.profile_read().items() if v[0]}
        f.close()
        t.join()
        return dt, info

    def scan():
        f, t = _pipe(data)
        t0 = time.perf_counter()
        with AlignmentFile(f, gpu_chunk_bytes=chunk) as s:
            bf = mscan.ByFlag([mscan.IsizeHist(), mscan.KmerHist(7, 8, 7, 0)], [mscan.Flags["Mapped"]])
            nrec = mscan.scan_reads(s, None, bf)
            dt = time.perf_counter() - t0
        f.close()
        t.join()
        assert nrec == n
        return dt

    pileup()                                                    # warm-up: module load, engine creation, allocations
    pileup(pinned=True)
    scan()
    runs = {"drain": [], "reader": [], "pileup": [], "pileup_pinned": [], "scan": []}
    info = None
    for _ in range(args.reps):
        runs["drain"].append(drain())
        runs["reader"].append(reader())
        dt, info = pileup()
        runs["pileup"].append(dt)
        runs["pileup_pinned"].append(pileup(pinned=True)[0])
        runs["scan"].append(scan())
    best = {k: min(v) for k, v in runs.items()}
    _, kernel_ms = pileup(profile=True)
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        card = torch.cuda.get_device_name(0)
    out = {"sam_bytes": len(data), "records": n, "chunk_bytes": chunk,
           "drain_s": best["drain"], "reader_s": best["reader"], "pileup_s": best["pileup"],
           "pileup_pinned_s": best["pileup_pinned"], "scan_s": best["scan"],
           "reader_over_drain": best["reader"] / best["drain"], "pileup_over_drain": best["pileup"] / best["drain"],
           "pileup_pinned_over_drain": best["pileup_pinned"] / best["drain"], "scan_over_drain": best["scan"] / best["drain"],
           "drain_gbs": len(data) / best["drain"] / 1e9, "pileup_gbs": len(data) / best["pileup"] / 1e9,
           "kernel_ms": kernel_ms, "kernel_ms_total": sum(kernel_ms.values()),
           "pipe_info": info, "runs": runs, "card": card}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
