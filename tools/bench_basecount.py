#!/usr/bin/env python
"""A / C / G / T counts of every position (AlignmentFile.count_coverage, csrc/basecount.cu) against the depth pass and
the GPU decode of the same BAM.

Input: config C2 at --scale (0.2: 2 M reads of 150 bp over 200 contigs of 50 kb, 30x) with random A/C/G/T bases and
random qualities 2-40, written as a coordinate-sorted BAM and as a shuffled copy, each decoded on the device.  Timed with
CUDA events (the engine's per-kernel profile) and a host clock around each synchronising call, best of --reps
alternated runs:
  any_sorted    k_bc_any on the sorted columns
  any_shuffled  k_bc_any on the shuffled columns
  depth         the fused depth pass on the sorted columns (bamgpu.depth_sorted), the yardstick
  decode        the GPU decode of the sorted BAM from its path (bamgpu.decode)
Byte model of a count: SEQ + QUAL + ops + the columns read (tid, pos, flag, l_seq, cig_off, rec_off), and the counters
read and written once (32 B a slot); the share of HBM peak is that over the kernel time at 7.7 TB/s.  The two counts
are checked equal.  Prints one JSON line (and writes it to --out).

  python tools/bench_basecount.py [--scale 0.2] [--reps 5] [--out file.json]
"""
import argparse
import json
import os
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12           # B/s, HGX B200 data sheet, one GPU
L_SEQ = 150


def _bgzf(data, level=1, block=0xff00):
    def one(i):
        p = data[i:i + block]
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        cd = c.compress(p) + c.flush()
        head = struct.pack("<BBBBIBBHBBHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, 66, 67, 2, len(cd) + 25)
        return head + cd + struct.pack("<II", zlib.crc32(p) & 0xFFFFFFFF, len(p))
    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        blocks = list(ex.map(one, range(0, len(data), block)))
    return b"".join(blocks) + bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def write_bam_fast(path, lengths, tid, pos, flag, mapq, cig_off, cig, seq_nt16, qual):
    """A BAM of fixed-length reads (SEQ / QUAL [n, L_SEQ]) from columns, built with numpy (record layout SAM spec 4.2)."""
    n = len(tid)
    nop = np.diff(cig_off.astype(np.int64))
    fixed = np.zeros(n, dtype=[("bs", "<i4"), ("ref", "<i4"), ("pos", "<i4"), ("ln", "u1"), ("mq", "u1"), ("bin", "<u2"),
                                ("nc", "<u2"), ("fl", "<u2"), ("ls", "<i4"), ("nr", "<i4"), ("np", "<i4"), ("tl", "<i4"),
                                ("name", "S12")])
    sq = (L_SEQ + 1) // 2
    body = 32 + 12 + 4 * nop + sq + L_SEQ
    fixed["bs"] = body; fixed["ref"] = tid; fixed["pos"] = pos; fixed["ln"] = 12; fixed["mq"] = mapq; fixed["bin"] = 4680
    fixed["nc"] = nop; fixed["fl"] = flag; fixed["ls"] = L_SEQ; fixed["nr"] = -1; fixed["np"] = -1
    fixed["name"] = np.char.mod("r%010d", np.arange(n)).astype("S12")
    text = ("@HD\tVN:1.4\tSO:coordinate\n" + "".join("@SQ\tSN:c%d\tLN:%d\n" % (c, l) for c, l in enumerate(lengths))).encode()
    head = b"BAM\x01" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(lengths))
    for c, l in enumerate(lengths):
        nm = b"c%d\0" % c
        head += struct.pack("<i", len(nm)) + nm + struct.pack("<i", int(l))
    starts = len(head) + np.concatenate(([0], np.cumsum(4 + body)))[:-1]
    out = np.zeros(int(starts[-1] + 4 + body[-1]), dtype=np.uint8)
    out[:len(head)] = np.frombuffer(head, np.uint8)
    packed = ((seq_nt16[:, 0::2] << 4) | seq_nt16[:, 1::2]).astype(np.uint8)
    fb = fixed.view(np.uint8).reshape(n, 48)
    cb = cig.astype("<u4").view(np.uint8).reshape(-1, 4)
    step = 1 << 18
    for a in range(0, n, step):
        b = min(n, a + step)
        s = starts[a:b]
        out[s[:, None] + np.arange(48)] = fb[a:b]
        o0, o1 = int(cig_off[a]), int(cig_off[b])
        rec = np.repeat(np.arange(a, b), nop[a:b])
        dst = starts[rec] + 48 + 4 * (np.arange(o0, o1) - cig_off[rec].astype(np.int64))
        out[dst[:, None] + np.arange(4)] = cb[o0:o1]
        t = s + 48 + 4 * nop[a:b]
        out[t[:, None] + np.arange(sq)] = packed[a:b]
        out[(t + sq)[:, None] + np.arange(L_SEQ)] = qual[a:b]
    with open(path, "wb") as fh:
        fh.write(_bgzf(out.tobytes()))


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=0.2, help="fraction of config C2 (10 M reads)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from metacov_b200 import CoverageEngine, _capi, bamgpu, synth
    if not torch.cuda.is_available():
        sys.exit("bench_basecount: no CUDA device (the counts have no CPU path)")
    w = synth.c2(args.scale)
    hb, _isz = synth.generate_host(w)
    n = len(hb.tid)
    rng = np.random.Generator(np.random.PCG64(6))
    seq = np.array([1, 2, 4, 8], dtype=np.uint8)[rng.integers(0, 4, (n, L_SEQ), dtype=np.uint8)]
    qual = rng.integers(2, 41, (n, L_SEQ), dtype=np.uint8)
    d = tempfile.mkdtemp()
    t0 = time.perf_counter()
    cols = [np.asarray(x) for x in (hb.tid, hb.pos, hb.flag, hb.mapq)]
    off, cig = np.asarray(hb.cig_off, np.uint32), np.asarray(hb.cig, np.uint32)
    p_sorted, p_shuf = os.path.join(d, "sorted.bam"), os.path.join(d, "shuffled.bam")
    write_bam_fast(p_sorted, w.contig_len, *cols, off, cig, seq, qual)
    perm = rng.permutation(n)
    nop = np.diff(off.astype(np.int64))
    off_p = np.concatenate(([0], np.cumsum(nop[perm]))).astype(np.uint32)
    idx = np.repeat(off[perm].astype(np.int64) - off_p[:-1].astype(np.int64), nop[perm]) + np.arange(int(off_p[-1]))
    cig_p = cig[idx]
    write_bam_fast(p_shuf, w.contig_len, *[c[perm] for c in cols], off_p, cig_p, seq[perm], qual[perm])
    t_write = time.perf_counter() - t0
    n_ops = int(off[-1])

    e_s, e_u = CoverageEngine(w.contig_len), CoverageEngine(w.contig_len)
    soa_s = bamgpu.decode(e_s, p_sorted)
    bamgpu.decode(e_u, p_shuf)

    def timed(eng, fn):
        eng.profile(True)
        eng.profile_read()                                   # (clears the totals)
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        eng.sync()
        wall = time.perf_counter() - t
        prof = eng.profile_read()
        eng.profile(False)
        return wall, prof

    runs = {"any_sorted": [], "any_shuffled": [], "depth": []}
    legs = [("any_sorted", e_s, lambda: e_s.base_counts(15, _capi.MCOV_BC_ALL), "k_bc_any"),
            ("any_shuffled", e_u, lambda: e_u.base_counts(15, _capi.MCOV_BC_ALL), "k_bc_any"),
            ("depth", e_s, lambda: bamgpu.depth_sorted(e_s, soa_s), None)]
    for _ in range(2):                                       # warm-up of every leg
        for _name, eng, fn, _k in legs:
            fn(); eng.sync()
    for _ in range(args.reps):
        for name, eng, fn, k in legs:
            wall, prof = timed(eng, fn)
            kern = prof[k][1] if k else sum(v[1] for kk, v in prof.items())
            assert k is None or prof[k][0] == 1, (name, prof)
            runs[name].append((kern, wall, sorted(prof)))
    # the decode, alternated with a count on its own engine
    dec = []
    e_d = CoverageEngine(w.contig_len)
    for _ in range(max(2, args.reps // 2)):
        torch.cuda.synchronize()
        t = time.perf_counter()
        bamgpu.decode(e_d, p_sorted)
        e_d.sync()
        dec.append(time.perf_counter() - t)
    e_d.close()
    # the two counts agree
    res = {}
    for name, eng, fn, _k in legs[:2]:
        fn()
        res[name] = np.concatenate([eng.copy_base_counts(c) for c in range(w.n_contigs)], axis=1)
    assert np.array_equal(res["any_sorted"], res["any_shuffled"])
    counted = int(res["any_sorted"].sum())
    # byte model of one count
    n_slots = int(e_s.n_slots)
    bytes_read = n * ((L_SEQ + 1) // 2 + L_SEQ + 4 + 4 + 2 + 4 + 4 + 8) + 4 * n_ops
    bytes_cnt = 2 * 16 * n_slots
    best = {k: min(v, key=lambda r: r[0]) for k, v in runs.items()}
    out = {"bench": "basecount", "card": card(), "scale": args.scale, "reads": n, "ops": n_ops, "slots": n_slots,
           "file_bytes": os.path.getsize(p_sorted), "counted_bases": counted, "write_s": round(t_write, 1), "reps": args.reps}
    for k, (kern, wall, names) in best.items():
        out[k] = {"kernel_ms": round(kern, 4), "call_ms": round(wall * 1e3, 3), "kernels": names}
        if k != "depth":
            out[k]["hbm_share"] = round((bytes_read + bytes_cnt) / HBM_PEAK / (kern * 1e-3), 4)
            out[k]["atomics_per_s"] = round(counted / (kern * 1e-3) / 1e9, 2)
    out["decode_ms"] = round(min(dec) * 1e3, 2)
    out["model_bytes"] = bytes_read + bytes_cnt
    out["all_kernel_ms"] = {k: [round(r[0], 4) for r in v] for k, v in runs.items()}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    e_s.close(); e_u.close()


if __name__ == "__main__":
    main()
