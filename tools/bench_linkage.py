#!/usr/bin/env python
"""Linkage (AlignmentFile.linkage, csrc/linkage.cu) against the count pass (k_bc_any) on the same file, and against the
host route (oracle/linkage.py over the decoded records).

Workloads: paired variants of bench_alleles.two_strain -- a random reference with two strains (1 % of positions carry
a second allele; a fragment comes from the minor strain with probability 0.2), fragments of two 150 bp mates with
inserts of 300-500 bp, both mates from the fragment's strain, 0.5 % sequencing error, --coverage over all reads:
  dense_c2   C2's table at --c2-scale (0.2: 200 x 50 kb = 10^7 slots)
  dense_c3   C3's contig-length table at --c3-scale (0.1: 50 k contigs, ~1.2 x 10^8 slots); contigs shorter than a
             fragment get no reads
Both are written as BAM and decoded on the device.  Kernel times are CUDA events (the engine's per-kernel profile; the
CUB sort and select are timed the same way), best of --reps runs that alternate linkage and the count pass.

Byte / atomic model (what the kernels must move at least, DRAM or L2):
  sites        16 B a slot (the counters, read once) + 32 B a site written
  observations 2 x 24 B a record (columns, read by the count and the write pass) + 16 B an observation written
  sort         32 B an observation a radix pass (read + write), ceil(bits / 8) passes
  unit calls   32 B an observation (read, write) + 32 B for the compaction
  pairs        16 B a call + 4 B an atomic (at least one per listed unit pair) + 16 B a candidate (counters read)
The share of HBM peak is the model over the kernel time at 7.7 TB/s (most of it is L2-resident at these sizes: an upper
bound on what the model can say).  The host route runs the oracle over the records of --host-frac of the contigs of
dense_c2 and is scaled to the whole file by records.  Prints one JSON line (and writes it to --out).

  python tools/bench_linkage.py [--reps 5] [--out profiles/r09_bench_linkage.json]
"""
import argparse
import json
import math
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_basecount import L_SEQ, card, write_bam_fast  # noqa: E402

HBM_PEAK = 7.7e12           # B/s, HGX B200 data sheet, one GPU
NT16 = np.array([1, 2, 4, 8], np.uint8)
PARAMS = dict(quality_threshold=15, min_coverage=5, min_freq=0.05, min_count=2, max_distance=1000, min_reads=20)


def paired_two_strain(lengths, coverage, seed, var_frac=0.01, minor=0.2, err=0.005):
    """Columns for write_bam_fast (+ names) of paired reads of two strains over a random reference."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lengths = np.asarray(lengths, np.int64)
    off = np.concatenate(([0], np.cumsum(lengths)))
    ref = rng.integers(0, 4, int(off[-1]), dtype=np.uint8)
    alt = ref.copy()
    var = rng.integers(0, len(ref), int(len(ref) * var_frac))
    alt[var] = (ref[var] + rng.integers(1, 4, len(var), dtype=np.uint8)) % 4
    room = np.maximum(lengths - 500 + 1, 0)
    n_frag = int(lengths.sum() * coverage // (2 * L_SEQ))
    ftid = rng.choice(len(lengths), n_frag, p=room / room.sum()).astype(np.int32)
    fpos = (rng.random(n_frag) * room[ftid]).astype(np.int64)
    ins = rng.integers(300, 501, n_frag)
    strain_b = rng.random(n_frag) < minor
    tid = np.repeat(ftid, 2)
    pos = np.stack([fpos, fpos + ins - L_SEQ], axis=1).reshape(-1).astype(np.int32)
    frag = np.repeat(np.arange(n_frag), 2)
    flag = np.tile(np.array([0x1 | 0x2 | 0x40, 0x1 | 0x2 | 0x80 | 0x10], np.uint16), n_frag)
    order = np.lexsort((pos, tid))
    tid, pos, frag, flag = tid[order], pos[order], frag[order], flag[order]
    n = len(tid)
    seq = np.empty((n, L_SEQ), np.uint8)
    step = 1 << 20
    for a in range(0, n, step):
        b = min(n, a + step)
        idx = off[tid[a:b]][:, None] + pos[a:b, None].astype(np.int64) + np.arange(L_SEQ)
        s = np.where(strain_b[frag[a:b]][:, None], alt[idx], ref[idx])
        e = rng.random(s.shape) < err
        s[e] = (s[e] + rng.integers(1, 4, int(e.sum()), dtype=np.uint8)) % 4
        seq[a:b] = NT16[s]
    qual = rng.integers(20, 41, (n, L_SEQ), dtype=np.uint8)
    mapq = np.full(n, 60, np.uint8)
    cig_off = np.arange(n + 1, dtype=np.uint32)
    cig = np.full(n, L_SEQ << 4, np.uint32)
    names = np.char.mod("f%010d", frag).astype("S12")
    return (tid, pos, flag, mapq, cig_off, cig, seq, qual), names


def host_route(cols, names, lengths, frac, seed):
    """The oracle over the records of a random `frac` of the contigs: (seconds, records, pairs)."""
    from oracle import linkage as ol
    tid, pos, flag, _mapq, _co, _cig, seq, qual = cols
    rng = np.random.default_rng(seed)
    pick = np.sort(rng.choice(len(lengths), max(1, int(len(lengths) * frac)), replace=False))
    sel = np.nonzero(np.isin(tid, pick))[0]
    remap = {int(c): k for k, c in enumerate(pick.tolist())}
    t = time.perf_counter()
    n = len(sel)
    pairs, _info = ol.linkage([int(lengths[c]) for c in pick], np.array([remap[int(x)] for x in tid[sel]], np.int32),
                              pos[sel], flag[sel], np.arange(n + 1, dtype=np.uint32), np.full(n, L_SEQ << 4, np.uint32),
                              [seq[i] for i in sel], [qual[i] for i in sel], [bytes(names[i]) for i in sel],
                              **PARAMS)
    return time.perf_counter() - t, n, len(pairs)


def bench_one(path, reps, n_rec):
    from metacov_b200 import AlignmentFile, _capi
    af = AlignmentFile(path, decode="gpu")
    eng = af._count_engine()
    t = time.perf_counter()
    af.count_coverage(af.references[0], 0, 1)
    t_count_first = time.perf_counter() - t
    t = time.perf_counter()
    pairs, info = af.linkage(**PARAMS)
    t_first = time.perf_counter() - t

    def timed(fn):
        eng.profile(True)
        eng.profile_read()
        t = time.perf_counter()
        r = fn()
        wall = time.perf_counter() - t
        prof = eng.profile_read()
        eng.profile(False)
        return r, wall, prof

    legs = {"linkage": lambda: af.linkage(**PARAMS),
            "count": lambda: eng.base_counts(15, _capi.MCOV_BC_ALL)}
    for _ in range(2):
        for fn in legs.values():
            fn()
    runs = {k: [] for k in legs}
    for _ in range(reps):
        for k, fn in legs.items():
            r, wall, prof = timed(fn)
            runs[k].append((sum(v[1] for v in prof.values()), wall, {kk: round(v[1], 4) for kk, v in prof.items()}))
            if k == "linkage":
                assert r[0].tobytes() == pairs.tobytes() and r[1] == info
    res = {"slots": int(eng.n_slots), "records": n_rec, "count_call_first_s": round(t_count_first, 3),
           "linkage_call_first_s": round(t_first, 3), "pairs": len(pairs), **info}
    for k, v in runs.items():
        kern, wall, names = min(v, key=lambda r: r[0])
        res[k] = {"kernel_ms": round(kern, 4), "call_ms": round(wall * 1e3, 3), "kernels": names,
                  "all_kernel_ms": [round(r[0], 4) for r in v], "all_call_ms": [round(r[1] * 1e3, 3) for r in v]}
    # the model
    n_obs, ns, n_cand = info["n_observations"], info["n_sites"], info["n_candidates"]
    sb = max(1, math.ceil(math.log2(max(ns, 2))))
    passes = math.ceil((128 - (61 - sb)) / 8)
    listed = int(sum(int(pairs[k].sum()) for k in ("n_AB", "n_Ab", "n_aB", "n_ab")))
    model = {"sites": 16 * res["slots"] + 32 * ns, "observations": 2 * 24 * n_rec + 16 * n_obs,
             "sort": 32 * n_obs * passes, "unit_calls": 64 * n_obs, "pairs": 16 * n_obs + 4 * listed + 16 * n_cand}
    res["model_bytes"] = model
    res["model_sort_passes"] = passes
    res["listed_unit_pairs"] = listed
    kern = res["linkage"]["kernel_ms"]
    res["linkage"]["hbm_share"] = round(sum(model.values()) / HBM_PEAK / (kern * 1e-3), 4)
    ks = res["linkage"]["kernels"]
    res["obs_pass_ms"] = round(ks.get("k_link_obs_count", 0) + ks.get("k_link_obs_write", 0), 4)
    res["aim_obs_pass_vs_count"] = round(res["obs_pass_ms"] / res["count"]["kernel_ms"], 3)
    res["aim_linkage_call_vs_count_call"] = round(min(r[1] for r in runs["linkage"]) / min(r[1] for r in runs["count"]), 3)
    af.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--coverage", type=float, default=30.0)
    ap.add_argument("--c2-scale", type=float, default=0.2)
    ap.add_argument("--c3-scale", type=float, default=0.1)
    ap.add_argument("--host-frac", type=float, default=0.02, help="share of dense_c2's contigs the oracle runs on")
    ap.add_argument("--skip", default="", help="comma-separated workloads to leave out")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from metacov_b200 import synth
    if not torch.cuda.is_available():
        sys.exit("bench_linkage: no CUDA device (the linkage kernels have no CPU path)")
    d = tempfile.mkdtemp()
    out = {"bench": "linkage", "card": card(), "reps": args.reps, "params": PARAMS}
    skip = set(filter(None, args.skip.split(",")))
    for name, lengths, host in (("dense_c2", synth.c2(args.c2_scale).contig_len, True),
                                ("dense_c3", synth.c3(args.c3_scale).contig_len, False)):
        if name in skip:
            continue
        t = time.perf_counter()
        cols, names = paired_two_strain(lengths, args.coverage, 7)
        pb = os.path.join(d, name + ".bam")
        write_bam_fast(pb, lengths, *cols, names=names)
        w = time.perf_counter() - t
        r = bench_one(pb, args.reps, len(cols[0]))
        r.update({"coverage": args.coverage, "write_s": round(w, 1), "file_bytes": os.path.getsize(pb)})
        if host:
            hs, hn, hp = host_route(cols, names, np.asarray(lengths), args.host_frac, 3)
            r["host_route"] = {"records": hn, "pairs": hp, "s": round(hs, 2),
                               "s_scaled_to_file": round(hs * r["records"] / max(hn, 1), 1)}
        os.remove(pb)
        out[name] = r
        print(json.dumps({name: r}), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
