#!/usr/bin/env python
"""Allele statistics and sites (AlignmentFile.allele_stats / allele_sites, csrc/alleles.cu) against the count pass
(k_bc_any) on the same input and against the host route they replace (copy_base_counts of every contig + the numpy
oracle).

Workloads:
  dense_c2   a random reference with two strains (1 % of positions carry a second allele in 20 % of the reads), 0.5 %
             sequencing error, 150 bp reads at --coverage, over C2's table at --c2-scale (0.2: 200 x 50 kb = 10^7 slots);
             written as BAM, decoded on the device, with the reference FASTA
  dense_c3   the same over C3's contig-length table scaled to --c3-scale (0.1: 50 k contigs, ~1.2 x 10^8 slots), at
             --c3-coverage
  sparse     C3's full table (500 k contigs, ~1.2 x 10^9 slots) with --sparse-reads reads; the reference uploaded too
Kernel times are CUDA events (the engine's per-kernel profile), best of --reps alternated runs; whole contigs are the
regions.  Byte model: 17 B a slot (counters + reference byte) read per pass; the region pass adds 64 B a chunk written and
read again and 64 B a region, the site pass 32 B a site (the second read of the tiles that hold a site is not counted).
The share of HBM peak is that over the kernel time at 7.7 TB/s.  Prints one JSON line (and writes it to --out).

  python tools/bench_alleles.py [--reps 5] [--out profiles/r07_bench_alleles.json]
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_basecount import L_SEQ, card, write_bam_fast  # noqa: E402

HBM_PEAK = 7.7e12           # B/s, HGX B200 data sheet, one GPU
NT16 = np.array([1, 2, 4, 8], np.uint8)


def two_strain(lengths, coverage, seed, var_frac=0.01, minor=0.2, err=0.005, n_reads=None):
    """Reads of two strains over a random reference: (columns for write_bam_fast, reference strings per contig).
    ``n_reads`` overrides the count that ``coverage`` gives."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lengths = np.asarray(lengths, np.int64)
    off = np.concatenate(([0], np.cumsum(lengths)))
    ref = rng.integers(0, 4, int(off[-1]), dtype=np.uint8)
    alt = ref.copy()
    var = rng.integers(0, len(ref), int(len(ref) * var_frac))
    alt[var] = (ref[var] + rng.integers(1, 4, len(var), dtype=np.uint8)) % 4
    n = int(n_reads if n_reads is not None else lengths.sum() * coverage // L_SEQ)
    room = np.maximum(lengths - L_SEQ + 1, 1)
    tid = np.sort(rng.choice(len(lengths), n, p=room / room.sum())).astype(np.int32)
    pos = (rng.random(n) * room[tid]).astype(np.int32)
    order = np.lexsort((pos, tid))
    tid, pos = tid[order], pos[order]
    seq = np.empty((n, L_SEQ), np.uint8)
    strain_b = rng.random(n) < minor
    step = 1 << 20
    for a in range(0, n, step):
        b = min(n, a + step)
        idx = off[tid[a:b]][:, None] + pos[a:b, None].astype(np.int64) + np.arange(L_SEQ)
        idx = np.minimum(idx, len(ref) - 1)
        s = np.where(strain_b[a:b, None], alt[idx], ref[idx])
        e = rng.random(s.shape) < err
        s[e] = (s[e] + rng.integers(1, 4, int(e.sum()), dtype=np.uint8)) % 4
        seq[a:b] = NT16[s]
    qual = rng.integers(20, 41, (n, L_SEQ), dtype=np.uint8)
    flag = np.where(rng.random(n) < 0.5, 16, 0).astype(np.uint16)
    mapq = np.full(n, 60, np.uint8)
    cig_off = np.arange(n + 1, dtype=np.uint32)
    cig = np.full(n, L_SEQ << 4, np.uint32)
    letters = np.frombuffer(b"ACGT", np.uint8)
    refs = [letters[ref[off[c]:off[c + 1]]].tobytes().decode() for c in range(len(lengths))]
    return (tid, pos, flag, mapq, cig_off, cig, seq, qual), refs


def write_fasta(path, refs):
    with open(path, "w") as fh:
        for c, s in enumerate(refs):
            fh.write(">c%d\n" % c)
            for a in range(0, len(s), 80):
                fh.write(s[a:a + 80] + "\n")


def write_workload(d, name, lengths, coverage, seed, n_reads=None):
    cols, refs = two_strain(lengths, coverage, seed, n_reads=n_reads)
    pb, pf = os.path.join(d, name + ".bam"), os.path.join(d, name + ".fa")
    write_bam_fast(pb, lengths, *cols)
    write_fasta(pf, refs)
    return pb, pf, len(cols[0])


def host_route(eng, n_contigs, lengths, refs, params):
    """What the feature replaces: every contig's counts to the host, then the numpy rules per contig."""
    from oracle import alleles as oa
    t = time.perf_counter()
    n_sites = 0
    for c in range(n_contigs):
        cnt = eng.copy_base_counts(c)
        r = oa.region_stats(cnt, refs[c], 0, int(lengths[c]), **params)
        n_sites += int((oa.evaluate(cnt, refs[c], **params)["kind"] != 0).sum())
        del r
    return time.perf_counter() - t, n_sites


def bench_one(name, path, fasta_path, reps, with_host):
    from metacov_b200 import AlignmentFile, FastaFile
    params = dict(min_coverage=5, min_freq=0.05, min_count=2)
    fa = FastaFile(fasta_path)
    af = AlignmentFile(path, decode="gpu")
    eng = af._count_engine()
    t = time.perf_counter()
    af.count_coverage(af.references[0], 0, 1)
    t_count_call = time.perf_counter() - t
    t = time.perf_counter()
    af.allele_stats(fasta=fa, **params)                  # (uploads the reference)
    t_first = time.perf_counter() - t
    n_slots = int(eng.n_slots)
    g = af.nreferences
    n_chunks = int(sum((int(l) + 2047) // 2048 for l in af.lengths))

    def timed(fn):
        eng.profile(True)
        eng.profile_read()
        t = time.perf_counter()
        r = fn()
        wall = time.perf_counter() - t
        prof = eng.profile_read()
        eng.profile(False)
        return r, wall, prof

    from metacov_b200 import _capi
    legs = {"stats": lambda: af.allele_stats(fasta=fa, **params),
            "sites": lambda: af.allele_sites(fasta=fa, **params),
            "count": lambda: eng.base_counts(15, _capi.MCOV_BC_ALL)}
    runs = {k: [] for k in legs}
    out = {}
    for _ in range(2):
        for fn in legs.values():
            fn()
    for _ in range(reps):
        for k, fn in legs.items():
            r, wall, prof = timed(fn)
            runs[k].append((sum(v[1] for v in prof.values()), wall, {kk: round(v[1], 4) for kk, v in prof.items()}))
            if k == "sites":
                out["n_sites"] = len(r)
    stats = af.allele_stats(fasta=fa, **params)
    res = {"slots": n_slots, "regions": g, "chunks": n_chunks, "count_call_s": round(t_count_call, 3),
           "first_stats_call_s": round(t_first, 3), "n_sites": out["n_sites"],
           "covered": int(stats["covered"].sum()), "snv": int(stats["snv"].sum())}
    model = {"stats": 17 * n_slots + 128 * n_chunks + 64 * g, "sites": 17 * n_slots + 32 * out["n_sites"],
             "count": None}
    for k, v in runs.items():
        kern, wall, names = min(v, key=lambda r: r[0])
        res[k] = {"kernel_ms": round(kern, 4), "call_ms": round(wall * 1e3, 3), "kernels": names,
                  "all_kernel_ms": [round(r[0], 4) for r in v]}
        if model[k]:
            res[k]["model_bytes"] = model[k]
            res[k]["hbm_share"] = round(model[k] / HBM_PEAK / (kern * 1e-3), 4)
    if with_host:
        refs = [fa.fetch(n.split()[0]) for n in af.references]
        res["host_route_s"], n_host = host_route(eng, g, af.lengths, refs, params)
        res["host_route_s"] = round(res["host_route_s"], 2)
        assert n_host == out["n_sites"], (n_host, out["n_sites"])
    af.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--coverage", type=float, default=30.0)
    ap.add_argument("--c2-scale", type=float, default=0.2)
    ap.add_argument("--c3-scale", type=float, default=0.1)
    ap.add_argument("--c3-coverage", type=float, default=30.0)
    ap.add_argument("--sparse-reads", type=int, default=200_000)
    ap.add_argument("--skip", default="", help="comma-separated workloads to leave out")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from metacov_b200 import synth
    if not torch.cuda.is_available():
        sys.exit("bench_alleles: no CUDA device (the allele kernels have no CPU path)")
    d = tempfile.mkdtemp()
    out = {"bench": "alleles", "card": card(), "reps": args.reps}
    skip = set(filter(None, args.skip.split(",")))
    work = [("dense_c2", synth.c2(args.c2_scale).contig_len, args.coverage, None, True),
            ("dense_c3", synth.c3(args.c3_scale).contig_len, args.c3_coverage, None, True),
            ("sparse", synth.c3(1.0).contig_len, 0, args.sparse_reads, False)]
    for name, lengths, cov, n_reads, host in work:
        if name in skip:
            continue
        t = time.perf_counter()
        pb, pf, n = write_workload(d, name, lengths, cov, 7, n_reads=n_reads)
        w = time.perf_counter() - t
        r = bench_one(name, pb, pf, args.reps, host)
        r.update({"reads": n, "coverage": cov, "write_s": round(w, 1), "file_bytes": os.path.getsize(pb)})
        out[name] = r
        for p in (pb, pf):
            os.remove(p)
        print(json.dumps({name: r}), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
