#!/usr/bin/env python
"""Genes (AlignmentFile.gene_stats / CoverageEngine.gene_stats, csrc/genes.cu) against the allele region pass over the
same intervals and against the host route they replace (copy_base_counts of every contig + the numpy oracle).

Workloads: tools/bench_alleles.two_strain (1 % of positions carry a second allele in 20 % of the reads, 0.5 %
sequencing error, 150 bp reads at --coverage, written as BAM and decoded on the device, with the reference FASTA), plus
genes of about 1 kb that tile about 88 % of each contig, on both strands, in all three phases:
  dense_c2   C2's table at --c2-scale (0.2: 200 x 50 kb = 10^7 slots)
  dense_c3   C3's contig-length table at --c3-scale (0.1: 50 k contigs, ~1.2 x 10^8 slots)
Kernel times are CUDA events (the engine's per-kernel profile), best of --reps alternated runs; call times are host
clocks around calls that end in a synchronise.  Legs: the gene call with its site list, without it, and allele_stats
(use_reference) over the same intervals.  Byte model of k_gene_chunks: 17 B a slot of the genes' codon spans (counters
+ reference byte) plus 40 B a chunk read and 72 B a chunk written (partial + record count); its share of HBM peak is
that over the kernel time at 7.7 TB/s.  The host route runs in full on dense_c2; on dense_c3 only its copy of the
counts is timed (a lower bound).  Prints one JSON line (and writes it to --out).

  python tools/bench_genes.py [--reps 5] [--out profiles/r10_bench_genes.json]
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

from bench_alleles import HBM_PEAK, write_workload  # noqa: E402
from bench_basecount import card  # noqa: E402

CHUNK_CODONS = 640          # kGnChunk (csrc/k_genes.cuh)


def tile_genes(lengths, seed, cover=0.88, mean_len=1000):
    """Genes of 600-1400 bp (300 or more at a contig's end) separated by gaps that leave about ``cover`` of each contig
    in a gene; strand and phase random.  Columns (tid, start, end, strand, phase) as int64 arrays."""
    rng = np.random.Generator(np.random.PCG64(seed))
    gap = mean_len * (1.0 - cover) / cover
    cols = [[], [], [], [], []]
    for t, n in enumerate(np.asarray(lengths, np.int64).tolist()):
        p = int(rng.integers(0, int(2 * gap) + 1))
        while True:
            ln = min(int(rng.integers(mean_len - 400, mean_len + 401)), n - p)
            if ln < 300:
                break
            for c, v in zip(cols, (t, p, p + ln, int(rng.choice([1, -1])), int(rng.integers(0, 3)))):
                c.append(v)
            p += ln + int(rng.integers(0, int(2 * gap) + 1))
    return [np.array(c, np.int64) for c in cols]


def host_route(eng, genes, refs, params, copy_only):
    """What the feature replaces: every contig's counts to the host, then the numpy gene rules per contig."""
    from oracle import genes as og
    tid = genes[0]
    t = time.perf_counter()
    n_sites = 0
    for c in range(len(refs)):
        cnt = eng.copy_base_counts(c)
        if copy_only:
            continue
        sel = np.nonzero(tid == c)[0]
        if len(sel):
            gl = [(0, int(genes[1][k]), int(genes[2][k]), int(genes[3][k]), int(genes[4][k])) for k in sel]
            n_sites += len(og.genes([cnt], [refs[c]], gl, **params)[1])
    return time.perf_counter() - t, n_sites


def bench_one(path, fasta_path, reps, host_copy_only):
    from metacov_b200 import AlignmentFile, FastaFile
    params = dict(min_coverage=5, min_freq=0.05, min_count=2)
    fa = FastaFile(fasta_path)
    af = AlignmentFile(path, decode="gpu")
    eng = af._count_engine()
    genes = tile_genes(af.lengths, 11)
    tid, start, end, strand, phase = genes
    af.allele_stats(["c0"], [0], [1], fasta=fa, **params)           # counts + the reference upload
    g = len(tid)
    k_codons = np.maximum(end - start - phase, 0) // 3
    span_slots = int(3 * k_codons.sum())
    n_chunks = int(((k_codons + CHUNK_CODONS - 1) // CHUNK_CODONS).sum())

    def timed(fn):
        eng.profile(True)
        eng.profile_read()
        t = time.perf_counter()
        r = fn()
        wall = time.perf_counter() - t
        prof = eng.profile_read()
        eng.profile(False)
        return r, wall, prof

    legs = {"genes_sites": lambda: eng.gene_stats(tid, start, end, strand, phase, sites=True, **params),
            "genes": lambda: eng.gene_stats(tid, start, end, strand, phase, **params),
            "allele_stats": lambda: eng.allele_stats(tid, start, end, use_reference=True, **params)}
    for _ in range(2):
        for fn in legs.values():
            fn()
    runs = {k: [] for k in legs}
    n_sites = None
    for _ in range(reps):
        for k, fn in legs.items():
            r, wall, prof = timed(fn)
            runs[k].append((wall, {kk: v[1] for kk, v in prof.items()}))
            if k == "genes_sites":
                n_sites = len(r[1])
    records, sites = eng.gene_stats(tid, start, end, strand, phase, sites=True, **params)
    res = {"slots": int(eng.n_slots), "genes": g, "gene_span_slots": span_slots, "chunks": n_chunks, "n_sites": n_sites,
           "codons": int(records["codons"].sum()), "codons_called": int(records["codons_called"].sum()),
           "snv": int((records["snv_n"] + records["snv_s"] + records["snv_m"]).sum()),
           "sub": int((records["sub_n"] + records["sub_s"] + records["sub_m"]).sum())}
    for k, v in runs.items():
        res[k] = {"call_ms": round(min(r[0] for r in v) * 1e3, 3), "all_call_ms": [round(r[0] * 1e3, 3) for r in v]}
        for name in v[0][1]:
            res[k][name + "_ms"] = round(min(r[1][name] for r in v), 4)
    kern = res["genes_sites"]["k_gene_chunks_ms"]
    model = 17 * span_slots + 112 * n_chunks
    res["k_gene_chunks_model_bytes"] = model
    res["k_gene_chunks_hbm_share"] = round(model / HBM_PEAK / (kern * 1e-3), 4)
    res["k_allele_chunks_hbm_share"] = round(17 * span_slots / HBM_PEAK / (res["allele_stats"]["k_allele_chunks_ms"] * 1e-3), 4)
    refs = [fa.fetch(n.split()[0]) for n in af.references]
    t_host, n_host = host_route(eng, genes, refs, params, host_copy_only)
    res["host_route_s" if not host_copy_only else "host_copy_only_s"] = round(t_host, 2)
    if not host_copy_only:
        assert n_host == n_sites, (n_host, n_sites)
    af.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--coverage", type=float, default=30.0)
    ap.add_argument("--c2-scale", type=float, default=0.2)
    ap.add_argument("--c3-scale", type=float, default=0.1)
    ap.add_argument("--skip", default="", help="comma-separated workloads to leave out")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from metacov_b200 import synth
    if not torch.cuda.is_available():
        sys.exit("bench_genes: no CUDA device (the gene kernels have no CPU path)")
    d = tempfile.mkdtemp()
    out = {"bench": "genes", "card": card(), "reps": args.reps}
    skip = set(filter(None, args.skip.split(",")))
    work = [("dense_c2", synth.c2(args.c2_scale).contig_len, False),
            ("dense_c3", synth.c3(args.c3_scale).contig_len, True)]
    for name, lengths, copy_only in work:
        if name in skip:
            continue
        t = time.perf_counter()
        pb, pf, n = write_workload(d, name, lengths, args.coverage, 7)
        w = time.perf_counter() - t
        r = bench_one(pb, pf, args.reps, copy_only)
        r.update({"reads": n, "coverage": args.coverage, "write_s": round(w, 1)})
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
