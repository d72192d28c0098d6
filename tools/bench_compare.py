#!/usr/bin/env python
"""Sample comparison (metacov_b200.compare, csrc/compare.cu): the signature pass, the all-pairs region pass and the site
pass, the whole `metacov compare` call, and the host route they replace (copy_base_counts of every contig of every
file + the numpy oracle).

Workloads:
  dense_c2     C2's table at --c2-scale (0.2: 10^7 slots), 4 samples of one two_strain seed (tools/bench_alleles.py) at
               minor 0 / 0.2 / 0.5 / 1.0, 150 bp reads at --coverage, written as BAM
  dense_c3     the same over C3's table at --c3-scale (0.1: ~1.2 x 10^8 slots) at --c3-coverage (10: ~1 GB a BAM)
  sig_c3_full  C3's full table (~1.2 x 10^9 slots) with --sig-samples random signature tensors made on the device (the
               pair kernels' cost does not depend on coverage)
Kernel times are CUDA events (the engine's per-kernel profile), best of --reps alternated runs; whole contigs are the
regions.  Byte model, S samples, P pairs, n slots: signature 17 B a slot (counters in, one byte out); region pass S B a
slot when every chunk's signature bytes come from DRAM once and are served to its other pairs from L2 (the L2 bound),
2P B a slot without that reuse (the per-pair bound), plus 48 B a (chunk, pair) of partials and 48 B a record; site pass
the same reads (count) plus 16 B a site written.  The share of HBM peak is the L2-bound bytes over the kernel time at
7.7 TB/s.  dense_c2's signatures (4 x 10 MB) fit the 126 MB L2, so its pair kernels read L2 after the first pass; the
other two workloads are larger than L2.  Prints one JSON line (and writes it to --out).

  python tools/bench_compare.py [--reps 5] [--out profiles/r08_bench_compare.json]
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

from bench_alleles import two_strain  # noqa: E402
from bench_basecount import card, write_bam_fast  # noqa: E402

HBM_PEAK = 7.7e12           # B/s, HGX B200 data sheet, one GPU
PARAMS = dict(min_coverage=5, min_freq=0.05, min_count=2)
MINORS = (0.0, 0.2, 0.5, 1.0)


def n_chunks(lengths):
    return int(sum((int(l) + 8191) // 8192 for l in lengths))


def timed(eng, fn):
    eng.profile(True)
    eng.profile_read()
    t = time.perf_counter()
    r = fn()
    wall = time.perf_counter() - t
    prof = eng.profile_read()
    eng.profile(False)
    return r, wall, {k: round(v[1], 4) for k, v in prof.items()}


def pair_legs(eng, sigs, pairs, lengths, reps):
    """Region and site passes over every pair, best of reps alternated runs."""
    g = len(lengths)
    tid = np.arange(g, dtype=np.int32)
    z = np.zeros(g, np.int32)
    ln = np.asarray(lengths, np.int32)
    legs = {"regions": lambda: eng.compare_stats(sigs, pairs, tid, z, ln),
            "sites": lambda: eng.compare_sites(sigs, pairs)}
    for _ in range(2):
        for fn in legs.values():
            fn()
    runs = {k: [] for k in legs}
    out = {}
    for _ in range(reps):
        for k, fn in legs.items():
            r, wall, prof = timed(eng, fn)
            runs[k].append((sum(prof.values()), wall, prof))
            out[k] = r
    n, S, P = int(eng.n_slots), len(sigs), len(pairs)
    nc = n_chunks(lengths)
    model = {"regions": (S * n + 48 * nc * P + 48 * g * P, 2 * P * n + 48 * nc * P + 48 * g * P),
             "sites": (S * n + 16 * len(out["sites"]), 2 * P * n + 16 * len(out["sites"]))}
    res = {"n_sites": len(out["sites"])}
    for k, v in runs.items():
        kern, wall, names = min(v, key=lambda r: r[0])
        res[k] = {"kernel_ms": round(kern, 4), "call_ms": round(wall * 1e3, 3), "kernels": names,
                  "all_kernel_ms": [round(r[0], 4) for r in v], "model_bytes_l2_bound": model[k][0],
                  "model_bytes_per_pair_bound": model[k][1],
                  "hbm_share": round(model[k][0] / HBM_PEAK / (kern * 1e-3), 4),
                  "ms_at_l2_bound": round(model[k][0] / HBM_PEAK * 1e3, 4),
                  "ms_at_per_pair_bound": round(model[k][1] / HBM_PEAK * 1e3, 4)}
    return res, out["regions"]


def signature_leg(af, eng, reps):
    af.allele_signature(**PARAMS)
    best = None
    for _ in range(reps):
        _r, wall, prof = timed(eng, lambda: af.allele_signature(**PARAMS))
        kern = prof.get("k_allele_signature", 0.0)
        if best is None or kern < best[0]:
            best = (kern, wall)
    n = int(eng.n_slots)
    return {"kernel_ms": round(best[0], 4), "call_ms": round(best[1] * 1e3, 3), "model_bytes": 17 * n,
            "hbm_share": round(17 * n / HBM_PEAK / (best[0] * 1e-3), 4)}


def host_route(paths, pairs):
    """What the feature replaces: every contig's counts of every file to the host, the numpy rules, the pairs.  The
    decode and the count of each file (GPU work both routes share) are taken out of the time."""
    from metacov_b200 import AlignmentFile
    from oracle import compare as oc
    shared = 0.0
    total = time.perf_counter()
    sigs = []
    for p in paths:
        t = time.perf_counter()
        af = AlignmentFile(p, decode="gpu")
        af.count_coverage(af.references[0], 0, 1, quality_threshold=15)
        shared += time.perf_counter() - t
        eng = af._count_engine()
        sigs.append([oc.signature(eng.copy_base_counts(c), **PARAMS) for c in range(af.nreferences)])
        af.close()
    fields = ("length", "covered_a", "covered_b", "compared", "con_snp", "pop_snp")
    stats = np.zeros((len(pairs), len(sigs[0])), dtype=[(f, "<i8") for f in fields])
    for k, (a, b) in enumerate(pairs):
        for c in range(len(sigs[0])):
            r = oc.pair_region(sigs[a][c], sigs[b][c], 0, len(sigs[a][c]))
            for f in fields:
                stats[f][k, c] = r[f]
    return time.perf_counter() - total - shared, stats


def cli_call(paths, d):
    from metacov_b200.cli import main
    out, sites = os.path.join(d, "c.csv"), os.path.join(d, "s.tsv")
    args = ["compare"] + [x for p in paths for x in ("-b", p)] + ["-o", out, "--sites-out", sites]
    t = time.perf_counter()
    main.main(args=args, standalone_mode=False)
    wall = time.perf_counter() - t
    rows = sum(1 for _ in open(out)) - 1
    n_sites = sum(1 for _ in open(sites)) - 1
    return wall, rows, n_sites, out


def bench_files(name, lengths, coverage, reps, with_host, d):
    from metacov_b200 import AlignmentFile
    from metacov_b200.compare import all_pairs, compare
    t = time.perf_counter()
    paths = []
    for minor in MINORS:
        cols, _refs = two_strain(lengths, coverage, 7, minor=minor)
        p = os.path.join(d, "%s_m%g.bam" % (name, minor))
        write_bam_fast(p, lengths, *cols)
        paths.append(p)
    res = {"write_s": round(time.perf_counter() - t, 1), "reads": len(cols[0]), "coverage": coverage,
           "file_bytes": os.path.getsize(paths[0]), "samples": len(paths)}
    pairs = all_pairs(len(paths))
    sigs = []
    for k, p in enumerate(paths):
        with AlignmentFile(p, decode="gpu") as af:
            eng = af._count_engine()
            af.count_coverage(af.references[0], 0, 1)
            if k == 0:
                res["signature"] = signature_leg(af, eng, reps)
            sigs.append(af.allele_signature(**PARAMS))
            if k == len(paths) - 1:
                res["slots"] = int(eng.n_slots)
                legs, stats = pair_legs(eng, sigs, pairs, af.lengths, reps)
                res.update(legs)
    res["compared"] = int(stats["compared"].sum())
    res["con_snp"] = int(stats["con_snp"].sum())
    res["pop_snp"] = int(stats["pop_snp"].sum())
    # the whole comparison as a user runs it (decode, count and signature of every file included)
    wall, rows, n_sites, out = cli_call(paths, d)
    res["cli_compare_s"] = round(wall, 3)
    res["cli_rows"], res["cli_sites"] = rows, n_sites
    assert n_sites == res["n_sites"], (n_sites, res["n_sites"])
    whole = compare(paths, sites=False)
    assert whole.stats.tobytes() == stats.tobytes()
    if with_host:
        host_s, host_stats = host_route(paths, pairs.tolist())
        res["host_route_s"] = round(host_s, 2)
        res["host_route_equal"] = bool(host_stats.tobytes() == stats.tobytes())
        assert res["host_route_equal"]
    for p in paths:
        os.remove(p)
    return res


def bench_sig(lengths, n_samples, reps):
    import torch
    from metacov_b200 import CoverageEngine
    from metacov_b200.compare import all_pairs
    eng = CoverageEngine(lengths)
    n = int(eng.n_slots)
    gen = torch.Generator(device="cuda").manual_seed(11)
    sigs = [torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=gen) for _ in range(n_samples)]
    torch.cuda.synchronize()
    res = {"slots": n, "samples": n_samples, "pairs": n_samples * (n_samples - 1) // 2}
    legs, stats = pair_legs(eng, sigs, all_pairs(n_samples), lengths, reps)
    res.update(legs)
    res["compared"] = int(stats["compared"].sum())
    del sigs
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--coverage", type=float, default=30.0)
    ap.add_argument("--c2-scale", type=float, default=0.2)
    ap.add_argument("--c3-scale", type=float, default=0.1)
    ap.add_argument("--c3-coverage", type=float, default=10.0)
    ap.add_argument("--c3-host", action="store_true", help="also time the host route on dense_c3 (minutes)")
    ap.add_argument("--sig-samples", type=int, default=8)
    ap.add_argument("--skip", default="", help="comma-separated workloads to leave out")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from metacov_b200 import synth
    if not torch.cuda.is_available():
        sys.exit("bench_compare: no CUDA device (the compare kernels have no CPU path)")
    d = tempfile.mkdtemp()
    out = {"bench": "compare", "card": card(), "reps": args.reps, "params": PARAMS}
    skip = set(filter(None, args.skip.split(",")))
    if "dense_c2" not in skip:
        out["dense_c2"] = bench_files("dense_c2", synth.c2(args.c2_scale).contig_len, args.coverage, args.reps, True, d)
        print(json.dumps({"dense_c2": out["dense_c2"]}), file=sys.stderr, flush=True)
    if "dense_c3" not in skip:
        out["dense_c3"] = bench_files("dense_c3", synth.c3(args.c3_scale).contig_len, args.c3_coverage, args.reps,
                                      args.c3_host, d)
        print(json.dumps({"dense_c3": out["dense_c3"]}), file=sys.stderr, flush=True)
    if "sig_c3_full" not in skip:
        out["sig_c3_full"] = bench_sig(synth.c3(1.0).contig_len, args.sig_samples, args.reps)
        print(json.dumps({"sig_c3_full": out["sig_c3_full"]}), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
