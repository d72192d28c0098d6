"""Where the time of k_stats_stream goes, CTA by CTA.

Builds a copy of the library with -DMCOV_SS_PROBE (k_stats_stream.cuh: consumer thread 0 of every CTA keeps clock64
cycles per phase of its serial chain -- stage wait, accumulation, piece end of whole and of split pieces, wait for
the walker warp to free the other histogram: `walk`), runs
the statistics of whole-contig regions after a fused pass, the way bench.py does, and prints per workload one JSON
line: mean and maximum over the CTAs of each phase, the phases of the longest CTA, and the event-timed kernel.

    python tools/probe_stats_chain.py [--work DIR] [--workloads c2:1,c4:0.1] [--steps 5]

The library is built under --work (default tools/bin/probe, ignored by git) and reused while it is newer than the
sources; the product build is not touched.
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import glob
import importlib.util
import json
import os
import shutil
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PHASES = ["wait", "accum", "end_whole", "end_split", "walk", "total", "pieces", "splits", "ns"]


def build(work):
    spec = importlib.util.spec_from_file_location("_mcov_build", os.path.join(ROOT, "metacov_b200", "_build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    pkg = os.path.join(work, "metacov_b200")
    lib = os.path.join(pkg, "libmetacov_b200.so")
    os.makedirs(pkg, exist_ok=True)
    for f in glob.glob(os.path.join(ROOT, "metacov_b200", "*.py")):
        shutil.copy(f, pkg)
    srcs = [os.path.join(b.CSRC, f) for f in os.listdir(b.CSRC)] + [os.path.join(b.INCLUDE, f) for f in os.listdir(b.INCLUDE)]
    if os.path.exists(lib) and all(os.path.getmtime(s) < os.path.getmtime(lib) for s in srcs):
        return work
    nvcc = b._nvcc()
    objs = []

    def one(src):
        obj = os.path.join(work, os.path.splitext(src)[0] + ".o")
        subprocess.run([nvcc] + b.NVCC_FLAGS + ["-DMCOV_SS_PROBE", "-c", os.path.join(b.CSRC, src), "-o", obj], check=True)
        return obj

    with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        objs = list(ex.map(one, b.CUDA_SOURCES + b.CXX_SOURCES))
    subprocess.run([nvcc, "-shared", "-o", lib] + objs + ["-lz", "-gencode", "arch=compute_100a,code=sm_100a"], check=True)
    return work


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception:
        return None


def probe(name, scale, steps):
    import torch
    from metacov_b200 import CoverageEngine, synth, _capi
    lib = _capi.lib
    lib.mcov_ss_probe.restype = C.c_int
    lib.mcov_ss_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    w = synth.WORKLOADS[name](scale)
    dbatch, _ = synth.generate_device(w, 0)
    lengths = w.contig_len
    tid = np.arange(len(lengths), dtype=np.int32)
    start = np.zeros_like(tid)
    end = lengths.astype(np.int32)
    rows, ev = [], []
    with CoverageEngine(lengths, device=0) as eng:
        def step():
            eng.depth_sorted(dbatch, wait=False)
            return eng.region_stats(tid, start, end)
        for _ in range(3):                 # plan, then passes that count the histograms of the plan
            step()
        for _ in range(steps):
            grid = lib.mcov_ss_probe(eng._ctx, None, 0, 1)
            eng.profile(True)
            step()
            kt = eng.profile_read()
            eng.profile(False)
            buf = np.zeros((grid, len(PHASES)), dtype=np.uint64)
            lib.mcov_ss_probe(eng._ctx, buf.ctypes.data, grid, 0)
            rows.append(buf.astype(np.float64))
            n, ms = kt.get("k_stats_stream", (0, 0.0))
            ev.append(1e3 * ms / max(n, 1))
    del dbatch
    torch.cuda.empty_cache()
    a = np.stack(rows)                                   # [steps][grid][phase]
    ns_per_cyc = float(np.median(a[:, :, 8] / np.maximum(a[:, :, 5], 1)))
    us = lambda cyc: round(cyc * ns_per_cyc / 1e3, 2)
    cyc = {p: k for k, p in enumerate(PHASES)}
    timed = ["wait", "accum", "end_whole", "end_split", "walk", "total"]
    med = np.median(a, axis=0)                            # per CTA, median over the steps
    longest = int(np.argmax(med[:, cyc["total"]]))
    out = {
        "workload": "%s x %g" % (name, scale), "gpu": gpu_info(), "ctas": int(med.shape[0]), "steps": steps,
        "ns_per_cycle": round(ns_per_cyc, 4),
        "k_stats_stream_us_events": [round(x, 2) for x in ev],
        "mean_us": {p: us(med[:, cyc[p]].mean()) for p in timed},
        "max_us": {p: us(med[:, cyc[p]].max()) for p in timed},
        "pieces_mean": round(float(med[:, cyc["pieces"]].mean()), 2),
        "splits_mean": round(float(med[:, cyc["splits"]].mean()), 2),
        "longest_cta": dict({p: us(med[longest, cyc[p]]) for p in timed}, cta=longest,
                            pieces=int(med[longest, cyc["pieces"]]), splits=int(med[longest, cyc["splits"]])),
    }
    whole = med[:, cyc["pieces"]] - med[:, cyc["splits"]]
    if whole.sum() > 0:
        out["end_whole_us_per_piece"] = us(med[:, cyc["end_whole"]].sum() / whole.sum())
    if med[:, cyc["splits"]].sum() > 0:
        out["end_split_us_per_piece"] = us(med[:, cyc["end_split"]].sum() / med[:, cyc["splits"]].sum())
    out["walk_us_per_walk"] = us(med[:, cyc["walk"]].sum() / max(1.0, whole.sum() + 0.5 * med[:, cyc["splits"]].sum()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--work", default=os.path.join(ROOT, "tools", "bin", "probe"))
    ap.add_argument("--workloads", default="c2:1,c4:0.1")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--build-only", action="store_true")
    args = ap.parse_args()
    work = build(os.path.abspath(args.work))
    if args.build_only:
        print("built", work)
        return
    sys.path.insert(0, work)
    for item in args.workloads.split(","):
        name, scale = item.split(":")
        print(json.dumps(probe(name, float(scale), args.steps)), flush=True)


if __name__ == "__main__":
    main()
