"""Cost of label alignment of the marginals (bisbm_marginals_align) on the C3 shape (1M nodes / 10M edges, planted 32 + 32,
Ka = Kb = 32, 256 chains) and the scaled C5 shape (5M nodes / 100M edges, Ka = Kb = 128, 32 chains), chains from
randomised starts, the planted partition as the reference.  Prints one JSON line per shape:

  kernel_us.overlap / .assign / .hist   mean kernel time per aligned sample of align_overlap_kernel, align_assign_kernel and
                                        the mapped marginal_kernel; .hist_unaligned: marginal_kernel without a reference
                                        (torch.profiler, CUDA activities, in runs of their own after the timed arms)
  overlap_GBps                          the label bytes the overlap pass must read (n x chains x label size) / its time
  moves_per_s.aligned / .unaligned      vertex moves per second of bisbm_marginalize sampling every `--every` sweeps, with and
                                        without the reference (device events of the library, arms alternated, `--reps` each)
  ratio                                 aligned / unaligned
  gpu                                   name and power limit of the card it ran on (read in the same call)

    python scripts/align_bench.py [--shapes c3 c5] [--sweeps 20] [--every 10] [--reps 3] [--out FILE]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"c3": (1000000, 10000000, 32, 256), "c5": (5000000, 100000000, 128, 32)}   # nodes, edges, K per type, chains


def kernel_us(torch, pool, n_samples, names):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_samples):
            pool.marginal_sample()
        torch.cuda.synchronize()
    us = {}
    for e in prof.key_averages():
        for key, name in names:
            if name in e.key:
                us[key] = us.get(key, 0.0) + (getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)) / n_samples
    return us


def run_shape(torch, host, shape, args):
    from bench import planted, planted_labels          # the generator of the C3 / C5 workloads
    nodes, n_edges, k, C = SHAPES[shape]
    na = nb = nodes // 2
    n = na + nb
    ref = planted_labels(na, nb, k, k)
    graph = host.Graph(planted(na, nb, k, k, n_edges, 0), na, nb)
    pool = host.ChainPool(graph, np.broadcast_to(ref, (C, n)), k, k, 1.0)
    seeds = np.arange(C, dtype=np.uint64) + 1
    pool.randomize(seeds)
    pool.marginals_clear()
    pool.marginalize(0, args.every, args.every, seeds)                 # warm-up of both arms
    pool.marginals_align(ref)
    pool.marginalize(0, args.every, args.every, seeds)
    rate = {"aligned": [], "unaligned": []}
    for _ in range(args.reps):
        for arm in ("unaligned", "aligned"):
            pool.marginals_align(ref if arm == "aligned" else None)
            pool.marginalize(0, args.sweeps, args.every, seeds)
            ms, _, moves = pool.last_timing()
            rate[arm].append(moves / ms * 1e3)
    pool.marginals_align(ref)
    us = kernel_us(torch, pool, 20, (("overlap", "align_overlap_kernel"), ("assign", "align_assign_kernel"), ("hist", "marginal_kernel")))
    pool.marginals_align(None)
    us["hist_unaligned"] = kernel_us(torch, pool, 20, (("hist", "marginal_kernel"),))["hist"]
    label_bytes = 1 if k <= 256 else 4
    ma, mu = float(np.median(rate["aligned"])), float(np.median(rate["unaligned"]))
    return {"workload": "%s: planted SBM %d nodes / %d edges, Ka=Kb=%d, %d chains from randomised starts, reference = planted "
                        "partition, bisbm_marginalize %d sweeps per call sampling every %d" % (shape, n, n_edges, k, C, args.sweeps, args.every),
            "kernel_us": {key: round(v, 2) for key, v in us.items()},
            "overlap_GBps": round(n * C * label_bytes / (us["overlap"] * 1e-6) / 1e9, 1),
            "moves_per_s": {"aligned": ma, "unaligned": mu, "samples": rate},
            "ratio": ma / mu,
            "kernel": pool.sweep_info()[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=["c3", "c5"], choices=sorted(SHAPES))
    ap.add_argument("--sweeps", type=int, default=20, help="sweeps per timed bisbm_marginalize call")
    ap.add_argument("--every", type=int, default=10, help="sweeps between two samples")
    ap.add_argument("--reps", type=int, default=3, help="timed calls per arm, alternated")
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("align_bench.py needs a CUDA device: libbisbm has no CPU path")
    host = importlib.import_module("bipartitesbm-mcmc_b200").host
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().split("\n")[0]
    lines = []
    for shape in args.shapes:
        res = run_shape(torch, host, shape, args)
        res["gpu"] = gpu
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
