"""Cost of parallel tempering on the C3 shape (1M nodes / 10M edges, planted 32 + 32, Ka = Kb = 32, 256 chains as 32
ladders x 8 rungs, geometric ladder 1 -> 1.5, a swap round every sweep).  Prints one JSON line:

  moves_per_s.tempering / .anneal_T1   vertex moves per second of bisbm_tempering_run and of bisbm_anneal at constant T = 1
                                       on the same pool (device events of the library, arms alternated, `--reps` each)
  ratio                                tempering / anneal
  round_us.entropy / .swap             mean kernel time per swap round of entropy_kernel and tempering_swap_kernel
                                       (torch.profiler, CUDA activities, in a separate run after the timed arms)
  swap_acceptance                      accepted / tried per adjacent rung pair
  gpu                                  name and power limit of the card it ran on

    python scripts/tempering_bench.py [--sweeps 10] [--reps 3] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=1000000)
    ap.add_argument("--edges", type=int, default=10000000)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--ladders", type=int, default=32)
    ap.add_argument("--rungs", type=int, default=8)
    ap.add_argument("--t-max", type=float, default=1.5)
    ap.add_argument("--sweeps", type=int, default=10, help="sweeps per timed call")
    ap.add_argument("--reps", type=int, default=3, help="timed calls per arm, alternated")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        raise SystemExit("tempering_bench.py needs a CUDA device: libbisbm has no CPU path")
    from bench import planted, planted_labels          # the generator of the C3 workload
    host = importlib.import_module("bipartitesbm-mcmc_b200").host
    na = nb = args.nodes // 2
    n, ka = na + nb, args.k
    C = args.ladders * args.rungs
    graph = host.Graph(planted(na, nb, ka, ka, args.edges, 0), na, nb)
    pool = host.ChainPool(graph, np.broadcast_to(planted_labels(na, nb, ka, ka), (C, n)), ka, ka, 1.0)
    seeds = np.arange(C, dtype=np.uint64) + 1
    pool.randomize(seeds)
    temps = host.geometric_ladder(1.0, args.t_max, args.rungs)
    pool.tempering_set(temps)
    pool.anneal("constant", 1.0, 0.0, 2 * n, 10 ** 18, seeds)         # warm-up of both arms
    pool.tempering_run(2, 1, seeds)
    rate = {"tempering": [], "anneal_T1": []}
    for _ in range(args.reps):
        pool.anneal("constant", 1.0, 0.0, args.sweeps * n, 10 ** 18, seeds)
        ms, _, moves = pool.last_timing()
        rate["anneal_T1"].append(moves / ms * 1e3)
        pool.tempering_run(args.sweeps, 1, seeds)
        ms, _, moves = pool.last_timing()
        rate["tempering"].append(moves / ms * 1e3)
    st = pool.tempering_stats()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pool.tempering_run(3, 1, seeds)
        torch.cuda.synchronize()
    us = {}
    for e in prof.key_averages():
        for key, name in (("entropy", "entropy_kernel"), ("swap", "tempering_swap_kernel")):
            if name in e.key:
                t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                us[key] = us.get(key, 0.0) + t / max(e.count, 1)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().split("\n")[0]
    mt, ma = float(np.median(rate["tempering"])), float(np.median(rate["anneal_T1"]))
    res = {"workload": "planted SBM %d nodes / %d edges, Ka=Kb=%d, %d chains = %d ladders x %d rungs, geometric ladder 1 -> %g, "
                       "swap round every sweep, %d sweeps per call" % (n, args.edges, ka, C, args.ladders, args.rungs, args.t_max, args.sweeps),
           "moves_per_s": {"tempering": mt, "anneal_T1": ma, "samples": rate},
           "ratio": mt / ma,
           "round_us": us,
           "swap_acceptance": (st["swaps_accepted"] / np.maximum(st["swaps_tried"], 1)).round(4).tolist(),
           "temps": [round(float(t), 6) for t in temps],
           "kernel": pool.sweep_info()[0],
           "gpu": gpu}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
