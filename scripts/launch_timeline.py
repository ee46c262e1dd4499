"""Where a step of the C3 workload (bench.py's default) goes between kernels: torch.profiler with CUDA activities over a
few steps of the same pool bench.py times (same graph, chains, seeds and warm-up).

Per step it reports the summed durations of the sweep2 kernels, of the small kernels between them (log q refresh, the
next-base initialiser where a build has one, the eta publish, anything else), and the idle time between consecutive
kernels (start of one minus end of the one before; negative where programmatic dependent launch lets two overlap).
One JSON line on stdout.

    python scripts/launch_timeline.py [--steps 3] [--warmup 5]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def kind(name):
    if "sweep2_kernel" in name:
        return "sweep2"
    for k in ("sweep2_preinit", "logq_refresh", "eta_publish"):
        if k in name:
            return k
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=1000000)
    ap.add_argument("--edges", type=int, default=10000000)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--sweeps-per-step", type=int, default=4)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    pkg = importlib.import_module("bipartitesbm-mcmc_b200")
    bench = importlib.import_module("bench")
    host = pkg.host
    na = nb = args.nodes // 2
    n = na + nb
    edges = bench.planted(na, nb, args.k, args.k, args.edges, 0)
    graph = host.Graph(edges, na, nb, device=0)
    pool = host.ChainPool(graph, np.tile(bench.planted_labels(na, nb, args.k, args.k), (args.chains, 1)), args.k, args.k, 1.0)
    seeds = pkg.dist.chain_seeds(0, pkg.dist.shard_chains(args.chains, 0, 1))
    pool.randomize(seeds)
    duration = args.sweeps_per_step * n
    for _ in range(args.warmup):
        pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
    torch.cuda.synchronize()
    sweep_launches = 0
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
            sweep_launches += pool.sweep_launches()
        torch.cuda.synchronize()
    fd, path = tempfile.mkstemp(suffix=".json")
    os.close(fd)
    prof.export_chrome_trace(path)
    ev = json.load(open(path))
    os.unlink(path)
    ev = ev["traceEvents"] if isinstance(ev, dict) else ev
    ks = sorted(((float(e["ts"]), float(e["dur"]), e["name"]) for e in ev if e.get("cat") == "kernel"), key=lambda x: x[0])
    dur = {}
    for _, d, name in ks:
        dur[kind(name)] = dur.get(kind(name), 0.0) + d
    gaps = [ks[i + 1][0] - (ks[i][0] + ks[i][1]) for i in range(len(ks) - 1)]
    span = ks[-1][0] + ks[-1][1] - ks[0][0]
    s = args.steps
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
    except Exception:
        gpu = None
    line = {"gpu": gpu, "steps": s, "kernels_per_step": len(ks) / s, "sweep2_launches_per_step": sweep_launches / s,
            "span_ms_per_step": span / s / 1e3,
            "kernel_ms_per_step": {k: v / s / 1e3 for k, v in sorted(dur.items())},
            "idle_ms_per_step": sum(g for g in gaps if g > 0) / s / 1e3,
            "overlap_ms_per_step": -sum(g for g in gaps if g < 0) / s / 1e3,
            "gap_us": {"median": float(np.median(gaps)), "p10": float(np.percentile(gaps, 10)), "p90": float(np.percentile(gaps, 90))},
            "sweep2_us_per_launch": dur.get("sweep2", 0.0) / max(1, sweep_launches)}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
