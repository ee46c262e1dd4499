"""Cost of the chain agreement (bisbm_chain_agreement) beside the cost of one sweep at the same shape.  Shapes:

  c3   1M nodes / 10M edges, planted 32 + 32, Ka = Kb = 32, 256 chains from randomised starts (u8 labels)
  c5   scaled C5 of bench.py: 5M nodes / 100M edges, planted 128 + 128, Ka = Kb = 128, 32 chains, counts in L2

Per shape, one JSON object in the line printed (and written to --out):

  table_ms                  agree_table_kernel's device time per call (all chunks, both types), torch.profiler
  final_ms / final_no_overlap_ms   agree_final_kernel's device time per call with and without the matching
  call_ms / call_no_overlap_ms     host wall time of the whole call (kernels, copy-out, composing the metrics), median
  sweep_ms                  device time of one sweep of the pool (bisbm_last_timing of a one-sweep anneal), median
  table_over_sweep          table_ms / sweep_ms
  label_bytes_read          bytes the table kernels read: per (row chain, column group, pass) the type's label rows
  gpu                       name and power limit of the card it ran on (read in the same call)

    python scripts/agreement_bench.py [--shapes c3 c5] [--reps 3] [--out FILE]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"c3": (1000000, 10000000, 32, 256), "c5": (5000000, 100000000, 128, 32)}
SMEM = 232448                                     # the B200's opt-in shared memory per block


def kernel_ms(torch, fn, names):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in names}
    for e in prof.key_averages():
        for k in names:
            if k in e.key:
                out[k] += (getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)) / 1e3
    return out


def run_shape(torch, host, name, reps):
    from bench import planted, planted_labels          # the generator of the benchmark workloads
    nodes, edges, K, chains = SHAPES[name]
    na = nb = nodes // 2
    n = na + nb
    graph = host.Graph(planted(na, nb, K, K, edges, 0), na, nb)
    lab = planted_labels(na, nb, K, K).astype(np.uint8 if 2 * K <= 256 else np.uint32)
    pool = host.ChainPool(graph, np.broadcast_to(lab, (chains, n)), K, K, 1.0)
    seeds = np.arange(chains, dtype=np.uint64) + 1
    pool.randomize(seeds)
    sweep = []
    for _ in range(reps + 1):
        pool.anneal("constant", 1.0, 0.0, n, 10 ** 18, seeds)
        sweep.append(pool.last_timing()[0])
    sweep_ms = float(np.median(sweep[1:]))
    pool.chain_agreement()                                   # warm-up (module load, shared-memory attributes)
    calls = {True: [], False: []}
    for _ in range(reps):
        for ov in (True, False):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pool.chain_agreement(overlap=ov)
            calls[ov].append((time.perf_counter() - t0) * 1e3)
    k_ov = kernel_ms(torch, lambda: pool.chain_agreement(overlap=True), ["agree_table_kernel", "agree_final_kernel"])
    k_no = kernel_ms(torch, lambda: pool.chain_agreement(overlap=False), ["agree_table_kernel", "agree_final_kernel"])
    rpp = min(K, SMEM // (K * 128))
    passes = -(-K // rpp)
    groups = (chains + 31) // 32
    ctas = sum(groups - c // 32 for c in range(chains))      # (row chain, column group at or above its own)
    return {"workload": "%s: planted SBM %d nodes / %d edges, Ka=Kb=%d, %d chains from randomised starts" % (name, n, edges, K, chains),
            "kernel": pool.sweep_info()[0],
            "table_ms": round(k_ov["agree_table_kernel"], 3),
            "final_ms": round(k_ov["agree_final_kernel"], 3),
            "final_no_overlap_ms": round(k_no["agree_final_kernel"], 3),
            "call_ms": round(float(np.median(calls[True])), 3),
            "call_no_overlap_ms": round(float(np.median(calls[False])), 3),
            "sweep_ms": round(sweep_ms, 3),
            "table_over_sweep": round(k_ov["agree_table_kernel"] / sweep_ms, 3),
            "passes_per_type": passes,
            "label_bytes_read": int(ctas * passes * n * (32 + 1) * (1 if 2 * K <= 256 else 4))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=["c3", "c5"], choices=list(SHAPES))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("agreement_bench.py needs a CUDA device: libbisbm has no CPU path")
    host = importlib.import_module("bipartitesbm-mcmc_b200").host
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().split("\n")[0]
    res = {"gpu": gpu}
    for s in args.shapes:
        res[s] = run_shape(torch, host, s, args.reps)
        print(json.dumps({s: res[s]}), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
