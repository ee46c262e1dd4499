"""Cost of the marginals resolved by mode (bisbm_marginal_modes_set) on the C3 shape (1M nodes / 10M edges, planted 32 + 32,
Ka = Kb = 32, 256 chains from randomised starts, a short burn-in), references from mode_references.  Prints one JSON line:

  kernel_us[M]              time per sample of the mode kernels for M references (the first M of mode_references): CUDA
                            events on the handle's stream around `--samples` marginal samples with the set, minus the same
                            without it right after
  profiler_us               per-kernel mean device time per sample at M = 4 from torch.profiler (CUDA activities, a run of
                            its own): the alignment kernels (all modes together), the selection and the mode histogram
  hist_us                   marginal_kernel per sample (the histogram every sample pays anyway), from the same events
  moves_per_s.with / .without   vertex moves per second of bisbm_marginalize sampling every `--every` sweeps with a set of
                            M = 4 and without one (device events of the library, arms alternated, `--reps` each)
  gpu                       name and power limit of the card it ran on (read in the same call)

    python scripts/modes_bench.py [--ms 1 2 4 8] [--samples 50] [--sweeps 20] [--every 10] [--reps 3] [--out FILE]
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

NODES, EDGES, K, CHAINS = 1000000, 10000000, 32, 256


def samples_ms(torch, pool, n_samples):
    """device time of n_samples marginal samples on the handle's stream"""
    st = torch.cuda.ExternalStream(pool.stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(n_samples):
        pool.marginal_sample()
    e1.record(st)
    e1.synchronize()
    return e0.elapsed_time(e1)


def profiler_us(torch, pool, n_samples):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_samples):
            pool.marginal_sample()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for name in ("align_overlap_kernel", "align_assign_kernel", "modes_select_kernel", "modes_marginal_kernel",
                     "marginal_kernel"):
            if name in e.key and not (name == "marginal_kernel" and "modes_marginal_kernel" in e.key):
                t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                out[name] = round(out.get(name, 0.0) + t / n_samples, 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ms", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--samples", type=int, default=50, help="marginal samples per timed kernel window")
    ap.add_argument("--burn", type=int, default=20, help="sweeps from the randomised starts before the modes are found")
    ap.add_argument("--sweeps", type=int, default=20, help="sweeps per timed bisbm_marginalize call")
    ap.add_argument("--every", type=int, default=10, help="sweeps between two samples")
    ap.add_argument("--reps", type=int, default=3, help="timed calls per arm, alternated")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("modes_bench.py needs a CUDA device: libbisbm has no CPU path")
    host = importlib.import_module("bipartitesbm-mcmc_b200").host
    from bench import planted, planted_labels          # the generator of the C3 workload
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().split("\n")[0]
    na = nb = NODES // 2
    n = na + nb
    graph = host.Graph(planted(na, nb, K, K, EDGES, 0), na, nb)
    pool = host.ChainPool(graph, np.broadcast_to(planted_labels(na, nb, K, K), (CHAINS, n)), K, K, 1.0)
    seeds = np.arange(CHAINS, dtype=np.uint64) + 1
    pool.randomize(seeds)
    pool.marginals_clear()
    pool.marginalize(args.burn, 0, args.every, seeds)      # u8 labels current, as in every sampling run
    refs, mode_of = host.mode_references(pool)
    m_max = max(args.ms)
    if len(refs) < m_max:                                  # fewer modes than asked for: repeat references (same cost)
        refs = np.concatenate([refs] * ((m_max + len(refs) - 1) // len(refs)))
    res = {"workload": "C3: planted SBM %d nodes / %d edges, Ka=Kb=%d, %d chains from randomised starts, %d sweeps of burn-in"
                       % (n, EDGES, K, CHAINS, args.burn),
           "modes_found": int(mode_of.max()) + 1, "kernel_us": {}}
    pool.marginal_modes_set(None)
    samples_ms(torch, pool, 5)
    base = samples_ms(torch, pool, args.samples)
    res["hist_us"] = round(base / args.samples * 1e3, 2)
    for M in args.ms:
        pool.marginal_modes_set(refs[:M])
        samples_ms(torch, pool, 5)
        t = samples_ms(torch, pool, args.samples)
        pool.marginal_modes_set(None)
        t0 = samples_ms(torch, pool, args.samples)           # the histogram alone, right after: the same clocks
        res["kernel_us"][str(M)] = round((t - t0) / args.samples * 1e3, 2)
    pool.marginal_modes_set(refs[:4])
    res["profiler_us_m4"] = profiler_us(torch, pool, 20)
    counted = pool.marginal_modes()["counted"]
    res["m4_weights"] = (counted[:4] / max(int(counted.sum()), 1)).round(4).tolist()
    rate = {"with": [], "without": []}
    for arm in ("without", "with"):                             # warm-up of both arms
        pool.marginal_modes_set(refs[:4] if arm == "with" else None)
        pool.marginalize(0, args.every, args.every, seeds)
    for _ in range(args.reps):
        for arm in ("without", "with"):
            pool.marginal_modes_set(refs[:4] if arm == "with" else None)
            pool.marginalize(0, args.sweeps, args.every, seeds)
            ms, _, moves = pool.last_timing()
            rate[arm].append(moves / ms * 1e3)
    mw, mo = float(np.median(rate["with"])), float(np.median(rate["without"]))
    res["moves_per_s"] = {"with": mw, "without": mo, "samples": rate, "sweeps_per_call": args.sweeps, "every": args.every}
    res["ratio"] = mw / mo
    res["kernel"] = pool.sweep_info()[0]
    res["gpu"] = gpu
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
