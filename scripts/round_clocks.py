"""Where a warp of the staged sweep kernel spends its rounds, on the C3 shape (bench.py's default workload).

Needs a library built with the round clocks compiled in:
    scripts/build_variant.sh rc -DBISBM_ROUND_CLOCKS
    BISBM_LIB=build/variants/libbisbm_rc.so python scripts/round_clocks.py

Every warp that takes vertices sums clock64 cycles over five phases: proposal + pass, dS / accept, commit, the wait for the
round's reads and the wait for its commits, at the two named barriers of a round (sweep2.cuh, BISBM_ROUND_CLOCKS).  Printed: each phase's share of warp time,
and the mean and max cycles of one vertex's proposal + pass.  Per CTA (thread 0) the build also sums the prologue (kernel
start -> first round: staging, tables, the first vertex batch, and under programmatic dependent launch the wait for the
launch before) and the epilogue (last round -> publish done), printed as mean cycles per CTA and, at the SM clock
nvidia-smi reports, microseconds.  One JSON line on stdout.
"""
import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PHASES = ["proposal+pass", "dS/accept", "commit", "wait_reads", "wait_commits"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=1000000)
    ap.add_argument("--edges", type=int, default=10000000)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--sweeps", type=int, default=8, help="measured sweeps (after as many warm-up sweeps)")
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"])
    args = ap.parse_args()
    lib_path = os.environ.get("BISBM_LIB")
    if not lib_path:
        raise SystemExit("set BISBM_LIB to a build with -DBISBM_ROUND_CLOCKS (scripts/build_variant.sh)")
    pkg = importlib.import_module("bipartitesbm-mcmc_b200")
    bench = importlib.import_module("bench")
    L = pkg.host.load_library()
    if not hasattr(L, "bisbm_round_clocks"):
        raise SystemExit("%s has no round clocks: build it with -DBISBM_ROUND_CLOCKS" % lib_path)
    L.bisbm_round_clocks.restype = ctypes.c_int
    L.bisbm_round_clocks.argtypes = [ctypes.POINTER(ctypes.c_ulonglong)]

    na = nb = args.nodes // 2
    n = na + nb
    ka = kb = args.k
    edges = bench.planted(na, nb, ka, kb, args.edges, 0)
    graph = pkg.host.Graph(edges, na, nb, device=0)
    base = bench.planted_labels(na, nb, ka, kb)
    pool = pkg.host.ChainPool(graph, np.tile(base, (args.chains, 1)).astype(np.uint32), ka, kb, 1.0)
    pool.set_precision(args.precision)
    seeds = pkg.dist.chain_seeds(0, np.arange(args.chains))
    pool.randomize(seeds)
    out = (ctypes.c_ulonglong * 11)()
    pool.anneal("constant", 1.0, 0.0, args.sweeps * n, 10 ** 18, seeds)       # warm-up: the chains leave their random start
    if L.bisbm_round_clocks(out) != 0:
        raise SystemExit(L.bisbm_last_error().decode())
    acc, _ = pool.anneal("constant", 1.0, 0.0, args.sweeps * n, 10 ** 18, seeds)
    ms, _, moves = pool.last_timing()
    if L.bisbm_round_clocks(out) != 0:
        raise SystemExit(L.bisbm_last_error().decode())
    c = [int(x) for x in out]
    total = sum(c[:5])
    shares = {p: c[i] / total for i, p in enumerate(PHASES)}
    line = {"lib": os.path.basename(lib_path), "precision": args.precision,
            "sweeps": args.sweeps, "moves_per_s_instrumented": moves / (ms * 1e-3), "acceptance": float(np.mean(acc)),
            "share": shares, "wait_share": shares["wait_reads"] + shares["wait_commits"],
            "pass_cycles_mean": c[0] / max(1, c[5]), "pass_cycles_max": c[6], "vertices": c[5], "warp_rounds": c[7],
            "cycles_per_warp_round": total / max(1, c[7])}
    try:
        mhz = float(subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=20).stdout.split()[0])
    except Exception:
        mhz = None
    ctas = max(1, c[10])
    line["per_cta"] = {"ctas": c[10], "prologue_cycles": c[8] / ctas, "epilogue_cycles": c[9] / ctas, "sm_mhz": mhz,
                       "prologue_us": c[8] / ctas / mhz if mhz else None, "epilogue_us": c[9] / ctas / mhz if mhz else None,
                       "sweep_launches": pool.sweep_launches()}
    print("per CTA: prologue %.0f cycles, epilogue %.0f cycles" % (c[8] / ctas, c[9] / ctas), file=sys.stderr)
    for p in PHASES:
        print("%-14s %6.2f %%" % (p, 100 * shares[p]), file=sys.stderr)
    print("proposal+pass per vertex: mean %.0f cycles, max %d" % (line["pass_cycles_mean"], c[6]), file=sys.stderr)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
