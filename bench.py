#!/usr/bin/env python
"""bench.py -- vertex-moves/sec of the Metropolis-Hastings sweep on synthetic planted bipartite SBMs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2], SURVEY.md 8(d) row C3): 1M nodes (5e5+5e5) / 10M edges,
planted 32+32, Ka=Kb=32, epsilon=1, T=1 constant, 256 batched chains per GPU with randomised
starts.  One "step" = SWEEPS_PER_STEP full sweeps of every chain (one bisbm_anneal call).
Chains are sharded over GPUs with the graph replicated (weak scaling: 256 chains per GPU).

value   = attempted single-vertex moves / s, all chains, state resident in HBM.
e2e     = the same through the C ABI with HOST buffers: every step uploads the chains' labels
          (pinned host memory), runs the sweeps and reads the labels back.
roofline= algorithmic HBM bytes per move (16 + 8*(2E/N) + 4*acceptance, SURVEY.md 8(d)) x moves
          / CUDA-event time of the sweep launches, against MEASURED_PEAKS.json hbm_gbs.
cpu_baseline / --impl reference = the UNMODIFIED reference (oracle/_ref/libref.so, built from
          the reference's sources by `make -C oracle ref`) or, if that build is absent, the oracle port,
          one chain per host core, anneal() only, on a bounded sample of the same workload.
--dump-outputs DIR (C3 workload, one process) = after the timed steps, what the last one computed, as DIR/<name>.npy
          (see dump_outputs); the inputs depend only on the arguments, so two builds can be compared output for output.
          The staged parallel sweep evaluates and commits in fixed rounds, so two runs of one build write identical
          files -- unless a block of some chain gets small enough to empty within one launch, where the order of the
          "would empty the block" veto's atomics decides (no block of the C3 workload comes near that).
"""
import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SWEEPS_PER_STEP = 4


def planted(na, nb, ka, kb, n_edges, seed, ratio=10.0):
    """SURVEY.md 8(d) generator: block of type-a node i = i*ka//na; block pair weight `ratio` on the
    paired diagonal, 1 elsewhere; uniform node within each block; multi-edges kept."""
    rng = np.random.default_rng(seed)
    w = np.ones((ka, kb))
    for r in range(ka):
        w[r, r * kb // ka] = ratio
    p = (w / w.sum()).ravel()
    pair = rng.choice(ka * kb, size=n_edges, p=p)
    r, s = pair // kb, pair % kb
    ba = np.arange(na) * ka // na
    bb = np.arange(nb) * kb // nb
    a_start = np.searchsorted(ba, np.arange(ka))
    a_cnt = np.bincount(ba, minlength=ka)
    b_start = np.searchsorted(bb, np.arange(kb))
    b_cnt = np.bincount(bb, minlength=kb)
    ea = a_start[r] + (rng.random(n_edges) * a_cnt[r]).astype(np.int64)
    eb = na + b_start[s] + (rng.random(n_edges) * b_cnt[s]).astype(np.int64)
    return np.stack([ea, eb], 1).astype(np.uint32)


def planted_chunked(na, nb, ka, kb, n_edges, seed, chunk=50_000_000):
    """The same generator in pieces of `chunk` edges (one RNG stream per piece), writing into one preallocated uint32 array:
    bounded host memory for the 10^9-edge graph of BASELINE configs[4]."""
    out = np.empty((n_edges, 2), dtype=np.uint32)
    done, k = 0, 0
    while done < n_edges:
        m = min(chunk, n_edges - done)
        out[done:done + m] = planted(na, nb, ka, kb, m, seed * 1000003 + k)
        done += m; k += 1
    return out


def planted_labels(na, nb, ka, kb):
    return np.concatenate([np.arange(na) * ka // na, ka + np.arange(nb) * kb // nb]).astype(np.uint32)


DUMP_CHAINS = 256       # --dump-outputs keeps every chain up to this many, else a seeded sample of this many
DUMP_NODES = 16384      # ... and the labels of a seeded sample of this many nodes: at most 16 MB of labels


def dump_outputs(out_dir, pool, acc, sweeps):
    """Write what one anneal() call handed back (per-chain acceptance ratio and sweeps done) and the state it left behind
    (per-chain description length, labels) as float64 / float32 .npy files.  The chains and nodes kept are a fixed sample
    (the same for every run with the same arguments), whose indices are written beside the labels."""
    rng = np.random.default_rng(0)
    C, n = pool.n_chains, pool.g.n
    chains = np.arange(C) if C <= DUMP_CHAINS else np.sort(rng.choice(C, DUMP_CHAINS, replace=False))
    nodes = np.arange(n) if n <= DUMP_NODES else np.sort(rng.choice(n, DUMP_NODES, replace=False))
    labels = pool.labels(out=np.empty((C, n), dtype=np.uint8 if pool.K(0) <= 256 else np.uint32))
    out = {"acceptance": acc[chains], "sweeps": sweeps[chains].astype(np.float64), "entropy": pool.entropy()[chains],
           "labels": labels[np.ix_(chains, nodes)].astype(np.float32), "labels_chains": chains.astype(np.float64),
           "labels_nodes": nodes.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class stdout_to_stderr:
    """file descriptor 1 points at stderr inside the block: under NCCL_DEBUG (VERSION / INFO) NCCL prints its banner to
    stdout while a communicator comes up, and stdout carries exactly ONE JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.keep = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.keep, 1)
        os.close(self.keep)
        return False


def init_nccl(local_rank):
    import torch
    import torch.distributed as dist
    with stdout_to_stderr():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()                      # the first collective creates the communicator
        torch.cuda.synchronize()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


# ------------------------------------------------------------------------------ CPU arm
_CPU_WORKER = r"""
import sys, time, numpy as np
sys.path.insert(0, sys.argv[1])
kind, path, na, nb, ka, kb, moves, seed = sys.argv[2], sys.argv[3], int(sys.argv[4]), int(sys.argv[5]), int(sys.argv[6]), int(sys.argv[7]), int(sys.argv[8]), int(sys.argv[9])
edges = np.load(path, mmap_mode="r")
n = na + nb
labels = np.concatenate([np.arange(na) * ka // na, ka + np.arange(nb) * kb // nb]).astype(np.uint32)
if kind == "reference":
    from oracle import ref as mod
    c = mod.RefChain(n, na, nb, np.asarray(edges), labels, ka, kb, 1.0, seed, 1000 + seed)
else:
    from oracle import port as mod
    c = mod.PortChain(n, na, nb, np.asarray(edges), labels, ka, kb, 1.0, seed, 1000 + seed)
c.init(True)
sweeps = max(1, moves // n)
print("READY", flush=True)
sys.stdin.readline()
t0 = time.perf_counter()
acc = c.anneal(3, 1.0, 0.0, sweeps * n, 10 ** 18)   # constant T = 1, no early stop; summary() skipped (SURVEY T4)
dt = time.perf_counter() - t0
print("DONE %d %.6f %.4f" % (sweeps * n, dt, acc), flush=True)
"""


def cpu_kind():
    from oracle import ref
    return "reference" if ref.available() else "port"


def run_cpu_sample(edges_path, na, nb, ka, kb, moves_per_proc, procs, kind):
    """One chain per core: `procs` processes each build the reference state (untimed), then all
    start anneal() together; returns aggregate moves/s over the slowest process's wall time."""
    ps = []
    for i in range(procs):
        cmd = [sys.executable, "-c", _CPU_WORKER, ROOT, kind, edges_path, str(na), str(nb), str(ka), str(kb),
               str(moves_per_proc), str(i + 1)]
        if hasattr(os, "sched_getaffinity"):
            cores = sorted(os.sched_getaffinity(0))
            cmd = ["taskset", "-c", str(cores[i % len(cores)])] + cmd
        ps.append(subprocess.Popen(cmd, stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True))
    for p in ps:
        line = p.stdout.readline()
        if not line.startswith("READY"):
            raise RuntimeError("cpu worker failed: " + line)
    for p in ps:
        p.stdin.write("go\n"); p.stdin.flush()
    moves, worst = 0, 0.0
    for p in ps:
        line = p.stdout.readline().split()
        moves += int(line[1]); worst = max(worst, float(line[2]))
        p.wait()
    return moves / worst, moves, worst


def cpu_procs(per_proc_gb):
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    avail_gb = 16.0
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                avail_gb = int(line.split()[1]) / 1e6
    except Exception:
        pass
    return max(1, min(cores, int(avail_gb * 0.5 / per_proc_gb), 64))


# ------------------------------------------------------------------------------ BASELINE configs[3]
C4_VALUES = (2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64)


def bench_c4(args, rank, world, local_rank):
    """(Ka, Kb) in C4_VALUES^2 x 8 restarts = 968 chains on the C3 graph (SURVEY.md 8(d) row C4, throughput subset),
    abrupt_cool annealing, through bisbm_grid_search; grid points are dealt round-robin to the GPUs."""
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("bipartitesbm-mcmc_b200")
    host = pkg.host
    torch.cuda.set_device(local_rank)
    if world > 1:
        init_nccl(local_rank)
    na = nb = args.nodes // 2
    n = na + nb
    edges = planted(na, nb, args.k, args.k, args.edges, 0)
    graph = host.Graph(edges, na, nb, device=local_rank)
    points = [(a, b) for a in C4_VALUES for b in C4_VALUES]
    restarts = 8
    # whole 32-chain groups of one K bucket per rank, buckets balanced by cost (host.grid_partition)
    mine = [points[i] for i in host.grid_partition(graph, points, restarts, world)[rank]]
    sweeps = args.sweeps_per_step
    hot = max(1, sweeps // 2)

    def step(seed):
        return host.grid_search(graph, mine, restarts, 1.0, "abrupt_cool", float(hot * n), 0.0, sweeps * n, 10 ** 18, seed=seed)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(args.warmup):
        step(100 + i)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    moves, dev_ms, best = 0.0, 0.0, (float("inf"), None)
    for i in range(args.steps):
        ent, acc, bi, lab, st = step(i + 1)
        moves += st["moves"]; dev_ms += st["device_ms"]; last_report = st["report"]
        if ent.min() < best[0]:
            best = (float(ent.min()), mine[bi[0]])
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    t = torch.tensor([wall, dev_ms], dtype=torch.float64, device="cuda")
    tmin = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([moves], dtype=torch.float64, device="cuda")
    be = torch.tensor([best[0], float(best[1][0]), float(best[1][1])], dtype=torch.float64, device="cuda")
    gathered = [be]
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        gathered = [torch.zeros_like(be) for _ in range(world)]
        dist.all_gather(gathered, be)           # the best partition's score and (Ka, Kb) of every rank
    if rank == 0:
        g = min((x.tolist() for x in gathered), key=lambda x: x[0])
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        bytes_per_move = 16.0 + 8.0 * (2.0 * args.edges / n) + 4.0 * 0.5
        achieved = bytes_per_move * float(tot[0]) / world / (float(t[1]) * 1e-3) / 1e9
        line = {"metric": "vertex-moves/sec", "value": float(tot[0]) / float(t[0]), "unit": "moves/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(t[0]) / args.steps * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64+int32", "data": "synthetic",
                "config": {"workload": "C4: (Ka,Kb) in %s^2 x %d restarts = %d chains on the planted SBM %d nodes / %d edges, abrupt_cool (%d hot + %d greedy sweeps per step), bisbm_grid_search, grid points dealt in whole 32-chain groups per K bucket over %d GPU(s)" % (
                    list(C4_VALUES), restarts, len(points) * restarts, n, args.edges, hot, sweeps - hot, world),
                    "l2": "inputs larger than L2", "k_buckets": "max(Ka,Kb) <= 32: padded to 8/16/32 (staged counts); larger: asymmetric strides that fit shared memory stay staged (64 x 16, 48 x 24 and transposes), the rest (12 of 121 points) padded to 64 x 64 with counts in L2"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                             "bytes_per_move": bytes_per_move, "note": "per-GPU algorithmic bytes over the slowest rank's device time"},
                "imbalance": {"device_ms_max": float(t[1]), "device_ms_min": float(tmin[0]), "max_over_min": float(t[1]) / max(float(tmin[0]), 1e-9)},
                "best": {"entropy": g[0], "ka": int(g[1]), "kb": int(g[2]), "planted": [args.k, args.k]},
                "buckets_rank0_last_step": last_report,
                "e2e": {"value": float(tot[0]) / float(t[0]), "unit": "moves/s", "h2d_bytes_per_step": 8 * len(mine), "d2h_bytes_per_step": 8 * len(mine) * restarts * 2 + 4 * n,
                        "api": "bisbm_grid_search: (Ka,Kb) list in, per-chain entropy + best labels out, every step (value is already end to end)"},
                "gpu_launches": None, "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def bench_c5(args, rank, world, local_rank):
    """BASELINE configs[4] scaled to what one GPU's share looks like: planted SBM with Ka = Kb = 128 (counts in L2: the
    staged kernel cannot hold 128 x 128 x 32 counters), --c5-nodes / --c5-edges (default 5M / 100M = 1/10 of the named
    50M / 1B), 32 chains per GPU, T = 1; every GPU runs its own chains over the replicated graph and the per-node marginal
    histograms (N x 256 x 4 B) are summed by the library's NCCL all-reduce, timed separately.  The reference cannot run
    this shape (k_ alone is N x 256 x 4 B per chain plus adj_map_): its number comes from a 1/50-scale graph."""
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("bipartitesbm-mcmc_b200")
    host = pkg.host
    torch.cuda.set_device(local_rank)
    if world > 1:
        init_nccl(local_rank)
    na = nb = args.c5_nodes // 2
    n = na + nb
    K = 128
    C = args.c5_chains
    t_gen = time.perf_counter()
    edges = planted(na, nb, K, K, args.c5_edges, 0) if args.c5_edges <= 200_000_000 else planted_chunked(na, nb, K, K, args.c5_edges, 0)
    t_gen = time.perf_counter() - t_gen
    t_build = time.perf_counter()
    graph = host.Graph(edges, na, nb, device=local_rank)
    t_build = time.perf_counter() - t_build
    lab = planted_labels(na, nb, K, K).astype(np.uint8 if 2 * K <= 256 else np.uint32)
    pool = host.ChainPool(graph, np.broadcast_to(lab, (C, n)), K, K, 1.0)
    seeds = pkg.dist.chain_seeds(0, pkg.dist.shard_chains(C * world, rank, world))
    pool.randomize(seeds)
    if world > 1:
        with stdout_to_stderr():
            pkg.dist.init_pool_comm(pool)
    sweeps = args.sweeps_per_step
    for _ in range(args.warmup):
        pool.anneal("constant", 1.0, 0.0, 1 * n, 10 ** 18, seeds)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    dev_ms, moves, accs = 0.0, 0, []
    for _ in range(args.steps):
        acc, _sw = pool.anneal("constant", 1.0, 0.0, sweeps * n, 10 ** 18, seeds)
        ms_, _la, mv_ = pool.last_timing()
        dev_ms += ms_; moves += mv_; accs.append(float(acc.mean()))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    # size-independent properties on one chain: the device counts equal a rebuild from its labels
    l0 = pool.labels(C - 1).astype(np.int64)
    ea, eb = edges[:, 0].astype(np.int64), edges[:, 1].astype(np.int64)
    m_ab = np.bincount(l0[ea] * K + (l0[eb] - K), minlength=K * K).reshape(K, K)
    m_dev = pool.m(C - 1)[:K, K:]
    ok = bool((m_dev == m_ab).all() and (pool.n_r(C - 1) == np.bincount(l0, minlength=2 * K)).all())
    # the one collective: histogram all-reduce
    pool.marginals_clear()
    pool.marginal_sample()
    torch.cuda.synchronize()
    ar_ms = None
    if world > 1:
        pool.marginals_allreduce()          # warm: the first collective of a communicator sets up its channels
        torch.cuda.synchronize()
        dist.barrier()
        t1 = time.perf_counter()
        pool.marginals_allreduce()
        torch.cuda.synchronize()
        ar_ms = (time.perf_counter() - t1) * 1e3
    kern, wpc_, cpg_, slice_ = pool.sweep_info()
    t = torch.tensor([wall, dev_ms, ar_ms or 0.0], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(moves)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        bytes_per_move = 16.0 + 8.0 * (2.0 * args.c5_edges / n) + 4.0 * float(np.mean(accs))
        achieved = bytes_per_move * float(tot[0]) / world / (float(t[1]) * 1e-3) / 1e9
        hist_bytes = n * 2 * K * 4
        line = {"metric": "vertex-moves/sec", "value": float(tot[0]) / float(t[0]), "unit": "moves/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": float(t[0]) / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64+int32", "data": "synthetic",
                "config": {"workload": "C5 scaled: planted SBM %d nodes / %d edges, Ka=Kb=128, %d chains/GPU, T=1 (BASELINE configs[4] names 50M / 1B on 8 GPUs)" % (n, args.c5_edges, C),
                           "l2": "inputs larger than L2", "sweep_plan": {"kernel": kern, "warps_per_cta": wpc_, "ctas_per_chain_group": cpg_, "slice": slice_},
                           "graph_generate_s": t_gen, "graph_build_s": t_build},
                "acceptance": float(np.mean(accs)), "invariants_ok": ok,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                             "bytes_per_move": bytes_per_move, "kernel": "sweep2_kernel<double, counts in L2>"},
                "allreduce": {"bytes": hist_bytes, "ms": float(t[2]) if world > 1 else None,
                              "GBps_bus": (2.0 * (world - 1) / world * hist_bytes / (float(t[2]) * 1e-3) / 1e9) if world > 1 and float(t[2]) > 0 else None},
                "e2e": {"value": float(tot[0]) / float(t[0]), "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": None}
        if not args.no_cpu_baseline and world == 1:
            try:
                sna = snb = max(1000, args.c5_nodes // 10) // 2       # 1/50 of the NAMED 50M-node graph when c5_nodes is 5M
                sedges = planted(sna, snb, K, K, max(1000, args.c5_edges // 10), 0)
                path = os.path.join(tempfile.gettempdir(), "bisbm_bench_edges_c5_%d.npy" % os.getpid())
                np.save(path, sedges)
                kind = cpu_kind()
                procs = max(1, min(cpu_procs(6.0), 8))
                v, mv, worst = run_cpu_sample(path, sna, snb, K, K, max(100000, args.cpu_moves // 4), procs, kind)
                os.unlink(path)
                line["cpu_baseline"] = {"value": v, "unit": "moves/s", "cores": procs, "kind": kind,
                                        "sample": "reference infeasible at the named size (k_ = N x 256 x 4 B per chain); measured on a 1/50-scale graph (%d nodes / %d edges, same mean degree and K): %d processes x %d moves of anneal() (T=1), %.1f s" % (
                                            sna + snb, len(sedges), procs, mv // procs, worst)}
            except Exception as ex:
                line["cpu_baseline"] = {"value": None, "unit": "moves/s", "cores": 0, "kind": "unavailable", "sample": str(ex)[:200]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def bench_marginalize(args, rank, world, local_rank):
    """BASELINE configs[1] wording (burn-in, then sample every 10 sweeps) on the C3 graph: sweeps + histogram accumulation,
    and the marginal kernel alone against its N x chains x 12 B per sample roofline (SURVEY.md 8(d))."""
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("bipartitesbm-mcmc_b200")
    host = pkg.host
    torch.cuda.set_device(local_rank)
    if world > 1:
        init_nccl(local_rank)
    na = nb = args.nodes // 2
    n = na + nb
    ka = kb = args.k
    C = args.chains
    edges = planted(na, nb, ka, kb, args.edges, 0)
    graph = host.Graph(edges, na, nb, device=local_rank)
    pool = host.ChainPool(graph, np.broadcast_to(planted_labels(na, nb, ka, kb), (C, n)), ka, kb, 1.0)
    seeds = pkg.dist.chain_seeds(0, pkg.dist.shard_chains(C * world, rank, world))
    every, samples = 10, max(1, args.sweeps_per_step // 2)
    if world > 1:
        with stdout_to_stderr():
            pkg.dist.init_pool_comm(pool)
    pool.marginals_clear()
    for _ in range(args.warmup):
        pool.marginalize(0, every, every, seeds)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    dev_ms, moves = 0.0, 0
    for _ in range(args.steps):
        pool.marginalize(0, every * samples, every, seeds)
        ms_, _la, mv_ = pool.last_timing()
        dev_ms += ms_; moves += mv_
    if world > 1:
        pkg.dist.allreduce_marginals(pool)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    # the marginal kernel alone: samples of the resident labels back to back
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.ExternalStream(pool.stream())
    reps = 20
    with torch.cuda.stream(stream):
        pool.marginal_sample()
        ev0.record(stream)
        for _ in range(reps):
            pool.marginal_sample()
        ev1.record(stream)
    torch.cuda.synchronize()
    k_ms = ev0.elapsed_time(ev1) / reps
    t = torch.tensor([wall], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(moves)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        alg = 12.0 * n * C            # SURVEY.md 8(d): per sample N x (4 B label read + 8 B histogram read-modify-write) per chain
        line = {"metric": "vertex-moves/sec", "value": float(tot[0]) / float(t[0]), "unit": "moves/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": float(t[0]) / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64+int32", "data": "synthetic",
                "config": {"workload": "marginalization on the planted SBM %d nodes / %d edges, Ka=Kb=%d, %d chains/GPU from the planted partition, T=1, one sample into the per-node label histogram every %d sweeps, %d samples per step" % (n, args.edges, ka, C, every, samples),
                           "l2": "inputs larger than L2"},
                "roofline": {"bound": "hbm", "kernel": "marginal_kernel<u8>", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": alg / (k_ms * 1e-3) / 1e9 / peak, "traffic": None, "alg_bytes_per_launch": alg, "avg_launch_ms": k_ms,
                             "note": "algorithmic bytes per sample = N x chains x 12 B (SURVEY.md 8(d)); the kernel reads 1 B per label from the u8 shadow and adds once per distinct label of a 32-chain group, so its real traffic is below that"},
                "marginal_share_of_step": k_ms * samples * args.steps / max(dev_ms, 1e-9),
                "e2e": {"value": float(tot[0]) / float(t[0]), "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                        "api": "bisbm_marginalize (histogram stays on the device; all-reduced once at the end when N > 1)"},
                "gpu_launches": None}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nodes", type=int, default=1000000)
    ap.add_argument("--edges", type=int, default=10000000)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--chains", type=int, default=256, help="chains per GPU")
    ap.add_argument("--sweeps-per-step", type=int, default=SWEEPS_PER_STEP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-moves", type=int, default=2000000, help="CPU sample: moves per process per step")
    ap.add_argument("--workload", default="c3", choices=["c3", "c4", "c5", "marginalize"],
                    help="c3: BASELINE configs[2] (headline); c4: configs[3], the (Ka,Kb) grid x 8 restarts through the in-process "
                         "search driver, points sharded over the GPUs; marginalize: configs[1] wording on the C3 graph "
                         "(sample every 10 sweeps into the device histogram)")
    ap.add_argument("--c5-nodes", type=int, default=5000000)
    ap.add_argument("--c5-edges", type=int, default=100000000)
    ap.add_argument("--c5-chains", type=int, default=32)
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"],
                    help="arithmetic of a move: fp64 like the reference's transition_ratio (headline) or fp32")
    ap.add_argument("--inflight-div", type=int, default=0, help="in-flight bound = half sweep / this (0: library default)")
    ap.add_argument("--warps", type=int, default=0, help="experiment builds only: warps per CTA (20, 24)")
    ap.add_argument("--no-spare-sms", action="store_true", help="A/B: leave the SMs that groups x CTAs do not fill idle")
    ap.add_argument("--no-fp32-extra", action="store_true", help="skip the short fp32 run reported under 'extra'")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="C3 workload: write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, < 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c3"):
        ap.error("--dump-outputs is implemented for the C3 workload of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:     # several ranks time one more sweep after the steps (the marginal all-reduce)
        ap.error("--dump-outputs is implemented for one process")
    na = nb = args.nodes // 2
    n = na + nb
    ka = kb = args.k
    workload = "planted bipartite SBM %d nodes / %d edges, Ka=Kb=%d, %d chains/GPU, T=1, eps=1" % (n, args.edges, ka, args.chains)
    config = {"workload": workload, "sweeps_per_step": args.sweeps_per_step, "chains_per_gpu": args.chains,
              "l2": "inputs larger than L2 (labels %.0f MB as gathered u8, CSR %.0f MB per GPU)" % (n * args.chains / 1e6,
                                                                                      args.edges * 8 / 1e6),
              "parallelism": "chains sharded over %d GPU(s), graph replicated" % world}

    # ---------------- reference arm: the reference's own CPU implementation on the host cores
    if args.impl == "reference":
        if rank != 0:
            return 0
        edges = planted(na, nb, ka, kb, args.edges, 0)
        path = os.path.join(tempfile.gettempdir(), "bisbm_bench_edges_%d.npy" % os.getpid())
        np.save(path, edges)
        kind = cpu_kind()
        procs = cpu_procs(3.5 if kind == "reference" else 1.5)
        vals = []
        for i in range(args.warmup + args.steps):
            # every step is a fresh bounded sample (state build untimed, anneal timed)
            v, moves, worst = run_cpu_sample(path, na, nb, ka, kb, args.cpu_moves, procs, kind)
            if i >= args.warmup:
                vals.append((v, moves, worst))
            if i == 0 and args.warmup > 1:
                pass
        os.unlink(path)
        value = float(np.mean([v for v, _, _ in vals]))
        ms = float(np.mean([w for _, _, w in vals])) * 1e3
        sample = "%d processes x %d moves of anneal() (T=1) on the full %d-node / %d-edge graph, every step from a fresh randomised start (chain phase: first sweeps, acceptance ~0.93), state build untimed" % (
            procs, vals[0][1] // procs, n, args.edges)
        line = {"impl": "reference", "metric": "vertex-moves/sec", "value": value, "unit": "moves/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64+int32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": "moves/s", "cores": procs, "kind": kind, "sample": sample},
                "e2e": {"value": value, "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    if args.workload == "c4":
        return bench_c4(args, rank, world, local_rank)
    if args.workload == "marginalize":
        return bench_marginalize(args, rank, world, local_rank)
    if args.workload == "c5":
        return bench_c5(args, rank, world, local_rank)

    # ---------------- our arm
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("bipartitesbm-mcmc_b200")
    host = pkg.host
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libbisbm has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        init_nccl(local_rank)
    edges = planted(na, nb, ka, kb, args.edges, 0)
    graph = host.Graph(edges, na, nb, device=local_rank)
    C = args.chains
    chain_ids = pkg.dist.shard_chains(C * world, rank, world)  # round-robin global chain ids of this rank
    base = planted_labels(na, nb, ka, kb)
    labels_host = torch.empty((C, n), dtype=torch.int32).pin_memory()
    labels_host.numpy().view(np.uint32)[:] = base[None, :]
    pool = host.ChainPool(graph, labels_host.numpy().view(np.uint32), ka, kb, 1.0)
    pool.set_precision(args.precision)
    if args.inflight_div:
        pool.set_option("inflight_div", args.inflight_div)
    if args.warps:
        pool.set_option("warps", args.warps)
    if args.no_spare_sms:
        pool.set_option("spare_sms", 0)
    seeds = pkg.dist.chain_seeds(0, chain_ids)
    pool.randomize(seeds)
    duration = args.sweeps_per_step * n

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # -------- value: state resident in HBM
    for _ in range(args.warmup):
        pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
    if world > 1:  # warm the one collective of the path too (NCCL communicator set-up is not a sweep cost)
        try:
            with stdout_to_stderr():
                pkg.dist.init_pool_comm(pool)        # the library's own communicator (bisbm_nccl_init)
            config["collective"] = "bisbm_marginals_allreduce (ncclAllReduce behind the C ABI)"
        except Exception as ex:                  # no loadable libnccl.so.2: torch.distributed's all-reduce on the same buffer
            config["collective"] = "torch.distributed all_reduce (libbisbm could not set up NCCL: %s)" % str(ex)[:120]
        pool.marginals_clear()
        pool.marginalize(0, 1, 1, seeds)
        pkg.dist.allreduce_marginals(pool)
    # the labels at the start of the timed region: the end-to-end arm (and the fp32 figure) restart from them, so every arm
    # times the SAME phase of the chains (throughput follows their state: profiles/r02_experiments.txt)
    lab_dtype = torch.uint8 if ka + kb <= 256 else torch.int32
    np_view = (lambda t: t.numpy()) if lab_dtype == torch.uint8 else (lambda t: t.numpy().view(np.uint32))
    snap_host = torch.empty((C, n), dtype=lab_dtype).pin_memory()
    pool.labels(out=np_view(snap_host))
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    ev_ms, launches, moves, accs, sweep_launches = 0.0, 0, 0, [], 0
    for _ in range(args.steps):
        acc, sw = pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
        ms_, la_, mv_ = pool.last_timing()
        ev_ms += ms_; launches += la_; moves += mv_; accs.append(float(acc.mean()))
        sweep_launches += pool.sweep_launches()
    if world > 1:
        # the path's only collective: one all-reduce of the per-node marginal histogram
        pool.marginals_clear()
        pool.marginalize(0, 1, 1, seeds)          # one more sweep + the histogram accumulation
        ms_, la_, mv_ = pool.last_timing()
        ev_ms += ms_; launches += la_; moves += mv_
        sweep_launches += pool.sweep_launches()
        pkg.dist.allreduce_marginals(pool)       # bisbm_marginals_allreduce: ncclAllReduce(sum, uint32) behind the C ABI
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs:       # before the e2e arm below restarts the chains from snap_host
        dump_outputs(args.dump_outputs, pool, acc, sw)
    t = torch.tensor([wall, ev_ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(moves)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    wall_max, ev_max = float(t[0]), float(t[1])
    total_moves = float(tot[0])
    value = total_moves / wall_max
    acceptance = float(np.mean(accs))
    kern, wpc_, cpg_, slice_ = pool.sweep_info()
    kernel_names = {0: "sweep_kernel<double, counts in L2>", 1: "sweep_kernel<double, staged counts> (round 1)",
                    2: "sweep2_kernel<float, staged counts>", 3: "sweep2_kernel<double, staged counts>",
                    4: "sweep2_kernel<float, counts in L2>", 5: "sweep2_kernel<double, counts in L2>",
                    6: "sweep2_kernel<float, counts over a cluster>", 7: "sweep2_kernel<double, counts over a cluster>"}
    kernel_name = kernel_names[kern]
    sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    groups = (C + 31) // 32
    spare = 0 if args.no_spare_sms or cpg_ <= 1 else max(0, min(sms - groups * cpg_, groups - 1))
    per_cta = slice_ // max(1, cpg_)
    config["sweep_plan"] = {"kernel": kernel_name, "warps_per_cta": wpc_, "ctas_per_chain_group": cpg_,
                            "slice_vertices_per_launch": slice_, "max_inflight": slice_ + (per_cta if spare else 0),
                            "spare_sm_ctas_per_launch": spare,
                            "inflight_bound": "half sweep / %d%s" % (args.inflight_div or 64, (
                                " (+ one CTA's share of %d positions in the launches where a chain group holds one of the %d spare-SM CTAs)" % (per_cta, spare)) if spare else "")}
    dtype = "f32+int32 (dS summed in f64)" if kern == 2 else "f64+int32"

    # -------- e2e: host buffers in, host buffers out, every step (8-bit labels: K = ka + kb <= 256 here)
    in_host = torch.empty((C, n), dtype=lab_dtype).pin_memory()
    out_host = torch.empty((C, n), dtype=lab_dtype).pin_memory()
    in_host.copy_(snap_host)                      # same starting labels as the resident arm's timed region
    config["e2e_start"] = "labels at the start of the resident arm's timed region (same phase of the chains)"
    # a changed byte per step so the library cannot take its "labels unchanged -> keep the counts" shortcut
    def perturb(t, step):
        a = np_view(t)
        v = step % n
        a[0, v] = (a[0, v] + 1) % ka if v < na else ka + (a[0, v] - ka + 1) % kb
    for _ in range(1):
        pool.set_labels(np_view(in_host))
        pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
        pool.labels(out=np_view(out_host))
    barrier()
    t1 = time.perf_counter()
    e2e_moves = 0
    for step in range(args.steps):
        perturb(in_host, step)
        pool.set_labels(np_view(in_host))                             # H2D: C*n label bytes (+ count rebuild on the device)
        pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
        pool.labels(out=np_view(out_host))                            # D2H: C*n label bytes
        in_host, out_host = out_host, in_host
        e2e_moves += pool.last_timing()[2]
    barrier()
    e2e_wall = time.perf_counter() - t1
    label_bytes = C * n * (1 if lab_dtype == torch.uint8 else 4)
    te = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    me = torch.tensor([float(e2e_moves)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(me, op=dist.ReduceOp.SUM)
    e2e_value = float(me[0]) / float(te[0])

    # -------- extra: the same pool with fp32 move arithmetic (short run, state resident), for the record
    extra = {}
    if not args.no_fp32_extra and args.precision == "fp64":
        pool.set_labels(np_view(snap_host))       # same phase of the chains again
        pool.set_precision("fp32")
        pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
        ms32, mv32 = 0.0, 0
        for _ in range(2):
            pool.anneal("constant", 1.0, 0.0, duration, 10 ** 18, seeds)
            ms_, _la, mv_ = pool.last_timing()
            ms32 += ms_; mv32 += mv_
        pool.set_precision("fp64")
        t32 = torch.tensor([ms32], dtype=torch.float64, device="cuda")
        m32 = torch.tensor([float(mv32)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t32, op=dist.ReduceOp.MAX)
            dist.all_reduce(m32, op=dist.ReduceOp.SUM)
        extra["fp32_move_arithmetic"] = {"value": float(m32[0]) / (float(t32[0]) * 1e-3), "unit": "moves/s",
                                         "timing": "CUDA events, 2 steps, state resident", "kernel": kernel_names[2]}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        bytes_per_move = 16.0 + 8.0 * (2.0 * args.edges / n) + 4.0 * acceptance
        # dominant kernel = the sweep kernel; per-launch algorithmic bytes / average launch duration
        # (the library counts its sweep-kernel launches; the rest are logq_refresh / bookkeep / next-base kernels)
        sweep_launches = max(1, sweep_launches)
        alg_bytes_per_launch = bytes_per_move * (moves / sweep_launches)
        achieved = bytes_per_move * moves / (ev_ms * 1e-3) / 1e9
        line = {"metric": "vertex-moves/sec", "value": value, "unit": "moves/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": wall_max / args.steps * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": config,
                "acceptance": acceptance,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": None, "kernel": kernel_name, "bytes_per_move": bytes_per_move,
                             "alg_bytes_per_launch": alg_bytes_per_launch,
                             "avg_launch_ms": ev_ms / sweep_launches, "peak_source": peak_src,
                             "sweep_kernel_launches": int(sweep_launches),
                             "note": "CUDA events on libbisbm's stream around each step; they also span the small kernels between the sweep launches (log q refresh, bookkeeping, next-base initialisation: profiles/r02_launch_shares.txt)"},
                "e2e": {"value": e2e_value, "unit": "moves/s", "h2d_bytes_per_step": label_bytes, "d2h_bytes_per_step": label_bytes,
                        "api": "bisbm_set_chains_u8 (pinned host labels in) -> bisbm_anneal -> bisbm_get_all_labels_u8 (host labels out), every step"},
                "gpu_launches": int(launches), "clocks": clocks, "extra": extra}
        traffic_file = os.path.join(ROOT, "profiles", "sweep_kernel_traffic.json")
        if os.path.exists(traffic_file):
            try:
                line["roofline"]["traffic"] = json.load(open(traffic_file)).get("dram_bytes_per_launch")
            except Exception:
                pass
        if not args.no_cpu_baseline and world == 1:
            try:
                path = os.path.join(tempfile.gettempdir(), "bisbm_bench_edges_%d.npy" % os.getpid())
                np.save(path, edges)
                kind = cpu_kind()
                procs = cpu_procs(3.5 if kind == "reference" else 1.5)
                v, mv, worst = run_cpu_sample(path, na, nb, ka, kb, args.cpu_moves, procs, kind)
                os.unlink(path)
                line["cpu_baseline"] = {"value": v, "unit": "moves/s", "cores": procs, "kind": kind,
                                        "sample": "%d processes x %d moves of anneal() (T=1) on the full graph from a fresh randomised start (acceptance ~0.93; the GPU arm is timed after its warm-up sweeps, acceptance in 'acceptance'), %.1f s, state build untimed" % (
                                            procs, mv // procs, worst)}
            except Exception as ex:  # the baseline is a reported number, never a reason to lose the bench line
                line["cpu_baseline"] = {"value": None, "unit": "moves/s", "cores": 0, "kind": "unavailable", "sample": str(ex)[:200]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
