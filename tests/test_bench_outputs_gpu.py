"""bench.py --dump-outputs on a small instance of the C3 workload: the outputs of the last timed step land in DIR as
float32 / float64 .npy files, under 64 MB; they are exactly what the timed arm's calls give when the same calls are made
again in this process (so they are the timed arm's last step, and a run's result does not depend on timing); --steps
sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

NA = NB = 10000
K = 8
EDGES = 200000
CHAINS = 40
SWEEPS = 2
WARMUP = 1
SMALL = ["--nodes", str(NA + NB), "--edges", str(EDGES), "--k", str(K), "--chains", str(CHAINS), "--sweeps-per-step", str(SWEEPS),
         "--no-cpu-baseline", "--no-fp32-extra"]


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(WARMUP),
                        "--dump-outputs", str(out_dir)] + SMALL, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0]), {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def _timed_arm_again(pkg, steps):
    """The calls bench.py makes up to the end of its timed steps, in this process: per-step acceptances and the pool."""
    import bench
    host, dist = pkg.host, pkg.dist
    n = NA + NB
    graph = host.Graph(bench.planted(NA, NB, K, K, EDGES, 0), NA, NB)
    pool = host.ChainPool(graph, np.tile(bench.planted_labels(NA, NB, K, K), (CHAINS, 1)), K, K, 1.0)
    pool.set_precision("fp64")
    seeds = dist.chain_seeds(0, dist.shard_chains(CHAINS, 0, 1))
    pool.randomize(seeds)
    for _ in range(WARMUP):
        pool.anneal("constant", 1.0, 0.0, SWEEPS * n, 10 ** 18, seeds)
    pool.labels(out=np.zeros((CHAINS, n), dtype=np.uint8))      # bench.py's snapshot of the labels before the timed steps
    accs = [pool.anneal("constant", 1.0, 0.0, SWEEPS * n, 10 ** 18, seeds)[0] for _ in range(steps)]
    return accs, pool


def test_dump_outputs_are_the_timed_arms_last_step(tmp_path, pkg):
    line3, d = _bench(tmp_path / "a", 3)
    assert line3["steps"] == 3
    assert sorted(d) == ["acceptance", "entropy", "labels", "labels_chains", "labels_nodes", "sweeps"]
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    assert (d["sweeps"] == SWEEPS).all() and (d["labels_chains"] == np.arange(CHAINS)).all()
    nodes = d["labels_nodes"].astype(np.int64)
    assert 0 < len(nodes) < NA + NB and (np.diff(nodes) > 0).all() and d["labels"].shape == (CHAINS, len(nodes))
    # the same calls again: bit for bit the dumped arrays, and the acceptance the JSON line reports for the timed steps
    accs, pool = _timed_arm_again(pkg, 3)
    assert line3["acceptance"] == float(np.mean([float(a.mean()) for a in accs]))
    assert (d["acceptance"] == accs[-1]).all()
    assert (d["entropy"] == pool.entropy()).all()
    assert (d["labels"] == pool.labels()[:, nodes]).all()
    # one timed step: a third of the sweep launches, the same sample of nodes
    line1, d1 = _bench(tmp_path / "b", 1)
    assert line1["steps"] == 1
    assert line3["roofline"]["sweep_kernel_launches"] == 3 * line1["roofline"]["sweep_kernel_launches"]
    assert (d1["labels_nodes"] == d["labels_nodes"]).all()
