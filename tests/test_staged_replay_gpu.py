"""The staged sweep kernel (sweep2_kernel, ids 3 / 2) replayed move by move against an exact host model of what each move
may see (tests/staged_model.cc, DESIGN.md 3.2).

Each call runs ONE sweep (duration = n), so every sweep restarts the model from the device's labels.  The model replays it
under the plan the library chose (plan_sweep / launch_full_sweep restated in helpers.sweep_plan, checked against
sweep_info()), and for every chain it did not mark ambiguous (a floating-point near-tie in an accept or epsilon test, or a
veto whose outcome depends on the order of atomics) the device's labels must be identical, its accepted count equal and its
entropy_accum delta equal to the model's sum of dS within the sum of the per-move tolerances.  This pins WHICH counts each
move reads -- a move that reads eta one launch too old, a CTA that misses its own earlier rounds, a vertex the spare-SM
position arithmetic skips -- which the count invariants and the distribution tests cannot see."""
import numpy as np
import pytest

from helpers import planted, replay_sweep, staged_model, sweep_plan

pytestmark = pytest.mark.gpu

BIG = 2 ** 62
SCHEDULES = {"exponential": 0, "linear": 1, "logarithmic": 2, "constant": 3, "abrupt_cool": 4}


def random_labels(rng, n_chains, na, nb, ka, kb):
    ka = np.broadcast_to(np.asarray(ka), (n_chains,))
    kb = np.broadcast_to(np.asarray(kb), (n_chains,))
    out = np.empty((n_chains, na + nb), dtype=np.uint32)
    for c in range(n_chains):
        out[c, :na] = rng.integers(0, ka[c], na)
        out[c, na:] = ka[c] + rng.integers(0, kb[c], nb)
    return out


def tiny_blocks(rng, labels, na, nb, ka, kb, tiny):
    """the first `tiny` blocks of each type hold one to three nodes"""
    for c in range(labels.shape[0]):
        for n0, nt, k, off in ((0, na, ka, 0), (na, nb, kb, ka)):
            perm = rng.permutation(nt)
            lab = off + tiny + np.arange(nt) % (k - tiny)
            pos = 0
            for b in range(tiny):
                sz = int(rng.integers(1, 4))
                lab[perm[pos:pos + sz]] = off + b
                pos += sz
            labels[c, n0:n0 + nt] = lab
    return labels


def hub_graph(rng, na, nb, n_edges, hubs, isolated):
    """random bipartite multigraph with `hubs` nodes per type of degree 33-255 and the last `isolated` nodes of each type
    without edges"""
    ea = rng.integers(0, na - isolated, n_edges)
    eb = na + rng.integers(0, nb - isolated, n_edges)
    extra = []
    for h in range(hubs):
        d = int(rng.integers(33, 200))
        extra.append(np.stack([np.full(d, h), na + rng.integers(0, nb - isolated, d)], 1))
        extra.append(np.stack([rng.integers(0, na - isolated, d), np.full(d, na + h)], 1))
    e = np.concatenate([np.stack([ea, eb], 1)] + extra)
    return e.astype(np.uint32)


def run_case(host, name, edges, na, nb, labels, ka, kb, eps, sweeps, precision, schedule="constant", p0=1.0, p1=0.0,
             inflight_div=None, max_inflight=0, vary_k=False, expect_sliced=True, min_warps=1):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    L = staged_model()
    n = na + nb
    n_chains = labels.shape[0]
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, labels, ka, kb, eps)
    pool.set_precision(precision)
    if inflight_div is not None:
        pool.set_option("inflight_div", inflight_div)
    if vary_k:
        pool.set_option("vary_k", 1)
    rp, col = graph.csr()
    seeds = (np.arange(n_chains, dtype=np.uint64) + 1) * np.uint64(0x9E3779B97F4A7C15 % 2 ** 61) + np.uint64(11)
    fp32 = precision == "fp32"
    compared = amb = moves = acc_total = 0
    worst = 0.0
    for sweep in range(sweeps):
        lab0 = pool.labels()
        ent0 = np.array([pool.entropy_accum(c) for c in range(n_chains)])
        acc, _ = pool.anneal(schedule, p0, p1, n, BIG, seeds, max_inflight)
        kernel, wpc, cpg, slice_ = pool.sweep_info()
        assert kernel == (2 if fp32 else 3), kernel
        div = inflight_div if inflight_div is not None else 64
        plans = [sweep_plan(nv, n_chains, sms, wpc, div, max_inflight) for nv in (na, nb)]
        assert plans[1][:2] == (cpg, slice_), (plans, cpg, slice_)           # the restated plan is the library's
        if expect_sliced:
            assert all(p[4] and p[0] >= 2 and p[1] < nv for p, nv in zip(plans, (na, nb))), plans
        else:
            assert all(not p[4] and p[2] >= min_warps for p in plans), plans
        got = pool.labels()
        d_acc = np.rint(acc * n).astype(np.uint64)
        d_ent = np.array([pool.entropy_accum(c) for c in range(n_chains)]) - ent0
        m = replay_sweep(L, na, nb, graph.n_edges, rp, col, lab0, ka, kb, eps, seeds, sweep, SCHEDULES[schedule], p0, p1,
                         plans, vary_k, fp32)
        ok = (m["flags"] & 1) == 0
        for c in np.flatnonzero(ok):
            assert (got[c] == m["labels"][c]).all(), (name, sweep, c, np.flatnonzero(got[c] != m["labels"][c])[:10])
            assert d_acc[c] == m["accepted"][c], (name, sweep, c, int(d_acc[c]), int(m["accepted"][c]))
            err = abs(d_ent[c] - m["dS"][c])
            assert err <= m["tol"][c] + 1e-9 * max(1.0, abs(m["dS"][c])), (name, sweep, c, d_ent[c], m["dS"][c], m["tol"][c])
            worst = max(worst, err)
        compared += int(ok.sum())
        amb += int((~ok).sum())
        moves += int(m["moves"][ok].sum())
        acc_total += int(m["accepted"][ok].sum())
    frac = compared / (compared + amb)
    print("\n%-28s %-4s chains compared %5d ambiguous %4d  moves %10d accepted %9d  max |d dS| %.2e" %
          (name, precision, compared, amb, moves, acc_total, worst))
    assert frac >= (0.80 if fp32 else 0.95), (name, frac)
    assert acc_total >= 0.01 * moves and acc_total > 1000, (name, acc_total, moves)
    pool = graph = None


PRECISIONS = ["fp64", "fp32"]
# fp32 decides an accept test to about 1e-4, so a chain meets a near-tie every ~10k moves: its cases run on graphs small enough
# that most chains stay comparable for a whole sweep (with the in-flight bound scaled so the plan is still sliced)
K32 = {"fp64": (16384, 65536, 64), "fp32": (640, 2560, 8)}     # nodes per type, edges, default inflight_div


@pytest.fixture(scope="module")
def k32_graphs():
    return {p: planted(nv, nv, 32, 32, ne, 3) for p, (nv, ne, _) in K32.items()}


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("variant", ["default", "rounds", "max_inflight"])
def test_replay_sliced_k32(host, k32_graphs, precision, variant):
    """Ka = Kb = 32, 256 chains: the benchmark's sweep2_kernel<R, 32, TYPE> -- by default one round per CTA and about 64
    launches per half sweep (eta ring, lazy log q refresh, spare-SM extras); `rounds` (inflight_div = 1, or 2 on the small
    fp32 graph so the slice stays below the half sweep): several rounds per CTA, several 448-vertex batches in fp64; an
    explicit max_inflight: sliced without extras."""
    nv, _, div = K32[precision]
    rng = np.random.default_rng(1)
    labels = random_labels(rng, 256, nv, nv, 32, 32)
    kw = {"default": {"inflight_div": div}, "rounds": {"inflight_div": 1 if precision == "fp64" else 2},
          "max_inflight": {"max_inflight": nv // 4}}[variant]
    run_case(host, "k32-" + variant, k32_graphs[precision], nv, nv, labels, 32, 32, 1.0, 2, precision, **kw)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_replay_sliced_generic(host, precision):
    """Ka != Kb with per-chain (ka, kb) varying inside a group, some chains with one block of a type, 200 chains (padding
    lanes), hubs of degree 33-199 fetched in place, isolated vertices (d = 0 proposals): the generic KF = 0 kernel."""
    rng = np.random.default_rng(2)
    na, nb, ne, div = (6000, 9000, 30000, 64) if precision == "fp64" else (500, 700, 2500, 4)
    edges = hub_graph(rng, na, nb, ne, 12, 40)
    n_chains = 200
    ka = (1 + np.arange(n_chains) % 5).astype(np.uint32)
    kb = (6 + np.arange(n_chains) % 6).astype(np.uint32)
    labels = random_labels(rng, n_chains, na, nb, ka, kb)
    run_case(host, "generic", edges, na, nb, labels, ka, kb, 0.5, 2, precision, inflight_div=div)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("vary_k", [False, True])
def test_replay_one_cta_multiwarp(host, precision, vary_k):
    """max_inflight = 5 on a small graph: a one-CTA plan with 5 warps per round (rounds misaligned to the 448-vertex
    batches), blocks of one to three nodes where the exact shared veto decides; in estimate mode blocks empty and reopen
    between rounds, so the occupied-block count must come from the same view as n_r."""
    rng = np.random.default_rng(3)
    na, nb = 1500, 1100
    edges = planted(na, nb, 8, 8, 6000, 4)
    labels = tiny_blocks(rng, random_labels(rng, 64, na, nb, 8, 8), na, nb, 8, 8, 3)
    run_case(host, "one-cta-5w" + ("-vary_k" if vary_k else ""), edges, na, nb, labels, 8, 8, 1.0, 3, precision,
             max_inflight=5, vary_k=vary_k, expect_sliced=False, min_warps=5)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_replay_sliced_vary_k(host, k32_graphs, precision):
    """estimate mode on the default sliced plan, with blocks of one to three nodes that empty"""
    nv, _, div = K32[precision]
    rng = np.random.default_rng(4)
    labels = tiny_blocks(rng, random_labels(rng, 256, nv, nv, 32, 32), nv, nv, 32, 32, 4)
    run_case(host, "k32-vary_k", k32_graphs[precision], nv, nv, labels, 32, 32, 1.0, 2, precision, inflight_div=div,
             vary_k=True)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("schedule", ["exponential", "abrupt_cool"])
def test_replay_schedules(host, k32_graphs, precision, schedule):
    """per-position beta of a cooling schedule; abrupt_cool switching to T = 0 near the end of the type-b half sweep (each
    call is one sweep, so its steps are 0 .. n - 1; a move with dS exactly 0 is a legitimate tie at T = 0)"""
    nv, _, div = K32[precision]
    p0, p1 = (1.0, 1.0 - 4.0 / nv) if schedule == "exponential" else (float(2 * nv - nv // 16), 0.0)
    rng = np.random.default_rng(5)
    labels = random_labels(rng, 128, nv, nv, 32, 32)
    run_case(host, "k32-" + schedule, k32_graphs[precision], nv, nv, labels, 32, 32, 1.0, 2, precision, schedule=schedule,
             p0=p0, p1=p1, inflight_div=div)
