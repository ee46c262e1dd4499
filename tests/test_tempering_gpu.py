"""Parallel tempering (bisbm_tempering_*) on the GPU: per-chain temperatures against constant-temperature pools bit for bit,
the swap rule against a host restatement, the exact stationary distribution of an enumerable model, cold-rung marginals,
determinism, invariants, argument errors and the --tempering command line."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from helpers import counts_from_labels, nmi, planted, planted_labels

pytestmark = pytest.mark.gpu

BIG = 2 ** 62           # steps_await that never stops an anneal early


def check_invariants(pool, edges, na, nb, chains):
    """m_rs / e_r / n_r / eta on the device equal a from-scratch rebuild from the labels."""
    for c in chains:
        ka, kb = int(pool.ka[c]), int(pool.kb[c])
        lab = pool.labels(c)
        assert (lab[:na] < ka).all() and (lab[na:] >= ka).all() and (lab[na:] < ka + kb).all()
        m, e, nr, eta = counts_from_labels(edges, na, nb, lab, ka, kb)
        assert (pool.m(c) == m).all() and (pool.m_r(c) == e).all() and (pool.n_r(c) == nr).all()
        assert (pool.eta(c) == eta).all()


def shared(host, graph):
    """a second handle over graph's device-resident graph (bisbm_share_graph): own chains, own sweep counter"""
    h = C.c_void_p()
    host._check(graph.L.bisbm_share_graph(graph.h, C.byref(h)))
    g = object.__new__(host.Graph)
    g.__dict__.update({k: v for k, v in graph.__dict__.items() if k != "h"})
    g.h = h
    return g


def hub_graph():
    """planted graph plus one type-a node joined to 300 type-b nodes: degree > 255 takes the round-1 kernel (0)"""
    na = nb = 400
    e = planted(na, nb, 4, 4, 6000, 5)
    hub = np.stack([np.zeros(300, dtype=np.uint32), na + np.arange(300, dtype=np.uint32)], 1)
    return np.concatenate([e, hub]).astype(np.uint32), na, nb, 4, 4


def small_graph():
    g = load_golden("c2_abrupt")
    return g["edges"], g["na"], g["nb"], 10, 10


def start_labels(na, nb, ka, kb, chains):
    return np.tile(np.concatenate([np.arange(na) % ka, ka + np.arange(nb) % kb]).astype(np.uint32), (chains, 1))


def ladders_of(rung, R):
    """[n_ladders][R]: the chain holding rung i of ladder l"""
    L = len(rung) // R
    at = np.zeros((L, R), dtype=np.int64)
    for c, r in enumerate(rung):
        at[c // R, r] = c
    return at


PLANS = {"staged_f64": (small_graph, "fp64", -1, 3), "staged_f32": (small_graph, "fp32", -1, 2),
         "l2_f64": (small_graph, "fp64", 5, 5), "hub_round1": (hub_graph, "fp64", -1, 0)}


@pytest.mark.parametrize("plan", sorted(PLANS))
def test_per_chain_beta_equals_constant_temperature_pools(host, plan):
    """No swap round (swap_every > sweeps): chain c of the ladder pool must be chain c of a pool annealed at the constant
    T = temps[c % 4] -- labels, entropy() and acceptance bit for bit -- on every sweep kernel; counts stay exact."""
    make, prec, kernel, kid = PLANS[plan]
    edges, na, nb, ka, kb = make()
    n = na + nb
    temps = [1.0, 1.25, 1.5, 2.0]            # exact in float: bisbm_anneal forms 1 / (double)(float)T
    chains, sweeps = 40, 6
    seeds = np.arange(chains, dtype=np.uint64) * 7 + 3
    graph = host.Graph(edges, na, nb)
    handles = [graph] + [shared(host, graph) for _ in temps]

    def pool_on(g):
        p = host.ChainPool(g, start_labels(na, nb, ka, kb, chains), ka, kb, 1.0)
        p.set_precision(prec)
        p.set_option("kernel", kernel)
        return p

    tp = pool_on(handles[0])
    tp.tempering_set(temps)
    tp.randomize(seeds)                      # keeps the ladder
    acc = tp.tempering_run(sweeps, sweeps + 1, seeds, max_inflight=1)
    assert tp.sweep_info()[0] == kid
    st = tp.tempering_stats()
    assert (st["rung_of_chain"] == np.arange(chains) % 4).all() and (st["swaps_tried"] == 0).all()
    assert (st["moves_tried"] == sweeps * n * chains // 4).all()
    lab, ent = tp.labels(), tp.entropy()
    for i, T in enumerate(temps):
        ref = pool_on(handles[1 + i])
        ref.randomize(seeds)
        acc_r, _ = ref.anneal("constant", T, 0.0, sweeps * n, BIG, seeds, max_inflight=1)
        sel = np.arange(i, chains, 4)
        assert (ref.labels()[sel] == lab[sel]).all(), (plan, T)
        assert (ref.entropy()[sel] == ent[sel]).all(), (plan, T)
        assert (acc_r[sel] == acc[sel]).all(), (plan, T)
        # the moves each rung is credited with are exactly those of its chains
        assert st["moves_accepted"][i] == int(round((acc[sel] * sweeps * n).sum()))
    # swaps on: the counts still equal a rebuild from the labels
    tp.tempering_run(sweeps, 1, seeds + 1)
    tp.tempering_run(3, 2, seeds + 2, max_inflight=1)
    check_invariants(tp, edges, na, nb, [0, 1, 2, 3, chains - 1])


def test_ladder_does_not_leak_into_anneal(host):
    edges, na, nb, ka, kb = small_graph()
    n = na + nb
    graph = host.Graph(edges, na, nb)
    other = shared(host, graph)
    seeds = np.arange(16, dtype=np.uint64) + 5
    a = host.ChainPool(graph, start_labels(na, nb, ka, kb, 16), ka, kb, 1.0)
    b = host.ChainPool(other, start_labels(na, nb, ka, kb, 16), ka, kb, 1.0)
    a.tempering_set([1.0, 1.5, 2.0, 3.0])
    for p in (a, b):
        p.randomize(seeds)
    acc_a, sw_a = a.anneal("constant", 1.5, 0.0, 5 * n, BIG, seeds, max_inflight=1)
    acc_b, sw_b = b.anneal("constant", 1.5, 0.0, 5 * n, BIG, seeds, max_inflight=1)
    assert (acc_a == acc_b).all() and (sw_a == sw_b).all()
    assert (a.labels() == b.labels()).all() and (a.entropy() == b.entropy()).all()


@pytest.mark.parametrize("vary_k", [0, 1])
def test_swap_rule_against_host(host, vary_k):
    """One sweep and one round per call: the rungs stay permutations, only pairs of the round's parity move, every pair with
    (beta_i - beta_{i+1})(S_i - S_{i+1}) >= 0 is swapped, the others are accepted as often as sum(p) says (|z| < 4), and
    the counters agree with what the host saw."""
    edges, na, nb, ka, kb = small_graph()
    temps = np.array([1.0, 1.01, 1.02, 1.03, 1.04])
    R, L = len(temps), 48
    beta = 1.0 / temps
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, start_labels(na, nb, ka, kb, R * L), ka, kb, 1.0)
    pool.set_option("vary_k", vary_k)
    seeds = np.arange(R * L, dtype=np.uint64) + 17
    pool.randomize(seeds)
    pool.tempering_set(temps)
    pool.tempering_run(40, 10 ** 6, seeds)           # burn-in, no round
    rung = pool.tempering_stats()["rung_of_chain"]
    tried = np.zeros(R - 1, dtype=np.int64)
    accepted = np.zeros(R - 1, dtype=np.int64)
    n_sure = n_sure_moved = 0
    n_rand = acc_rand = 0
    sum_p = sum_pq = 0.0
    for k in range(60):
        pool.tempering_run(1, 1, seeds, swap_seed=99)
        new = pool.tempering_stats()["rung_of_chain"]
        S = pool.entropy()
        at0, at1 = ladders_of(rung, R), ladders_of(new, R)
        for l in range(L):
            assert sorted(new[l * R:(l + 1) * R]) == list(range(R))
            for i in range(R):
                if (i % 2 == k % 2 and i + 1 < R) or (i % 2 != k % 2 and i > 0):
                    continue
                assert at1[l, i] == at0[l, i]                 # rungs outside the round's pairs do not move
            for i in range(k % 2, R - 1, 2):
                ci, cj = at0[l, i], at0[l, i + 1]
                swapped = at1[l, i] == cj and at1[l, i + 1] == ci
                assert swapped or (at1[l, i] == ci and at1[l, i + 1] == cj)
                tried[i] += 1
                accepted[i] += swapped
                x = (beta[i] - beta[i + 1]) * (S[ci] - S[cj])
                if x >= 0:
                    n_sure += 1
                    n_sure_moved += swapped
                else:
                    p = np.exp(x)
                    n_rand += 1
                    sum_p += p
                    sum_pq += p * (1 - p)
                    acc_rand += swapped
        rung = new
    z = (acc_rand - sum_p) / np.sqrt(max(sum_pq, 1e-12))
    st = pool.tempering_stats()
    print("vary_k=%d: %d sure pairs, %d random pairs (sum p %.1f, accepted %d, z %.2f), acceptance per pair %s" % (
        vary_k, n_sure, n_rand, sum_p, acc_rand, z, accepted / tried))
    assert n_sure_moved == n_sure
    assert n_rand >= 200 and sum_pq > 20
    assert abs(z) < 4
    assert (st["swaps_tried"] == tried).all() and (st["swaps_accepted"] == accepted).all()


def test_equal_temperatures_compose_transpositions(host):
    """All rungs at one temperature: every proposed swap is accepted, the rung assignment is the host-composed sequence of
    even / odd transpositions (across calls: the round counter lives on the handle), and the round trips follow."""
    edges, na, nb, ka, kb = small_graph()
    R, L = 5, 3
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, start_labels(na, nb, ka, kb, R * L), ka, kb, 1.0)
    seeds = np.arange(R * L, dtype=np.uint64) + 1
    pool.tempering_set([1.3] * R)
    at = np.arange(R * L).reshape(L, R)
    trip = np.where(np.arange(R * L) % R == 0, 1, 0)
    trips = np.zeros(L, dtype=np.int64)
    k = 0
    for sweeps in (7, 3, 1, 12):
        pool.tempering_run(sweeps, 1, seeds)
        for _ in range(sweeps):
            for l in range(L):
                for i in range(k % 2, R - 1, 2):
                    at[l, i], at[l, i + 1] = at[l, i + 1], at[l, i]
                cold, hot = at[l, 0], at[l, R - 1]
                if trip[cold] == 2:
                    trips[l] += 1
                trip[cold] = 1
                if trip[hot] == 1:
                    trip[hot] = 2
            k += 1
        st = pool.tempering_stats()
        assert (ladders_of(st["rung_of_chain"], R) == at).all()
    assert (st["swaps_tried"] == st["swaps_accepted"]).all()
    assert st["swaps_tried"].tolist() == [L * ((k + 1) // 2), L * (k // 2), L * ((k + 1) // 2), L * (k // 2)]
    assert (st["round_trips"] == trips).all() and trips.sum() > 0


def stationary_model():
    """13 node pairs, each joined by 3 parallel edges: S spans ~9 nats over the 900 states, so one sweep at T = 1.6 leaves a
    state far from the T = 1 distribution (with single edges the spread is ~3 nats and a wrong swap rule that lets chains
    reach the cold rung from a hotter one passes the chi-square test unnoticed)"""
    na = nb = 5
    e = [(i, na + i) for i in range(5)] + [(i, na + (i + 1) % 5) for i in range(5)] + [(0, na + 2), (1, na + 3), (3, na + 0)]
    return np.array(e * 3, dtype=np.uint32), na, nb


def all_states(na, nb):
    """every labelling with Ka = Kb = 2 and no empty block (global ids: a in {0, 1}, b in {2, 3})"""
    side = lambda n: [s for s in itertools.product((0, 1), repeat=n) if 0 < sum(s) < n]
    return np.array([list(a) + [2 + x for x in b] for a in side(na) for b in side(nb)], dtype=np.uint32)


def chi2_levels(S_all, S_samples, T):
    """chi-square p-value of the energy-level histogram of S_samples against exp(-S/T) over the enumerated states"""
    from scipy.stats import chisquare
    lv_all = np.round(S_all, 6)
    levels, g = np.unique(lv_all, return_counts=True)
    w = g * np.exp(-(levels - levels.min()) / T)
    exp_ = len(S_samples) * w / w.sum()
    idx = np.searchsorted(levels, np.round(S_samples, 6))
    assert (levels[np.minimum(idx, len(levels) - 1)] == np.round(S_samples, 6)).all(), "a sample outside the enumerated states"
    obs = np.bincount(idx, minlength=len(levels)).astype(np.float64)
    bo, be, co, ce = [], [], 0.0, 0.0
    for o, e in zip(obs, exp_):
        co += o; ce += e
        if ce >= 5:
            bo.append(co); be.append(ce); co = ce = 0.0
    if ce > 0:
        bo[-1] += co; be[-1] += ce
    return chisquare(bo, be).pvalue, len(bo)


def test_exact_stationary_distribution(host):
    """1024 ladders of 4 rungs (T = 1 .. 4) on a 5 + 5 node graph with Ka = Kb = 2 (900 states, all enumerated): after
    burn-in ONE sample per ladder; the energy-level histograms of the cold and the hottest rung must follow exp(-S/T)
    (chi-square p > 1e-3).  Control: a pool without swaps at T = 1 (a failure there is the base sampler's)."""
    edges, na, nb = stationary_model()
    states = all_states(na, nb)
    assert len(states) == 900
    g0 = host.Graph(edges, na, nb)
    S_all = host.ChainPool(g0, states, 2, 2, 1.0).entropy()
    rng = np.random.default_rng(7)
    temps = [1.0, 1.6, 2.5, 4.0]
    R, L = 4, 1024
    start = states[rng.integers(0, len(states), R * L)]
    seeds = np.arange(R * L, dtype=np.uint64) * 3 + 11
    g1 = host.Graph(edges, na, nb)
    pool = host.ChainPool(g1, start, 2, 2, 1.0)
    pool.tempering_set(temps)
    pool.tempering_run(400, 1, seeds, swap_seed=5)
    st = pool.tempering_stats()
    S = pool.entropy()
    at = ladders_of(st["rung_of_chain"], R)
    p_cold, nb_cold = chi2_levels(S_all, S[at[:, 0]], 1.0)
    p_hot, nb_hot = chi2_levels(S_all, S[at[:, R - 1]], 4.0)
    g2 = host.Graph(edges, na, nb)
    ctl = host.ChainPool(g2, start[:L], 2, 2, 1.0)
    ctl.anneal("constant", 1.0, 0.0, 400 * (na + nb), BIG, seeds[:L])
    p_ctl, _ = chi2_levels(S_all, ctl.entropy(), 1.0)
    print("stationary: p cold %.4g (%d bins), p hot %.4g (%d bins), control p %.4g, swap acceptance %s, round trips %d" % (
        p_cold, nb_cold, p_hot, nb_hot, p_ctl, st["swaps_accepted"] / np.maximum(st["swaps_tried"], 1), st["round_trips"].sum()))
    assert p_ctl > 1e-3, "the base sampler (no swaps) does not sample exp(-S)"
    assert p_cold > 1e-3 and p_hot > 1e-3


def test_cold_rung_marginals(host):
    edges, na, nb, ka, kb = small_graph()
    n = na + nb
    R, L = 4, 10
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, start_labels(na, nb, ka, kb, R * L), ka, kb, 1.0)
    seeds = np.arange(R * L, dtype=np.uint64) + 3
    pool.tempering_set([1.0, 1.1, 1.2, 1.3])
    pool.tempering_run(5, 1, seeds)
    pool.marginals_clear()
    pool.tempering_run(1, 1, seeds, sample_every=1)
    cold = np.flatnonzero(pool.tempering_stats()["rung_of_chain"] == 0)
    assert len(cold) == L
    lab = pool.labels()
    want = np.zeros((n, ka + kb), dtype=np.int64)
    for c in cold:
        np.add.at(want, (np.arange(n), lab[c]), 1)
    assert (pool.marginals().astype(np.int64) == want).all()
    pool.tempering_run(6, 2, seeds, sample_every=3)
    assert (pool.marginals().sum(1) == 3 * L).all()


def test_determinism_multi_cta(host):
    """Two runs of the same calls on fresh handles agree bit for bit (multi-CTA staged plan; blocks of 5000 nodes cannot
    empty within a launch)."""
    na = nb = 20000
    edges = planted(na, nb, 4, 4, 400000, 3)
    R, L = 4, 16
    seeds = np.arange(R * L, dtype=np.uint64) + 123
    out = []
    for _ in range(2):
        graph = host.Graph(edges, na, nb)
        pool = host.ChainPool(graph, np.tile(planted_labels(na, nb, 4, 4), (R * L, 1)), 4, 4, 1.0)
        pool.randomize(seeds)
        pool.tempering_set(host.geometric_ladder(1.0, 1.5, R))
        pool.marginals_clear()
        acc = pool.tempering_run(3, 1, seeds, swap_seed=3, sample_every=1)
        acc2 = pool.tempering_run(2, 1, seeds + 1, swap_seed=3, sample_every=1)
        assert pool.sweep_info()[0] == 3 and pool.sweep_info()[2] > 1
        out.append((pool.labels(), pool.entropy(), acc, acc2, pool.marginals(), pool.tempering_stats()))
        del pool, graph
    a, b = out
    for x, y in zip(a[:5], b[:5]):
        assert (x == y).all()
    for k in a[5]:
        assert (a[5][k] == b[5][k]).all(), k


def test_errors_and_ladder_lifetime(host):
    edges, na, nb, ka, kb = small_graph()
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, start_labels(na, nb, ka, kb, 12), ka, kb, 1.0)
    Lb, h = pool.L, graph.h
    seeds = np.arange(12, dtype=np.uint64)

    def t_set(temps, rung=None):
        t = np.ascontiguousarray(temps, dtype=np.float64)
        r = None if rung is None else np.ascontiguousarray(rung, dtype=np.uint32).ctypes.data_as(C.POINTER(C.c_uint32))
        return Lb.bisbm_tempering_set(h, len(t), t.ctypes.data_as(C.POINTER(C.c_double)), r)

    def t_run(swap_every=1):
        return Lb.bisbm_tempering_run(h, 1, swap_every, 0, seeds.ctypes.data_as(C.POINTER(C.c_uint64)), 1, 0, None)

    def t_stats():
        return Lb.bisbm_tempering_stats(h, None, None, None, None, None, None)

    assert t_run() == 3 and t_stats() == 3                           # BISBM_ERR_STATE: no ladder
    assert t_set([1.0] * 5) == 1                                      # 5 does not divide 12
    assert t_set([1.0, 0.0, 2.0]) == 1 and t_set([1.0, -1.0, 2.0]) == 1
    assert t_set([1.0, np.nan, 2.0]) == 1 and t_set([1.0, np.inf, np.inf]) == 1
    assert t_set([1.0, 2.0, 1.5]) == 1                                # decreasing
    assert t_set([1.0, 2.0, 3.0], [0, 1, 1] * 4) == 1                 # not a permutation
    assert t_set([1.0, 2.0, 3.0], [0, 1, 3] * 4) == 1                 # out of range
    assert t_stats() == 3                                             # a rejected set leaves no ladder
    assert t_set([1.0, 2.0, 3.0], [2, 0, 1] * 4) == 0
    assert (pool.tempering_stats()["rung_of_chain"] == [2, 0, 1] * 4).all()
    assert t_run(swap_every=0) == 1
    pool.randomize(seeds)                                             # keeps the ladder
    assert t_run() == 0 and t_stats() == 0
    assert Lb.bisbm_tempering_set(h, 0, None, None) == 0 and t_stats() == 3   # n_rungs = 0 clears
    assert t_set([1.0, 2.0]) == 0
    pool.set_labels(start_labels(na, nb, ka, kb, 12))                 # bisbm_set_chains clears the ladder
    assert t_stats() == 3 and t_run() == 3
    with pytest.raises(host.BisbmError) as ei:
        pool.tempering_stats()
    assert ei.value.code == 3


CLI = os.path.join(ROOT, "bin", "mcmc")


def test_cli_tempering(pkg, tmp_path):
    """--marginalize --tempering on a planted graph: one label line of N ids, NMI against the planted partition within 0.1
    of plain --marginalize; the combinations it does not support exit 1 with their message."""
    pkg.build.build_all()
    g = load_golden("c2_const_k46")
    path = os.path.join(str(tmp_path), "g.edgelist")
    np.savetxt(path, g["edges"], fmt="%d", delimiter="\t")
    mb = os.path.join(str(tmp_path), "mb.txt")
    np.savetxt(mb, g["labels0"], fmt="%d")
    base = [CLI, "-e", path, "-y", "500", "500", "--membership_path", mb, "-b", "30", "-t", "120", "-f", "4", "--seed", "5"]
    run = lambda *a: subprocess.run(base + [str(x) for x in a], capture_output=True, text=True, timeout=300)
    plain = run("--marginalize", "--chains", 64)
    temp = run("--marginalize", "--chains", 64, "--tempering", 1, 1.3, 1.7, 2.2, "--swap_every", 2)
    assert plain.returncode == 0 and temp.returncode == 0, temp.stderr
    lp = np.array(plain.stdout.split(), dtype=np.int64)
    lt = np.array(temp.stdout.split(), dtype=np.int64)
    assert lt.size == 1000 and temp.stdout.count("\n") == 1
    n_p, n_t = nmi(lp, g["labels0"]), nmi(lt, g["labels0"])
    print("NMI plain %.4f tempering %.4f" % (n_p, n_t))
    assert n_t >= n_p - 0.1
    for extra, msg in [(["--marginalize", "--estimate", "--chains", 64], "does not combine with --estimate"),
                       (["--marginalize", "-g"], "agglomerative paths"), ([], "needs --marginalize"),
                       (["--marginalize", "--chains", 64, "--gpus", 2], "runs on one GPU"),
                       (["--marginalize", "--chains", 66], "multiple of the number of --tempering")]:
        p = run("--tempering", 1, 1.3, 1.7, 2.2, *extra)
        assert p.returncode == 1 and msg in p.stderr, (extra, p.stderr)
