"""Marginals resolved by mode (bisbm_marginal_modes_set / _get / _argmax) on the GPU: exact equality with a host recomputation
(optimal assignments by scipy) over every sweep kernel's label array, one mode against alignment, a known two-mode split,
the threshold, the marginalize / tempering / estimate-mode samples, non-interference with everything that exists, the state
rules and errors, the statistical purpose (the planted mode of a pool with randomised chains against the oracle) and the
command line."""
import os
import subprocess

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from conftest import ROOT, load_golden
from helpers import planted, planted_labels
from oracle import port

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "bin", "mcmc")
BIG = 10 ** 9
NONE = 0xffffffff


def _k46():
    g = load_golden("c2_const_k46")
    return g["edges"], g["na"], g["nb"], g["labels0"].astype(np.uint32)


def _overlap(lab, ref, lo, hi, k0, K):
    O = np.zeros((K, K), dtype=np.int64)
    np.add.at(O, (lab[lo:hi].astype(np.int64) - k0, ref[lo:hi].astype(np.int64) - k0), 1)
    return O


def _types(n, na, ka, kb):
    return ((0, na, 0, ka), (na, n, ka, kb))


def best_overlaps(labs, refs, na, ka, kb):
    """ov[c][m]: the nodes of chain c that agree with refs[m] after the optimal within-type permutation (scipy)"""
    n = labs.shape[1]
    ov = np.zeros((len(labs), len(refs)), dtype=np.int64)
    for c in range(len(labs)):
        for m, ref in enumerate(refs):
            for lo, hi, k0, K in _types(n, na, ka, kb):
                O = _overlap(labs[c], ref, lo, hi, k0, K)
                r, s = linear_sum_assignment(O, maximize=True)
                ov[c, m] += O[r, s].sum()
    return ov


def expected_modes(ov, min_overlap, n, counted):
    """chain_mode of the contract: the arg-max (lowest m among equals), M below the threshold, NONE if not counted"""
    M = ov.shape[1]
    best = ov.argmax(1)
    mode = np.where(ov[np.arange(len(ov)), best] < min_overlap * n, M, best)
    return np.where(counted, mode, NONE).astype(np.int64), best


def check_maps(labs, refs, maps, nearest, ov, na, ka, kb):
    """every map is a within-type permutation whose overlap with the nearest reference is the optimum"""
    n = labs.shape[1]
    for c in range(len(labs)):
        m = maps[c].astype(np.int64)
        assert sorted(m[:ka]) == list(range(ka)) and sorted(m[ka:]) == list(range(ka, ka + kb)), c
        ref = refs[nearest[c]]
        got = sum(_overlap(labs[c], ref, lo, hi, k0, K)[np.arange(K), m[k0:k0 + K] - k0].sum()
                  for lo, hi, k0, K in _types(n, na, ka, kb))
        assert got == ov[c, nearest[c]], c


class Tracker:
    """the host's account of a mode set: after every sample, the labels the sample read, checked against what the device
    reports, and the histograms and counters the samples must sum to"""

    def __init__(self, pool, refs, na, ka, kb, min_overlap=0.0):
        self.pool, self.refs, self.na, self.ka, self.kb, self.mo = pool, np.asarray(refs), na, ka, kb, min_overlap
        self.M, self.n = len(refs), len(refs[0])
        self.hist = np.zeros((self.M, self.n, ka + kb), dtype=np.int64)
        self.counted = np.zeros(self.M + 1, dtype=np.int64)

    def sample(self, labs, counted):
        got = self.pool.marginal_modes()
        ov = best_overlaps(labs, self.refs, self.na, self.ka, self.kb)
        want, nearest = expected_modes(ov, self.mo, self.n, counted)
        assert (got["chain_mode"].astype(np.int64) == want).all(), np.flatnonzero(got["chain_mode"] != want)[:5]
        check_maps(labs, self.refs, got["map"], nearest, ov, self.na, self.ka, self.kb)
        for c in np.flatnonzero(want < self.M):
            np.add.at(self.hist[want[c]], (np.arange(self.n), got["map"][c][labs[c]]), 1)
        for c in np.flatnonzero(want != NONE):
            self.counted[want[c]] += 1
        return got

    def check(self):
        got = self.pool.marginal_modes()
        assert (got["counted"].astype(np.int64) == self.counted).all(), (got["counted"], self.counted)
        assert (got["hist"].astype(np.int64) == self.hist).all()
        s = got["hist"].astype(np.int64).sum(2)
        assert (s.sum(0) == self.counted[:self.M].sum()).all()
        assert (self.pool.marginal_modes_argmax() == got["hist"].argmax(2)).all()
        return got


def _threshold_between(ov, n):
    """a min_overlap halfway between the lowest and the highest best overlap of these labels: a sample of them leaves some
    chains unassigned and assigns others (chains at T = 1 keep moving towards the references, so a threshold is chosen
    from the labels it will be applied to)"""
    best = ov.max(1)
    assert best.min() < best.max()
    return (float(best.min()) + float(best.max())) / (2 * n)


# case -> (graph, precision, forced kernel (-1: the planner's choice), kernel id that must run (None: any, sliced));
# the case table of test_coassign_gpu.py
CASES = {"staged_f64": ("k46", "fp64", -1, 3), "staged_f32": ("k46", "fp32", -1, 2), "l2": ("k46", "fp64", 5, 5),
         "round1_i32": ("k46", "fp64", 0, 0), "sliced": ("big", "fp64", -1, None)}


@pytest.mark.parametrize("case", list(CASES))
def test_modes_equal_the_host(host, case):
    """100 chains (padding lanes), (4, 6) blocks, 3 references; constant-T sweeps, a sample and the labels, four times"""
    gname, prec, kernel, kid = CASES[case]
    if gname == "k46":
        edges, na, nb, mb = _k46()
    else:
        na = nb = 20000
        edges = planted(na, nb, 8, 8, 200000, 11)
        mb = planted_labels(na, nb, 4, 6)
    n, R, ka, kb = na + nb, 100, 4, 6
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(mb, (R, 1)), ka, kb, 1.0)
    pool.set_precision(prec)
    pool.set_option("kernel", kernel)
    seeds = np.arange(R, dtype=np.uint64) + 17
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
    labs = pool.labels()
    refs = np.stack([mb, labs[7], labs[50]])
    for k in range(4):
        pool.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
        labs = pool.labels()
        if k % 2 == 0:
            # a new set (which zeroes the histograms and counters) every two samples, its threshold from the labels
            # the first of them reads
            mo = _threshold_between(best_overlaps(labs, refs, na, ka, kb), n)
            pool.marginal_modes_set(refs, mo)
            t = Tracker(pool, refs, na, ka, kb, mo)
        pool.marginal_sample()
        t.sample(labs, np.ones(R, dtype=bool))
        if k % 2 == 1:
            got = t.check()
            assert got["counted"][:3].sum() > 0 and got["counted"][3] > 0       # both sides of the threshold
            assert got["counted"].sum() == 2 * R
    info = pool.sweep_info()
    if kid is None:
        assert info[2] > 1, info                    # a sliced multi-CTA plan
    else:
        assert info[0] == kid, info


def test_one_mode_is_alignment(host):
    edges, na, nb, mb = _k46()
    n, R = na + nb, 100
    pool = host.ChainPool(host.Graph(edges, na, nb), np.tile(mb, (R, 1)), 4, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 5
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 3 * n, BIG, seeds)
    ref = pool.labels(3)
    pool.marginals_align(ref)
    pool.marginal_modes_set(ref[None, :], 0.0)
    pool.marginals_clear()
    for _ in range(3):
        pool.anneal("constant", 1.0, 0.0, n, BIG, seeds)
        pool.marginal_sample()
        got = pool.marginal_modes()
        assert (got["chain_mode"] == 0).all()
        assert (got["map"] == pool.marginals_alignment()).all()
    assert (got["hist"][0] == pool.marginals()).all()
    assert got["counted"].tolist() == [3 * R, 0]
    assert (pool.marginal_modes_argmax()[0] == pool.marginal_argmax()).all()


def _two_mode_pool(host):
    """the set-up of test_a_known_two_mode_split: two greedy fixed points, 64 chains alternating between them"""
    na = nb = 2000
    graph = host.Graph(planted(na, nb, 6, 6, 40000, 8, ratio=2.0), na, nb)
    n = na + nb
    rnd = np.random.default_rng(2)
    starts = [np.concatenate([rnd.integers(0, 6, na), 6 + rnd.integers(0, 6, nb)]).astype(np.uint32) for _ in range(2)]
    pre = host.ChainPool(graph, np.stack(starts), 6, 6, 1.0)
    pre.anneal("abrupt_cool", 0.0, 0.0, 60 * n, BIG, np.array([1, 2], dtype=np.uint64))
    fixed = pre.labels()
    R = 64
    pool = host.ChainPool(graph, np.stack([fixed[c % 2] for c in range(R)]), 6, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 100
    pool.anneal("abrupt_cool", 0.0, 0.0, 3 * n, BIG, seeds)
    return pool, seeds, n, na


def test_known_modes(host):
    pool, seeds, n, na = _two_mode_pool(host)
    R, S = pool.n_chains, 4
    refs, mode_of_chain = host.mode_references(pool)
    assert len(refs) == 2 and mode_of_chain.tolist() == [c % 2 for c in range(R)]
    pool.marginal_modes_set(refs)
    t = Tracker(pool, refs, na, 6, 6)
    for _ in range(S):
        pool.anneal("abrupt_cool", 0.0, 0.0, n, BIG, seeds)
        labs = pool.labels()
        pool.marginal_sample()
        got = t.sample(labs, np.ones(R, dtype=bool))
        assert got["chain_mode"].tolist() == [c % 2 for c in range(R)]
    got = t.check()
    assert got["counted"].tolist() == [32 * S, 32 * S, 0]
    # each mode's arg-max is its own fixed point, relabelled to its reference: the reference itself
    am = pool.marginal_modes_argmax()
    for m in range(2):
        assert (am[m] == refs[m]).mean() > 0.95


def test_threshold(host):
    edges, na, nb, mb = _k46()
    n, R = na + nb, 100
    pool = host.ChainPool(host.Graph(edges, na, nb), np.tile(mb, (R, 1)), 4, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 31
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
    rng = np.random.default_rng(3)
    # two random partitions: chains at T = 1 approach the planted one, but none reaches these
    refs = np.stack([np.concatenate([rng.integers(0, 4, na), 4 + rng.integers(0, 6, nb)]) for _ in range(2)]).astype(np.uint32)
    assert best_overlaps(pool.labels(), refs, na, 4, 6).max() < n     # no chain equals a reference
    pool.marginal_modes_set(refs, 1.0)
    pool.marginal_sample()
    pool.marginal_sample()
    got = pool.marginal_modes()
    assert got["counted"].tolist() == [0, 0, 2 * R] and (got["hist"] == 0).all() and (got["chain_mode"] == 2).all()
    pool.marginal_modes_set(refs, 0.0)
    pool.marginal_sample()
    got = pool.marginal_modes()
    assert got["counted"][2] == 0 and got["counted"].sum() == R and (got["chain_mode"] < 2).all()


def test_marginalize_samples(host):
    edges, na, nb, mb = _k46()
    n, R = na + nb, 100
    pool = host.ChainPool(host.Graph(edges, na, nb), np.tile(mb, (R, 1)), 4, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 3
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
    labs = pool.labels()
    refs = np.stack([mb, labs[0], labs[1]])
    pool.marginal_modes_set(refs)
    t = Tracker(pool, refs, na, 4, 6)
    for _ in range(3):
        pool.marginalize(0, 3, 3, seeds)             # one sample, after the last sweep
        t.sample(pool.labels(), np.ones(R, dtype=bool))
    assert t.check()["counted"].sum() == 3 * R


def test_tempering_counts_the_cold_rung(host):
    edges, na, nb, mb = _k46()
    n, R, rungs = na + nb, 100, 4
    pool = host.ChainPool(host.Graph(edges, na, nb), np.tile(mb, (R, 1)), 4, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 8
    pool.randomize(seeds)
    pool.tempering_set([1.0, 1.3, 1.7, 2.2])
    pool.tempering_run(3, 1, seeds, swap_seed=9)
    labs = pool.labels()
    refs = np.stack([mb, labs[2], labs[5]])
    pool.marginal_modes_set(refs)
    t = Tracker(pool, refs, na, 4, 6)
    for k in range(3):
        pool.tempering_run(3, 1, seeds, swap_seed=k + 1, sample_every=3)
        rung = pool.tempering_stats()["rung_of_chain"]
        assert (rung == 0).sum() == R // rungs
        got = t.sample(pool.labels(), rung == 0)
        assert (got["chain_mode"][rung != 0] == NONE).all()
    assert t.check()["counted"].sum() == 3 * (R // rungs)


def test_estimate_mode(host):
    """vary_k with bounds (6, 8) over a (4, 6) start: blocks empty, and an empty block that is empty in the reference too
    keeps its id"""
    edges, na, nb, mb = _k46()
    n, R = na + nb, 100
    lab = np.concatenate([mb[:na], mb[na:] + 2]).astype(np.uint32)
    pool = host.ChainPool(host.Graph(edges, na, nb), np.tile(lab, (R, 1)), 6, 8, 1.0)
    pool.set_option("vary_k", 1)
    seeds = np.arange(R, dtype=np.uint64) + 41
    pool.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
    refs = np.stack([lab, pool.labels(4)])
    pool.marginal_modes_set(refs)
    t = Tracker(pool, refs, na, 6, 8)
    fixed_checked = 0
    for _ in range(4):
        pool.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
        labs = pool.labels()
        pool.marginal_sample()
        got = t.sample(labs, np.ones(R, dtype=bool))
        for c in range(R):
            ref = refs[got["chain_mode"][c]]
            for g in range(14):
                if not (labs[c] == g).any() and not (ref == g).any():
                    assert got["map"][c][g] == g, (c, g)
                    fixed_checked += 1
    occ = np.asarray(pool.occupied_blocks()).reshape(R, 2)
    assert (occ < [6, 8]).any() and fixed_checked > 0
    t.check()


def test_non_interference(host):
    """twin pools with equal seeds (each on its own graph handle, which holds the co-assignment set), both with an
    alignment reference and a query set, one with a mode set: bit-identical labels, histogram, alignment maps and
    co-assignment counts after marginalize and tempering samples; 2 M + 2 more launches per sample"""
    edges, na, nb, mb = _k46()
    n, R, M = na + nb, 100, 2
    seeds = np.arange(R, dtype=np.uint64) + 13
    q = np.random.default_rng(6).permutation(n)[:200]
    refs = np.stack([mb, np.roll(mb, 1)]).astype(np.uint32)
    refs[1, :na] = refs[1, :na] % 4
    refs[1, na:] = 4 + (refs[1, na:] % 6)
    out = []
    for with_set in (True, False):
        p = host.ChainPool(host.Graph(edges, na, nb), np.tile(mb, (R, 1)), 4, 6, 1.0)
        p.randomize(seeds)
        p.marginals_align(mb)
        p.coassign_set(q)
        if with_set:
            p.marginal_modes_set(refs)
        p.marginals_clear()
        p.marginalize(2, 6, 3, seeds)
        p.tempering_set([1.0, 1.5])
        p.tempering_run(4, 1, seeds, swap_seed=3, sample_every=2)
        out.append((p.labels(), p.marginals(), p.marginals_alignment(), p.coassign(), p.last_timing()[1]))
    a, b = out
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all() and (a[2] == b[2]).all()
    assert (a[3][0] == b[3][0]).all() and a[3][1] == b[3][1]
    assert a[4] == b[4] + 2 * (2 * M + 2)


def test_state_rules_and_errors(host):
    edges, na, nb, mb = _k46()
    n, R = na + nb, 40
    graph = host.Graph(edges, na, nb)
    L = host.load_library()
    ref1 = np.ascontiguousarray(mb, dtype=np.uint32)
    # no pool
    assert L.bisbm_marginal_modes_set(graph.h, 1, host._p(ref1, host.C.c_uint32), 0.0) == 3
    pool = host.ChainPool(graph, np.tile(mb, (R, 1)), 4, 6, 1.0)
    for call in (pool.marginal_modes, pool.marginal_modes_argmax):
        with pytest.raises(host.BisbmError) as ei:
            call()                                   # no set yet
        assert ei.value.code == 3
    seeds = np.arange(R, dtype=np.uint64) + 1
    rng = np.random.default_rng(8)
    other = np.concatenate([rng.integers(0, 4, na), 4 + rng.integers(0, 6, nb)]).astype(np.uint32)
    refs = np.stack([mb, other])
    pool.marginal_modes_set(refs)
    got = pool.marginal_modes()                      # before any sample
    assert (got["chain_mode"] == NONE).all() and (got["map"] == NONE).all() and (got["counted"] == 0).all()
    pool.marginal_sample()
    assert pool.marginal_modes()["counted"].tolist() == [R, 0, 0]
    # bisbm_marginal_modes_set zeroes
    pool.marginal_modes_set(refs)
    assert pool.marginal_modes()["counted"].tolist() == [0, 0, 0] and (pool.marginal_modes()["hist"] == 0).all()
    pool.marginal_sample()
    # randomize keeps everything
    pool.randomize(seeds)
    assert pool.marginal_modes()["counted"].tolist() == [R, 0, 0]
    pool.marginal_sample()
    assert pool.marginal_modes()["counted"].sum() == 2 * R
    # marginals_clear zeroes and keeps the references
    pool.marginals_clear()
    got = pool.marginal_modes()
    assert (got["counted"] == 0).all() and (got["hist"] == 0).all()
    pool.marginal_sample()
    assert pool.marginal_modes()["counted"].sum() == R
    # errors: bad labels, min_overlap, a mixed pool; the set in place is kept
    for bad in (0, na):
        r = refs.copy()
        r[1, bad] = 10 if bad == 0 else 1
        with pytest.raises(host.BisbmError) as ei:
            pool.marginal_modes_set(r)
        assert ei.value.code == 1
    for mo in (float("nan"), -0.01, 1.01):
        with pytest.raises(host.BisbmError) as ei:
            pool.marginal_modes_set(refs, mo)
        assert ei.value.code == 1
    assert pool.marginal_modes()["counted"].sum() == R
    het = host.ChainPool(host.Graph(edges, na, nb), np.stack([mb, np.concatenate([mb[:na], mb[na:] + 1])]), [4, 5], [6, 6], 1.0)
    with pytest.raises(host.BisbmError) as ei:
        het.marginal_modes_set(mb)
    assert ei.value.code == 1 and "one (ka, kb)" in str(ei.value)
    # set_chains clears the set
    pool.set_labels(np.tile(mb, (R, 1)))
    with pytest.raises(host.BisbmError) as ei:
        pool.marginal_modes()
    assert ei.value.code == 3
    # NULL clears
    pool.marginal_modes_set(refs)
    pool.marginal_modes_set(None)
    with pytest.raises(host.BisbmError) as ei:
        pool.marginal_modes_argmax()
    assert ei.value.code == 3
    # a replay merge that changes a chain's (ka, kb) clears the set
    one = host.ChainPool(host.Graph(edges, na, nb), mb[None, :], 4, 6, 1.0)
    one.marginal_modes_set(mb)
    one.marginal_sample()
    one.replay_init(0, 1, 2)
    assert one.replay_agg_merge(0, 1, 0) == (3, 6)
    with pytest.raises(host.BisbmError) as ei:
        one.marginal_modes()
    assert ei.value.code == 3


def test_size_errors(host):
    """more blocks per type than shared memory holds; histograms no quarter of the free memory holds (the set is kept)"""
    na, nb = 2000, 10
    g = host.Graph(np.array([[0, na]], dtype=np.uint32), na, nb)
    lab = np.concatenate([np.arange(na) % 1900, 1900 + np.zeros(nb, dtype=np.int64)]).astype(np.uint32)
    p = host.ChainPool(g, lab[None, :], 1900, 1, 1.0)
    with pytest.raises(host.BisbmError) as ei:
        p.marginal_modes_set(lab)
    assert ei.value.code == 1 and "shared memory" in str(ei.value)
    na = nb = 60000
    g = host.Graph(np.array([[0, na]], dtype=np.uint32), na, nb)
    lab = np.concatenate([np.arange(na) % 1000, 1000 + np.arange(nb) % 1000]).astype(np.uint32)
    p = host.ChainPool(g, lab[None, :], 1000, 1000, 1.0)
    p.marginal_modes_set(lab)
    with pytest.raises(host.BisbmError) as ei:
        p.marginal_modes_set(np.tile(lab, (200, 1)))           # 200 x 120000 x 2000 uint32 = 192 GB of histograms
    assert ei.value.code == 1 and "quarter" in str(ei.value)
    p.marginal_sample()
    counted, mp = np.zeros(2, dtype=np.uint64), np.zeros(2000, dtype=np.uint32)
    host._check(p.L.bisbm_marginal_modes_get(g.h, None, host._p(counted, host.C.c_uint64), None, host._p(mp, host.C.c_uint32)))
    assert counted.tolist() == [1, 0] and (mp == np.arange(2000)).all()


def test_planted_mode_matches_oracle_marginals(host):
    """The purpose.  The data and oracle of test_aligned_random_starts_match_oracle_marginals: half the pool starts at the
    planted partition, half from randomised starts (burnt in as there).  References: the planted partition for the planted
    mode, and one per further mode of the randomised half (mode_references over chain 0 -- still at the planted partition --
    and the randomised chains, so that randomised chains in the planted mode join it).  The planted mode's histogram must
    pass the original bars of test_marginals_match_oracle; the single-reference aligned histogram of the same run fails
    the KS bar (DESIGN.md 3.9 records the values)."""
    from scipy.stats import ks_2samp
    g = load_golden("c2_const_k46")
    na, nb, edges, mb = g["na"], g["nb"], g["edges"], g["labels0"].astype(np.uint32)
    n = na + nb
    H, burn, sweeps, every = 64, 30, 120, 4
    hist_o = np.zeros((n, 10), dtype=np.int64)
    for s in range(H):
        o = port.PortChain(n, na, nb, edges, mb, 4, 6, 1.0, 300 + s, 400 + s)
        o.init(False)
        o.anneal("constant", 1.0, 0, burn * n, 10 ** 9)
        for k in range(sweeps // every):
            o.anneal("constant", 1.0, 0, every * n, 10 ** 9)
            np.add.at(hist_o, (np.arange(n), o.labels()), 1)
    po = hist_o / hist_o.sum(1, keepdims=True)
    graph = host.Graph(edges, na, nb)
    rand = host.ChainPool(graph, np.tile(mb, (H, 1)), 4, 6, 1.0)
    rs = np.arange(H, dtype=np.uint64) + 9
    rand.randomize(rs)
    rand.anneal("exponential", 3.0, 0.99, 300 * n, 10 ** 9, rs)
    rand.anneal("constant", 1.0, 0.0, 200 * n, 10 ** 9, rs)
    pool = host.ChainPool(graph, np.concatenate([np.tile(mb, (H, 1)), rand.labels()]), 4, 6, 1.0)
    refs, mode_of = host.mode_references(pool, chains=np.r_[0, H:2 * H])
    refs[0] = mb                                     # the planted mode is represented by the planted partition
    M = len(refs)
    pool.marginal_modes_set(refs)
    pool.marginals_align(mb)
    pool.marginals_clear()
    seeds = np.arange(2 * H, dtype=np.uint64) + 9
    pool.marginalize(burn, sweeps, every, seeds)
    got = pool.marginal_modes()
    S = sweeps // every
    assert got["counted"].sum() == 2 * H * S and got["counted"][M] == 0

    def bars(hist):
        pg = hist / hist.sum(1, keepdims=True)
        return (ks_2samp(po.max(1), pg.max(1)).pvalue, (po.argmax(1) == pg.argmax(1)).mean(), 0.5 * np.abs(po - pg).sum(1).mean())

    p, agree, tv = bars(got["hist"][0].astype(np.int64))
    p_a, agree_a, tv_a = bars(pool.marginals().astype(np.int64))
    last = got["chain_mode"]
    ov0 = best_overlaps(pool.labels(), refs[:1], na, 4, 6)[:, 0] / n
    print("modes %d (randomised chains in the planted mode at the start: %d), weights %s" %
          (M, int((mode_of[H:] == 0).sum()), np.round(got["counted"][:M] / got["counted"].sum(), 4).tolist()))
    print("last sample: planted-start chains in mode 0: %d / %d, randomised chains in mode 0: %d; overlap with the planted "
          "partition of mode-0 chains: min %.3f median %.3f" % ((last[:H] == 0).sum(), H, (last[H:] == 0).sum(),
                                                               ov0[last == 0].min(), np.median(ov0[last == 0])))
    print("planted mode: KS p=%.3f argmax agreement=%.3f mean TV=%.3f | single-reference aligned: KS p=%.3g agreement=%.3f "
          "mean TV=%.3f" % (p, agree, tv, p_a, agree_a, tv_a))
    assert p > 0.01 and agree > 0.9 and tv < 0.1
    # the single-reference aligned histogram of the same samples misses the original KS bar and is far further from the
    # oracle (with half the pool started in the planted mode its TV alone stays under 0.1: 0.075 measured, DESIGN.md 3.9)
    assert p_a <= 0.01 and tv_a > 5 * tv


def _run_cli(*args):
    p = subprocess.run([str(a) for a in [CLI, *args]], capture_output=True, text=True, timeout=600)
    return p.returncode, p.stdout, p.stderr


@pytest.mark.parametrize("extra,per_sample", [([], 64), (["--align", "--agreement_out", "AGREE", "--coassign", "Q",
                                                          "--coassign_out", "CO"], 64),
                                              (["--tempering", 1, 1.2, 1.5, 2], 16)], ids=["plain", "combined", "tempering"])
def test_cli(pkg, tmp_path, extra, per_sample):
    """bin/mcmc --marginalize --chains 64 --randomize with and without --modes_out: stdout byte-identical, the file's
    counts sum to the counted samples, its label lines have the stdout format"""
    pkg.build.build_all()
    edges, na, nb, _ = _k46()
    d = str(tmp_path)
    path = os.path.join(d, "g.edgelist")
    np.savetxt(path, edges, fmt="%d", delimiter="\t")
    np.savetxt(os.path.join(d, "Q"), np.arange(0, 1000, 7), fmt="%d")
    extra = [os.path.join(d, x) if x in ("AGREE", "Q", "CO") else x for x in extra]
    out = os.path.join(d, "modes.txt")
    common = ["-e", path, "-y", 500, 500, "-n", 125, 125, 125, 125, 83, 83, 83, 83, 84, 84, "-z", 4, 6, "--marginalize",
              "--randomize", "-b", 20, "-t", 40, "-f", 4, "--chains", 64, "--seed", 5]
    rc0, out0, err0 = _run_cli(*common, *extra)
    assert rc0 == 0, err0
    rc, so, se = _run_cli(*common, *extra, "--modes_out", out)
    assert rc == 0, se
    assert so == out0
    lines = [l for l in se.splitlines() if l.startswith("marginal modes:")]
    assert len(lines) == 1, se
    with open(out) as f:
        rows = f.read().split("\n")
    head = list(map(int, rows[0].split()))
    M = head[0]
    assert M >= 1 and len(head) == M + 2 and sum(head[1:]) == per_sample * 10 and head[-1] == 0
    assert rows[M + 1:] == [""]
    for m, r in enumerate(rows[1:M + 1]):
        assert r.endswith(" ")
        lab = np.array(r.split(), dtype=np.int64)
        assert lab.shape == (1000,)
        if head[1 + m]:         # a mode no sample went to has an empty histogram (arg-max 0 everywhere)
            assert (lab[:500] < 4).all() and ((lab[500:] >= 4) & (lab[500:] < 10)).all()
