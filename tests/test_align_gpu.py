"""Label alignment of the marginals (bisbm_marginals_align) on the GPU: exact recovery of permuted copies of a partition,
optimality of every chain's permutation against scipy's assignment solver, the statistical purpose (randomised starts
give the marginals of chains that share label identity), tempering, determinism, state rules and the command line."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_golden
from helpers import planted, planted_labels
from oracle import port

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "bin", "mcmc")


def overlap(lab, ref, lo, hi, k0, K):
    """O[r][r'] over nodes lo..hi-1: chain block r, reference block r' (type-local ids, k0 = the type's first global id)"""
    O = np.zeros((K, K), dtype=np.int64)
    np.add.at(O, (lab[lo:hi].astype(np.int64) - k0, ref[lo:hi].astype(np.int64) - k0), 1)
    return O


def composed_hist(labs, maps, chains, n, width):
    hist = np.zeros((n, width), dtype=np.int64)
    for c in chains:
        np.add.at(hist, (np.arange(n), maps[c][labs[c]]), 1)
    return hist


def check_optimal(labs, maps, ref, na, ka, kb, chains):
    """each map is a within-type permutation whose overlap with the reference is scipy's maximum"""
    from scipy.optimize import linear_sum_assignment
    n = len(ref)
    for c in chains:
        m = maps[c].astype(np.int64)
        assert sorted(m[:ka]) == list(range(ka)) and sorted(m[ka:]) == list(range(ka, ka + kb)), c
        for lo, hi, k0, K in ((0, na, 0, ka), (na, n, ka, kb)):
            O = overlap(labs[c], ref, lo, hi, k0, K)
            r, s = linear_sum_assignment(O, maximize=True)
            assert O[np.arange(K), m[k0:k0 + K] - k0].sum() == O[r, s].sum(), c


def test_exact_recovery_of_permuted_copies(host):
    """80 chains (not a multiple of 32: padding lanes), each the planted partition with its own permutation of block ids
    within each type.  Aligned to the planted partition, the histogram is 80 x one-hot(planted) and each map inverts its
    chain's permutation; without a reference the sample spreads over the columns as before."""
    g = load_golden("c2_const_k46")
    na, nb, edges, ref = g["na"], g["nb"], g["edges"], g["labels0"].astype(np.uint32)
    n, ka, kb, R = na + nb, 4, 6, 80
    rng = np.random.default_rng(7)
    perms = [(rng.permutation(ka), rng.permutation(kb)) for _ in range(R)]
    labs = np.stack([np.concatenate([pa[ref[:na]], ka + pb[ref[na:] - ka]]) for pa, pb in perms]).astype(np.uint32)
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, labs, ka, kb, 1.0)
    pool.marginals_clear()
    pool.marginal_sample()
    raw = pool.marginals().astype(np.int64)
    assert (raw == composed_hist(labs, [np.arange(ka + kb)] * R, range(R), n, ka + kb)).all()
    assert (raw.max(1) < R).any()
    pool.marginals_align(ref)
    pool.marginals_clear()
    pool.marginal_sample()
    hist = pool.marginals().astype(np.int64)
    expect = np.zeros((n, ka + kb), dtype=np.int64)
    expect[np.arange(n), ref] = R
    assert (hist == expect).all()
    maps = pool.marginals_alignment()
    for c, (pa, pb) in enumerate(perms):
        assert (maps[c][pa] == np.arange(ka)).all() and (maps[c][ka + pb] == ka + np.arange(kb)).all(), c


def _pool_k46(host, kernel):
    g = load_golden("c2_const_k46")
    graph = host.Graph(g["edges"], g["na"], g["nb"])
    R = 40
    pool = host.ChainPool(graph, np.tile(g["labels0"], (R, 1)).astype(np.uint8), 4, 6, 1.0)
    if kernel is not None:
        pool.set_option("kernel", kernel)
    seeds = np.arange(R, dtype=np.uint64) + 5
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 3 * graph.n, 10 ** 9, seeds)
    return pool, g["na"], 4, 6, g["labels0"].astype(np.uint32)


def _pool_k32(host):
    na = nb = 2000
    graph = host.Graph(planted(na, nb, 32, 32, 60000, 5), na, nb)
    R = 64
    ref = planted_labels(na, nb, 32, 32)
    pool = host.ChainPool(graph, np.tile(ref, (R, 1)).astype(np.uint8), 32, 32, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 9
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 3 * graph.n, 10 ** 9, seeds)
    return pool, na, 32, 32, ref


def _pool_k300(host):
    """no sweep: 300 blocks per type (i32 labels only) and a large assignment"""
    na = nb = 2000
    ka = kb = 300
    graph = host.Graph(planted(na, nb, 8, 8, 20000, 3), na, nb)
    R = 33
    ref = planted_labels(na, nb, ka, kb)
    lab0 = np.concatenate([np.arange(na) % ka, ka + np.arange(nb) % kb]).astype(np.uint32)
    pool = host.ChainPool(graph, np.tile(lab0, (R, 1)), ka, kb, 1.0)
    pool.randomize(np.arange(R, dtype=np.uint64) + 1)
    return pool, na, ka, kb, ref


@pytest.mark.parametrize("case", ["k46_staged_u8", "k32", "k46_round1_i32", "k300_i32"])
def test_alignment_is_optimal(host, case):
    pool, na, ka, kb, ref = {"k46_staged_u8": lambda: _pool_k46(host, None), "k32": lambda: _pool_k32(host),
                             "k46_round1_i32": lambda: _pool_k46(host, 0), "k300_i32": lambda: _pool_k300(host)}[case]()
    if case != "k300_i32":
        assert pool.sweep_info()[0] == (0 if case == "k46_round1_i32" else 3)
    n, R, W = len(ref), pool.n_chains, ka + kb
    labs = pool.labels()
    pool.marginals_align(ref)
    pool.marginals_clear()
    pool.marginal_sample()
    maps = pool.marginals_alignment()
    check_optimal(labs, maps, ref, na, ka, kb, range(R))
    assert (pool.marginals() == composed_hist(labs, maps, range(R), n, W)).all()
    # a chain equal to the reference keeps its labels (set_chains clears the reference: it is set again)
    labs[1] = ref
    pool.set_labels(labs.astype(np.uint8) if case in ("k46_staged_u8", "k32") else labs)
    with pytest.raises(host.BisbmError) as ei:
        pool.marginals_alignment()
    assert ei.value.code == 3
    pool.marginals_align(ref)
    pool.marginals_clear()
    pool.marginal_sample()
    maps = pool.marginals_alignment()
    assert (maps[1] == np.arange(W)).all()
    check_optimal(labs, maps, ref, na, ka, kb, [0, 1, R - 1])
    assert (pool.marginals() == composed_hist(labs, maps, range(R), n, W)).all()


def _matched(a, b, na, ka, kb):
    """b relabelled, within each type, by the one permutation that best matches it to a"""
    from scipy.optimize import linear_sum_assignment
    out = b.copy()
    for lo, hi, k0, K in ((0, na, 0, ka), (na, len(a), ka, kb)):
        O = overlap(b, a, lo, hi, k0, K)
        r, s = linear_sum_assignment(O, maximize=True)
        perm = np.empty(K, dtype=np.int64)
        perm[r] = s
        out[lo:hi] = k0 + perm[b[lo:hi] - k0]
    return out


def test_aligned_random_starts_match_oracle_marginals(host):
    """The purpose: 64 chains from RANDOMISED starts, a burn-in (exponential cooling from T = 3, then T = 1), the
    lowest-entropy chain as reference, aligned samples -- against oracle chains that share label identity (the common
    planted start of test_marginals_match_oracle).  Arg-max agreement after one global within-type matching must pass that
    test's 0.9.  Its KS bar is not applied and its TV bar is loosened from 0.1 to 0.2, for a measured reason that alignment
    cannot remove (DESIGN.md 3.6): from random starts
    only 3 of these 64 chains reach the planted mode (> 0.95 of nodes after matching; median 0.80), so their per-node
    marginals are flatter than those of chains started in it (measured on a B200: agreement 0.951, mean TV 0.148, KS p ~ 0).
    Alignment is what makes the histogram meaningful at all: without it the same samples give TV 0.72."""
    from scipy.optimize import linear_sum_assignment
    g = load_golden("c2_const_k46")
    na, nb, edges, mb = g["na"], g["nb"], g["edges"], g["labels0"]
    n = na + nb
    R, burn, sweeps, every = 64, 30, 120, 4
    hist_o = np.zeros((n, 10), dtype=np.int64)
    for s in range(R):
        o = port.PortChain(n, na, nb, edges, mb, 4, 6, 1.0, 300 + s, 400 + s)
        o.init(False)
        o.anneal("constant", 1.0, 0, burn * n, 10 ** 9)
        for k in range(sweeps // every):
            o.anneal("constant", 1.0, 0, every * n, 10 ** 9)
            np.add.at(hist_o, (np.arange(n), o.labels()), 1)
    po = hist_o / hist_o.sum(1, keepdims=True)

    def compare(hist_g):
        """(arg-max agreement, mean TV) after one global within-type matching of the GPU arg-max to the oracle's"""
        col = np.arange(10)
        for lo, hi, k0, K in ((0, na, 0, 4), (na, n, 4, 6)):
            r, s = linear_sum_assignment(overlap(hist_g.argmax(1), hist_o.argmax(1), lo, hi, k0, K), maximize=True)
            col[k0 + r] = k0 + s
        hist_m = np.zeros_like(hist_g)
        hist_m[:, col] = hist_g
        pg = hist_m / hist_m.sum(1, keepdims=True)
        return (po.argmax(1) == pg.argmax(1)).mean(), 0.5 * np.abs(po - pg).sum(1).mean()

    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(mb, (R, 1)), 4, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 9
    pool.randomize(seeds)
    pool.anneal("exponential", 3.0, 0.99, 300 * n, 10 ** 9, seeds)
    pool.anneal("constant", 1.0, 0.0, 200 * n, 10 ** 9, seeds)
    pool.marginals_clear()
    pool.marginals_align(pool.labels(int(np.argmin(pool.entropy()))))
    pool.marginalize(0, sweeps, every, seeds)
    hist_g = pool.marginals().astype(np.int64)
    assert (hist_g.sum(1) == R * (sweeps // every)).all()
    agree, tv = compare(hist_g)
    pool.marginals_align(None)
    pool.marginals_clear()
    pool.marginalize(0, sweeps, every, seeds)
    agree_u, tv_u = compare(pool.marginals().astype(np.int64))
    print("aligned: argmax agreement=%.3f mean TV=%.3f | unaligned: %.3f %.3f" % (agree, tv, agree_u, tv_u))
    assert agree > 0.9 and tv < 0.2
    assert tv_u > 0.5 and agree_u < agree


def test_tempering_cold_rung_samples_are_aligned(host):
    g = load_golden("c2_const_k46")
    na, nb, edges, ref = g["na"], g["nb"], g["edges"], g["labels0"].astype(np.uint32)
    n, R = na + nb, 64
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(ref, (R, 1)), 4, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 3
    pool.randomize(seeds)
    pool.tempering_set([1.0, 1.2, 1.5, 2.0])
    pool.tempering_run(10, 1, seeds, swap_seed=2)
    pool.marginals_align(ref)
    pool.marginals_clear()
    pool.tempering_run(1, 1, seeds, swap_seed=2, sample_every=1)
    labs, rung, maps = pool.labels(), pool.tempering_stats()["rung_of_chain"], pool.marginals_alignment()
    check_optimal(labs, maps, ref, na, 4, 6, range(R))          # every chain's map is computed
    cold = np.flatnonzero(rung == 0)
    assert len(cold) == R // 4
    assert (pool.marginals() == composed_hist(labs, maps, cold, n, 10)).all()


def _aligned_run(host, graph, mb, R, seeds):
    pool = host.ChainPool(graph, np.tile(mb, (R, 1)), 4, 6, 1.0)
    pool.randomize(seeds)
    pool.marginals_clear()
    pool.marginals_align(mb)
    pool.marginalize(20, 40, 4, seeds)
    return pool.marginals(), pool.marginals_alignment()


def test_determinism_and_state_rules(host):
    g = load_golden("c2_const_k46")
    na, nb, edges, mb = g["na"], g["nb"], g["edges"], g["labels0"].astype(np.uint32)
    n, R = na + nb, 48
    graph = host.Graph(edges, na, nb)
    seeds = np.arange(R, dtype=np.uint64) + 21
    # two pools on graphs of their own: a pool's draws are keyed by the sweeps its handle has run
    h1, m1 = _aligned_run(host, host.Graph(edges, na, nb), mb, R, seeds)
    h2, m2 = _aligned_run(host, host.Graph(edges, na, nb), mb, R, seeds)
    assert (h1 == h2).all() and (m1 == m2).all()
    assert h1.sum() == n * R * 10
    # randomize and marginals_clear keep the reference
    pool = host.ChainPool(graph, np.tile(mb, (R, 1)), 4, 6, 1.0)
    with pytest.raises(host.BisbmError) as ei:
        pool.marginals_alignment()                               # no reference, no aligned sample
    assert ei.value.code == 3
    pool.marginals_align(mb)
    with pytest.raises(host.BisbmError) as ei:
        pool.marginals_alignment()                               # a reference, but no aligned sample yet
    assert ei.value.code == 3
    pool.randomize(seeds)
    pool.marginals_clear()
    pool.marginal_sample()
    labs, maps = pool.labels(), pool.marginals_alignment()
    check_optimal(labs, maps, mb, na, 4, 6, range(R))
    assert (pool.marginals() == composed_hist(labs, maps, range(R), n, 10)).all()
    # NULL clears it: the next sample counts the raw labels again
    pool.marginals_align(None)
    pool.marginals_clear()
    pool.marginal_sample()
    assert (pool.marginals() == composed_hist(labs, [np.arange(10)] * R, range(R), n, 10)).all()
    with pytest.raises(host.BisbmError) as ei:
        pool.marginals_alignment()
    assert ei.value.code == 3
    # errors: bad reference labels (type a out of range, type b below ka), a heterogeneous pool
    for bad in (0, na):
        r = mb.copy()
        r[bad] = 10 if bad == 0 else 1
        with pytest.raises(host.BisbmError) as ei:
            pool.marginals_align(r)
        assert ei.value.code == 1
    het = host.ChainPool(graph, np.stack([mb, np.concatenate([mb[:na], mb[na:] + 1])]), [4, 5], [6, 6], 1.0)
    with pytest.raises(host.BisbmError) as ei:
        het.marginals_align(mb)
    assert ei.value.code == 1 and "one (ka, kb)" in str(ei.value)


def test_block_count_changes_drop_the_reference(host):
    """A replay merge that changes a chain's (ka, kb) drops the reference (its maps no longer fit the chain); a histogram
    left at another width by a pool of other K is refused when the reference is set, before any sweep runs."""
    g = load_golden("c2_const_k46")
    na, nb, edges, mb = g["na"], g["nb"], g["edges"], g["labels0"].astype(np.uint32)
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, mb[None, :], 4, 6, 1.0)
    pool.marginals_align(mb)
    pool.marginals_clear()
    pool.marginal_sample()
    assert (pool.marginals_alignment() == np.arange(10)).all()
    pool.replay_init(0, 1, 2)
    assert pool.replay_agg_merge(0, 1, 0) == (3, 6)
    with pytest.raises(host.BisbmError) as ei:
        pool.marginals_alignment()
    assert ei.value.code == 3
    pool.marginal_sample()                                       # unaligned again
    # widths: (4, 5) and (3, 6) chains leave a 9-wide histogram; a (4, 6) pool of the same shapes keeps the buffers
    het = np.stack([np.concatenate([mb[:na], 4 + np.minimum(mb[na:] - 4, 4)]), np.concatenate([np.minimum(mb[:na], 2), mb[na:] - 1])])
    graph2 = host.Graph(edges, na, nb)
    p9 = host.ChainPool(graph2, het, [4, 3], [5, 6], 1.0)
    p9.marginals_clear()
    p10 = host.ChainPool(graph2, np.stack([mb, mb]), 4, 6, 1.0)
    with pytest.raises(host.BisbmError) as ei:
        p10.marginals_align(mb)
    assert ei.value.code == 3 and "marginals_clear" in str(ei.value)
    p10.marginals_clear()
    p10.marginals_align(mb)
    p10.marginal_sample()
    assert (p10.marginals_alignment() == np.arange(10)).all()
    assert (p10.marginals().argmax(1) == mb).all()


def test_estimate_mode_empty_blocks_stay_in_place(host):
    """vary_k: a chain whose last blocks are empty; empty blocks are zero rows and columns and keep their ids"""
    g = load_golden("c2_const_k46")
    na, nb, edges, mb = g["na"], g["nb"], g["edges"], g["labels0"].astype(np.uint32)
    graph = host.Graph(edges, na, nb)
    ka, kb = 6, 8                       # upper bounds: blocks 4, 5 (type a) and 6 + 4 .. 6 + 7 (type b) stay empty
    ref = np.concatenate([mb[:na], mb[na:] + 2]).astype(np.uint32)
    lab = ref.copy()
    lab[:na] = np.array([1, 0, 3, 2], dtype=np.uint32)[mb[:na]]
    pool = host.ChainPool(graph, np.stack([lab, ref]), ka, kb, 1.0)
    pool.set_option("vary_k", 1)
    pool.marginals_align(ref)
    pool.marginals_clear()
    pool.marginal_sample()
    maps = pool.marginals_alignment()
    assert maps[0].tolist() == [1, 0, 3, 2, 4, 5] + list(range(6, 14))
    assert (maps[1] == np.arange(14)).all()


def _run_cli(*args):
    p = subprocess.run([CLI] + [str(a) for a in args], capture_output=True, text=True, timeout=600)
    return p.returncode, p.stdout, p.stderr


def test_cli_align(pkg, tmp_path):
    """--marginalize --randomize --align prints a valid partition close to the planted one (after one within-type
    matching); with --tempering too; --gpus 2 --align agrees with one GPU (or fails cleanly on a one-GPU box)."""
    import torch
    pkg.build.build_all()
    g = load_golden("c2_const_k46")
    na, mb = g["na"], g["labels0"].astype(np.int64)
    path = os.path.join(str(tmp_path), "g.edgelist")
    np.savetxt(path, g["edges"], fmt="%d", delimiter="\t")
    common = ["-e", path, "-y", 500, 500, "-n", 125, 125, 125, 125, 83, 83, 83, 83, 84, 84, "-z", 4, 6, "--marginalize",
              "--randomize", "--align", "-b", 200, "-t", 120, "-f", 4, "--chains", 64, "--seed", 5]

    def valid(out):
        lab = np.array(out.split(), dtype=np.int64)
        assert lab.size == 1000 and (lab[:500] < 4).all() and (lab[500:] >= 4).all() and (lab[500:] < 10).all()
        return lab

    rc, out, err = _run_cli(*common)
    assert rc == 0, err
    lab1 = valid(out)
    assert (_matched(mb, lab1, na, 4, 6) == mb).mean() > 0.8
    rc, out, err = _run_cli(*common[:-4], "--chains", 64, "--tempering", 1, 1.2, 1.5, 2, "--seed", 5)
    assert rc == 0, err
    assert (_matched(mb, valid(out), na, 4, 6) == mb).mean() > 0.8
    rc2, out2, err2 = _run_cli(*common, "--gpus", 2)
    if torch.cuda.device_count() < 2:
        assert rc2 == 1 and "device 1 out of range" in err2
        return
    assert rc2 == 0, err2
    assert (_matched(lab1, valid(out2), na, 4, 6) == lab1).mean() > 0.9
