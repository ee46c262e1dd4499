"""Parallel (many-chain) mode on the GPU through the C ABI: exact invariants after every call,
exactness of sequential chains (max_inflight=1), and statistical parity with the oracle."""
import numpy as np
import pytest

from conftest import load_golden
from helpers import counts_from_labels, nmi, planted, planted_labels
from oracle import port

pytestmark = pytest.mark.gpu


def check_invariants(pool, edges, na, nb, chains):
    """m_rs / e_r / n_r / eta on the device equal a from-scratch rebuild from the labels."""
    for c in chains:
        ka, kb = int(pool.ka[c]), int(pool.kb[c])
        lab = pool.labels(c)
        assert (lab[:na] < ka).all() and (lab[na:] >= ka).all() and (lab[na:] < ka + kb).all()
        m, e, nr, eta = counts_from_labels(edges, na, nb, lab, ka, kb)
        assert (pool.m(c) == m).all()
        assert (pool.m_r(c) == e).all()
        assert (pool.n_r(c) == nr).all() and (nr >= 1).all()
        assert (pool.eta(c) == eta).all()


@pytest.mark.parametrize("inflight,precision", [(1, "fp64"), (1, "fp32"), (0, "fp32"), (0, "fp64")])
def test_invariants_small_graph(host, inflight, precision):
    g = load_golden("c2_abrupt")
    na, nb = g["na"], g["nb"]
    graph = host.Graph(g["edges"], na, nb)
    C = 40  # not a multiple of 32: exercises the padded lanes
    pool = host.ChainPool(graph, np.tile(g["labels0"], (C, 1)), 10, 10, 1.0)
    pool.set_precision(precision)
    check_invariants(pool, g["edges"], na, nb, [0, 39])
    e0 = pool.entropy()
    assert abs(e0[0] - g["init_entropy"]) <= 1e-9 * g["init_entropy"]
    seeds = np.arange(C, dtype=np.uint64) + 1
    pool.randomize(seeds)
    check_invariants(pool, g["edges"], na, nb, [0, 17, 39])
    lab = pool.labels()
    assert not (lab[0] == lab[1]).all()
    e1 = pool.entropy()
    acc, sw = pool.anneal("constant", 1.0, 0.0, 20 * 1000, 10 ** 9, seeds, max_inflight=inflight)
    assert (sw == 20).all() and (acc > 0.05).all() and (acc <= 1.0).all()
    check_invariants(pool, g["edges"], na, nb, [0, 5, 31, 32, 39])
    e2 = pool.entropy()
    if inflight == 1:
        # sequential chains: the accumulated dS is the entropy difference (to the rounding of the move
        # arithmetic: double, or fp32 per move summed in double over ~1e4 accepted moves)
        tol = 1e-7 if precision == "fp64" else 1e-6
        for c in (0, 33, 39):
            assert abs((e2[c] - e1[c]) - pool.entropy_accum(c)) <= tol * abs(e1[c])


def test_heterogeneous_k_and_single_block_types(host):
    g = load_golden("c1_seed1")
    na, nb = g["na"], g["nb"]
    graph = host.Graph(g["edges"], na, nb)
    kas = np.array([1, 2, 5, 3, 1], dtype=np.uint32)
    kbs = np.array([1, 3, 5, 1, 4], dtype=np.uint32)
    labs = np.stack([np.concatenate([np.arange(na) % a, a + np.arange(nb) % b]) for a, b in zip(kas, kbs)]).astype(np.uint32)
    pool = host.ChainPool(graph, labs, kas, kbs, 0.1)
    seeds = np.arange(5, dtype=np.uint64) + 11
    acc, sw = pool.anneal("exponential", 10.0, 0.99, 200 * 32, 10 ** 9, seeds)
    check_invariants(pool, g["edges"], na, nb, range(5))
    assert (pool.labels(0) == labs[0]).all()  # (1,1): nothing can move


def test_early_stop_and_abrupt_cool(host):
    g = load_golden("c2_abrupt")
    graph = host.Graph(g["edges"], g["na"], g["nb"])
    pool = host.ChainPool(graph, np.tile(g["labels0"], (8, 1)), 10, 10, 1.0)
    seeds = np.arange(8, dtype=np.uint64) + 5
    acc, sw = pool.anneal("abrupt_cool", 100.0, 0.0, 20000, 100, seeds)
    # same command as golden c2_abrupt: T=0 from step 100 on, u reaches steps_await within the first sweeps
    assert (sw >= 1).all() and (sw <= 20).all()
    e = pool.entropy()
    assert (e < g["init_entropy"]).all()  # greedy descent only lowers the description length
    check_invariants(pool, g["edges"], g["na"], g["nb"], [0, 7])


def test_statistical_parity_with_oracle_nmi_and_entropy(host):
    """SURVEY.md 4(iv): 128 oracle chains vs 128 GPU chains on bisbm-1000 at (Ka,Kb)=(4,6), randomised
    starts, abrupt_cool T0 = 1e5 steps then greedy, 200 sweeps; compare the samples of final
    entropy() and of NMI against the planted file partition with a two-sample KS test (p > 0.01).  The oracle
    samples are the q46_* arrays of tests/golden/parity_mid.npz (tests/golden/make_parity_fixture.py)."""
    from scipy.stats import ks_2samp
    g = load_golden("c2_const_k46")
    fx = load_golden("parity_mid")
    na, nb, edges, mb = g["na"], g["nb"], g["edges"], g["labels0"]
    n = na + nb
    R = 128
    ent_o, nmi_o, acc_o = fx["q46_entropy"], fx["q46_nmi"], fx["q46_accept"]
    assert len(ent_o) >= 128
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(mb, (R, 1)), 4, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 77
    pool.randomize(seeds)
    acc_g, _ = pool.anneal("abrupt_cool", 1e5, 0.0, 200 * n, 10 ** 9, seeds)
    ent_g = pool.entropy()
    labs = pool.labels()
    nmi_g = [nmi(labs[c], mb) for c in range(R)]
    check_invariants(pool, edges, na, nb, [0, R - 1])
    p_ent = ks_2samp(ent_o, ent_g).pvalue
    p_nmi = ks_2samp(nmi_o, nmi_g).pvalue
    p_acc = ks_2samp(acc_o, acc_g).pvalue
    print("entropy oracle %.1f+-%.1f gpu %.1f+-%.1f p=%.3f | nmi oracle %.3f gpu %.3f p=%.3f | acc %.4f %.4f p=%.3f | plan %s" % (
        np.mean(ent_o), np.std(ent_o), np.mean(ent_g), np.std(ent_g), p_ent, np.mean(nmi_o), np.mean(nmi_g), p_nmi,
        np.mean(acc_o), np.mean(acc_g), p_acc, pool.sweep_info()))
    assert p_ent > 0.01 and p_nmi > 0.01 and p_acc > 0.01


def test_marginals_match_oracle(host):
    """Per-node marginals at T=1 from a common non-randomised start (label identity shared,
    SURVEY.md H9): GPU pool vs oracle chains; KS on the per-node max-marginal values and
    agreement of the arg-max labels."""
    from scipy.stats import ks_2samp
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
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(mb, (R, 1)), 4, 6, 1.0)
    pool.marginals_clear()
    pool.marginalize(burn, sweeps, every, np.arange(R, dtype=np.uint64) + 9)
    hist_g = pool.marginals().astype(np.int64)
    assert hist_g.shape == (n, 10) and (hist_g.sum(1) == R * (sweeps // every)).all()
    assert (hist_o.sum(1) == R * (sweeps // every)).all()
    po = hist_o / hist_o.sum(1, keepdims=True)
    pg = hist_g / hist_g.sum(1, keepdims=True)
    p = ks_2samp(po.max(1), pg.max(1)).pvalue
    agree = (po.argmax(1) == pg.argmax(1)).mean()
    tv = 0.5 * np.abs(po - pg).sum(1).mean()
    print("marginals: KS p=%.3f argmax agreement=%.3f mean TV=%.3f" % (p, agree, tv))
    assert (pool.marginal_argmax() == hist_g.argmax(1)).all()
    assert p > 0.01 and agree > 0.9 and tv < 0.1


def test_large_graph_invariants_and_logq_expansion(host):
    """A graph big enough for many warps per chain (stale-count concurrency) and for blocks with
    e_r >= 16384 (second-order log q expansion path)."""
    na = nb = 20000
    ka = kb = 4
    edges = planted(na, nb, ka, kb, 400000, 3)
    graph = host.Graph(edges, na, nb)
    C = 64
    pool = host.ChainPool(graph, np.tile(planted_labels(na, nb, ka, kb), (C, 1)), ka, kb, 1.0)
    seeds = np.arange(C, dtype=np.uint64) + 123
    pool.randomize(seeds)
    e1 = pool.entropy()
    acc, sw = pool.anneal("constant", 1.0, 0.0, 3 * (na + nb), 10 ** 9, seeds)
    check_invariants(pool, edges, na, nb, [0, 63])
    e2 = pool.entropy()
    ms, launches, moves = pool.last_timing()
    assert moves == 3 * (na + nb) * C and launches >= 6 and ms > 0
    # stale reads make the accumulated dS approximate, but it must track the true change closely
    for c in (0, 63):
        d_true, d_acc = e2[c] - e1[c], pool.entropy_accum(c)
        assert abs(d_true - d_acc) <= 0.10 * abs(d_true) + 10.0
    # sequential chains: exact
    pool2 = host.ChainPool(graph, np.tile(planted_labels(na, nb, ka, kb), (C, 1)), ka, kb, 1.0)
    pool2.randomize(seeds)
    f1 = pool2.entropy()
    pool2.anneal("constant", 1.0, 0.0, 1 * (na + nb), 10 ** 9, seeds, max_inflight=1)
    f2 = pool2.entropy()
    for c in (0, 63):
        assert abs((f2[c] - f1[c]) - pool2.entropy_accum(c)) <= 1e-6 * abs(f1[c])


@pytest.mark.parametrize("kernel", [-1, 0, 4])
def test_large_k_kernels(host, kernel):
    """K too large for one CTA's shared memory (KA*KB*128 B > 220 KB): the counts stay in L2 and commits are global
    atomics -- sweep2_kernel<double, .., STAGED = false> (kernel 5) by default, the round-1 kernel (0) on request, and
    sweep2_kernel<float, .., STAGED = false> (4) as the automatic choice in fp32 precision.  Same invariants; sequential
    chains are exact.  The retired kernel ids 1 (round-1 staged) and 7 (sweep2 over a thread-block cluster) are
    rejected."""
    na = nb = 3000
    ka = kb = 48
    edges = planted(na, nb, 8, 8, 60000, 11)
    graph = host.Graph(edges, na, nb)
    C = 33
    lab0 = np.concatenate([np.arange(na) % ka, ka + np.arange(nb) % kb]).astype(np.uint32)
    option = -1 if kernel == 4 else kernel
    precision = "fp32" if kernel == 4 else "fp64"
    pool = host.ChainPool(graph, np.tile(lab0, (C, 1)), ka, kb, 1.0)
    for retired in (1, 7):
        with pytest.raises(host.BisbmError) as ei:
            pool.set_option("kernel", retired)
        assert ei.value.code == 1     # BISBM_ERR_ARG
    pool.set_option("kernel", option)
    pool.set_precision(precision)
    seeds = np.arange(C, dtype=np.uint64) + 31
    pool.randomize(seeds)
    e1 = pool.entropy()
    pool.anneal("constant", 1.0, 0.0, 4 * (na + nb), 10 ** 9, seeds)
    assert pool.sweep_info()[0] == {-1: 5, 0: 0, 4: 4}[kernel]
    check_invariants(pool, edges, na, nb, [0, 31, 32])
    pool.anneal("abrupt_cool", 2.0 * (na + nb), 0.0, 6 * (na + nb), 10 ** 9, seeds, max_inflight=1)
    check_invariants(pool, edges, na, nb, [0, 32])
    e2 = pool.entropy()
    assert (e2 < e1).all()
    pool2 = host.ChainPool(graph, np.tile(lab0, (C, 1)), ka, kb, 1.0)
    pool2.set_option("kernel", option)
    pool2.set_precision(precision)
    pool2.randomize(seeds)
    f1 = pool2.entropy()
    pool2.anneal("constant", 1.0, 0.0, 2 * (na + nb), 10 ** 9, seeds, max_inflight=1)
    f2 = pool2.entropy()
    for c in (0, 32):
        assert abs((f2[c] - f1[c]) - pool2.entropy_accum(c)) <= 1e-6 * abs(f1[c])


def test_ka_kb_grid_of_chains(host):
    """BASELINE configs[3] in miniature: a det_k_bisbm-style (Ka, Kb) grid x restarts in ONE pool
    (heterogeneous K per chain), abrupt_cool annealing; the description length must be lowest near
    the planted (4, 6)."""
    g = load_golden("c2_const_k46")
    na, nb, edges = g["na"], g["nb"], g["edges"]
    grid = [(a, b) for a in (2, 3, 4, 6, 8) for b in (2, 4, 6, 8, 12)]
    restarts = 2
    kas = np.array([a for a, b in grid for _ in range(restarts)], dtype=np.uint32)
    kbs = np.array([b for a, b in grid for _ in range(restarts)], dtype=np.uint32)
    labs = np.stack([np.concatenate([np.arange(na) * a // na, a + np.arange(nb) * b // nb]) for a, b in zip(kas, kbs)]).astype(np.uint32)
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, labs, kas, kbs, 1.0)
    seeds = np.arange(len(kas), dtype=np.uint64) + 1
    pool.randomize(seeds)
    n = na + nb
    pool.anneal("abrupt_cool", 60.0 * n, 0.0, 120 * n, 10 ** 9, seeds)
    check_invariants(pool, edges, na, nb, [0, 13, len(kas) - 1])
    ent = pool.entropy().reshape(len(grid), restarts).min(1)
    best = grid[int(np.argmin(ent))]
    print("grid minimum at", best, "entropy", ent.min())
    assert abs(best[0] - 4) <= 2 and abs(best[1] - 6) <= 2


def test_isolated_nodes_hub_vertex_and_many_chain_groups(host):
    """Edge cases of the parallel kernel: degree-0 vertices (proposal is uniform over all K blocks,
    accu_r = 1), a hub of degree > 255 (16-bit histogram bins, neighbour ids reloaded every 32), and
    more chain groups than SMs (one CTA per group, whole half sweep in one launch)."""
    g = load_golden("isolated")
    na, nb, edges = g["na"], g["nb"], g["edges"]
    graph = host.Graph(edges, na, nb)
    C = 32 * 160 + 7
    pool = host.ChainPool(graph, np.tile(g["labels0"], (C, 1)), g["ka"], g["kb"], 0.1)
    seeds = np.arange(C, dtype=np.uint64) + 3
    pool.randomize(seeds)
    acc, sw = pool.anneal("constant", 1.0, 0.0, 50 * (na + nb), 10 ** 9, seeds)
    assert (sw == 50).all() and (acc > 0).all()
    check_invariants(pool, edges, na, nb, [0, 31, 32, 5000, C - 1])
    lab = pool.labels()
    iso = np.setdiff1d(np.arange(na + nb), np.unique(edges))
    assert len(iso) > 0 and any(len(np.unique(lab[:, v])) > 1 for v in iso)  # isolated nodes do move

    rng = np.random.default_rng(5)
    na2 = nb2 = 400
    e = np.stack([rng.integers(0, na2, 3000), na2 + rng.integers(0, nb2, 3000)], 1)
    hub = np.stack([np.zeros(300, dtype=np.int64), na2 + rng.integers(0, nb2, 300)], 1)   # vertex 0: degree >= 300
    edges2 = np.concatenate([e, hub]).astype(np.uint32)
    graph2 = host.Graph(edges2, na2, nb2)
    assert graph2.max_degree > 255
    lab0 = np.concatenate([np.arange(na2) % 5, 5 + np.arange(nb2) % 4]).astype(np.uint32)
    pool2 = host.ChainPool(graph2, np.tile(lab0, (64, 1)), 5, 4, 1.0)
    s2 = np.arange(64, dtype=np.uint64) + 9
    pool2.randomize(s2)
    f1 = pool2.entropy()
    pool2.anneal("constant", 1.0, 0.0, 20 * (na2 + nb2), 10 ** 9, s2, max_inflight=1)
    check_invariants(pool2, edges2, na2, nb2, [0, 63])
    f2 = pool2.entropy()
    for c in (0, 63):
        assert abs((f2[c] - f1[c]) - pool2.entropy_accum(c)) <= 1e-6 * abs(f1[c])


def test_k32_specialised_kernel(host):
    """Ka = Kb = 32 takes the compile-time-stride instantiation of the sweep kernel (the bench workload):
    same invariants, and sequential chains are exact."""
    na = nb = 6000
    ka = kb = 32
    edges = planted(na, nb, ka, kb, 150000, 17)
    graph = host.Graph(edges, na, nb)
    C = 96
    pool = host.ChainPool(graph, np.tile(planted_labels(na, nb, ka, kb), (C, 1)), ka, kb, 1.0)
    seeds = np.arange(C, dtype=np.uint64) + 41
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 5 * (na + nb), 10 ** 9, seeds)
    check_invariants(pool, edges, na, nb, [0, 50, 95])
    f1 = pool.entropy()
    d0 = np.array([pool.entropy_accum(c) for c in (0, 95)])
    pool.anneal("constant", 1.0, 0.0, 2 * (na + nb), 10 ** 9, seeds + np.uint64(1000), max_inflight=1)
    f2 = pool.entropy()
    for k, c in enumerate((0, 95)):
        assert abs((f2[c] - f1[c]) - (pool.entropy_accum(c) - d0[k])) <= 1e-6 * abs(f1[c])
    check_invariants(pool, edges, na, nb, [0, 95])


def test_fp32_kernel_is_selected_and_matches_double_statistically(host):
    """The default parallel path evaluates a move in double (sweep2_kernel<double>); BISBM_PRECISION_FP32 switches
    the same pool to the fp32 instantiation.  The two use different arithmetic on the same draws, so the comparison is
    statistical: final description length and acceptance of 128 + 128 strictly sequential chains on the oracle-parity
    workload."""
    from scipy.stats import ks_2samp
    g = load_golden("c2_const_k46")
    na, nb, edges, mb = g["na"], g["nb"], g["edges"], g["labels0"]
    n = na + nb
    graph = host.Graph(edges, na, nb)
    R = 128
    out = {}
    for prec, want_kernel in (("fp32", 2), ("fp64", 3)):
        pool = host.ChainPool(graph, np.tile(mb, (R, 1)), 4, 6, 1.0)
        pool.set_precision(prec)
        seeds = np.arange(R, dtype=np.uint64) + 4242
        pool.randomize(seeds)
        acc, _ = pool.anneal("abrupt_cool", 1e5, 0.0, 200 * n, 10 ** 9, seeds, max_inflight=1)
        kern, wpc, cpg, sl = pool.sweep_info()
        assert kern == want_kernel and cpg == 1
        check_invariants(pool, edges, na, nb, [0, R - 1])
        out[prec] = (pool.entropy(), acc)
    p_ent = ks_2samp(out["fp32"][0], out["fp64"][0]).pvalue
    p_acc = ks_2samp(out["fp32"][1], out["fp64"][1]).pvalue
    print("fp32 vs fp64: entropy %.1f / %.1f (KS p=%.3f), acceptance %.4f / %.4f (KS p=%.3f)" % (
        out["fp32"][0].mean(), out["fp64"][0].mean(), p_ent, out["fp32"][1].mean(), out["fp64"][1].mean(), p_acc))
    assert p_ent > 0.01 and p_acc > 0.01


def test_full_size_c3_properties(host):
    """BASELINE configs[2] at FULL size (1M nodes / 10M edges, Ka = Kb = 32, 256 chains on one GPU) through
    size-independent properties: after sweeps of the default plan (sweep2_kernel<double>, 18 CTAs per chain group, slices of
    n/64) the device counts of any chain equal a from-scratch rebuild from its labels (m_rs, e_r, n_r, eta -- so no
    delta was lost or applied twice across the ~130 slice launches of a sweep), every block stays non-empty, the
    accumulated dS tracks the true change of the description length, and chains started from different
    randomisations stay different."""
    na = nb = 500000
    ka = kb = 32
    edges = planted(na, nb, ka, kb, 10_000_000, 0)
    graph = host.Graph(edges, na, nb)
    C = 256
    lab0 = planted_labels(na, nb, ka, kb)
    pool = host.ChainPool(graph, np.broadcast_to(lab0, (C, na + nb)), ka, kb, 1.0)
    seeds = np.arange(C, dtype=np.uint64) + 7
    pool.randomize(seeds)
    e1 = pool.entropy()
    acc, sw = pool.anneal("constant", 1.0, 0.0, 2 * (na + nb), 10 ** 18, seeds)
    kern, wpc, cpg, sl = pool.sweep_info()
    # slices: at most n/64 vertices (the default staleness bound) and a whole number of vertices per warp
    assert kern == 3 and cpg * (C // 32) <= 148 and na // 64 - cpg * wpc < sl <= na // 64 and sl % (cpg * wpc) == 0
    assert (sw == 2).all() and (acc > 0.5).all() and (acc < 1.0).all()
    check_invariants(pool, edges, na, nb, [0, 131, 255])
    e2 = pool.entropy()
    for c in (0, 131, 255):
        d_true, d_acc = e2[c] - e1[c], pool.entropy_accum(c)
        assert abs(d_true - d_acc) <= 0.10 * abs(d_true) + 50.0
    l0, l1 = pool.labels(0), pool.labels(255)
    assert (l0 != l1).mean() > 0.5
    ms, launches, moves = pool.last_timing()
    assert moves == 2 * (na + nb) * C
    print("C3 full size: %.3e moves/s (device events), acceptance %.4f" % (moves / (ms * 1e-3), acc.mean()))


@pytest.mark.parametrize("schedule,p0,p1", [("exponential", 2.0, 0.999), ("linear", 1.5, 0.0003), ("logarithmic", 1.0, 2.0)])
def test_cooling_schedules_match_oracle_on_southern_women(host, schedule, p0, p1):
    """BASELINE configs[0] (southernWomen, K = 5 + 5, eps = 1e-3) under the three time-dependent cooling schedules:
    128 oracle chains vs 128 GPU chains (n = 32, so every GPU chain is strictly sequential), randomised starts,
    150 sweeps.  Two-sample KS on the final description length and on the acceptance ratio: the temperature of
    every step, the T -> 0 handling and the accept test have to agree with the reference's anneal().
    On 32 nodes the ORDER in which a sweep visits the vertices matters for an annealing run (the temperature is a
    function of the step index): the reference shuffles all vertices together, parallel mode visits the type-a vertices
    first, then the type-b ones (documented deviation).  The strict comparison (p > 0.01) is therefore against the oracle
    run with that visiting order (ora_anneal_alternating: everything else is the reference's anneal); against the
    reference's own order the deviation must stay small (p > 0.001, difference of the means < 0.3 standard deviations)."""
    from scipy.stats import ks_2samp
    g = load_golden("c1_seed1")
    na, nb, edges, lab0 = g["na"], g["nb"], g["edges"], g["labels0"]
    n = na + nb
    ka, kb = int(g["ka"]), int(g["kb"])
    R, sweeps = 128, 150
    res = {}
    for alt in (True, False):
        ent_o, acc_o = [], []
        for s in range(R):
            o = port.PortChain(n, na, nb, edges, lab0, ka, kb, 1e-3, 5000 + s, 6000 + s)
            o.init(True)
            acc_o.append(o.anneal(schedule, p0, p1, sweeps * n, 10 ** 9, alternate=alt))
            ent_o.append(o.entropy())
        res[alt] = (np.array(ent_o), np.array(acc_o))
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(lab0, (R, 1)), ka, kb, 1e-3)
    seeds = np.arange(R, dtype=np.uint64) + 99
    pool.randomize(seeds)
    acc_g, sw = pool.anneal(schedule, p0, p1, sweeps * n, 10 ** 9, seeds)
    assert (sw == sweeps).all()
    check_invariants(pool, edges, na, nb, [0, R - 1])
    ent_g = pool.entropy()
    out = {}
    for alt in (True, False):
        ent_o, acc_o = res[alt]
        out[alt] = (ks_2samp(ent_o, ent_g).pvalue, ks_2samp(acc_o, acc_g).pvalue)
        print("%s vs oracle (%s order): entropy oracle %.2f+-%.2f gpu %.2f+-%.2f p=%.3f | acceptance %.4f %.4f p=%.3f" % (
            schedule, "type-alternating" if alt else "reference", np.mean(ent_o), np.std(ent_o), np.mean(ent_g), np.std(ent_g),
            out[alt][0], np.mean(acc_o), np.mean(acc_g), out[alt][1]))
    assert out[True][0] > 0.01 and out[True][1] > 0.01
    assert out[False][0] > 0.001 and out[False][1] > 0.001
    assert abs(np.mean(res[False][0]) - np.mean(ent_g)) < 0.3 * np.std(res[False][0])


@pytest.mark.parametrize("ka,kb", [(10, 120), (6, 200), (5, 200), (36, 36), (38, 37)])
def test_asymmetric_and_borderline_k(host, ka, kb):
    """K shapes around the limits of shared-memory staging: the kernel (staged counts / counts in L2) is chosen once per
    call for BOTH half sweeps -- the two keep different label arrays current, so a per-type choice would lose moves --
    and the histogram commit never leaves a lane's bins.  Counts must equal a rebuild from the labels."""
    na = nb = 3000
    edges = planted(na, nb, 6, 6, 60000, 23)
    graph = host.Graph(edges, na, nb)
    C = 40
    lab0 = np.concatenate([np.arange(na) % ka, ka + np.arange(nb) % kb]).astype(np.uint32)
    pool = host.ChainPool(graph, np.tile(lab0, (C, 1)), ka, kb, 1.0)
    seeds = np.arange(C, dtype=np.uint64) + 61
    pool.randomize(seeds)
    acc, sw = pool.anneal("constant", 1.0, 0.0, 3 * (na + nb), 10 ** 9, seeds)
    assert (sw == 3).all() and (acc > 0).all()
    check_invariants(pool, edges, na, nb, [0, 31, 39])
    kern = pool.sweep_info()[0]
    assert kern in (3, 5)   # sweep2_kernel<double>: staged counts (fewer warps when shared memory is short) or counts in L2
    f1 = pool.entropy()
    d0 = np.array([pool.entropy_accum(c) for c in (0, 39)])
    pool.anneal("constant", 1.0, 0.0, 1 * (na + nb), 10 ** 9, seeds + np.uint64(7), max_inflight=1)
    check_invariants(pool, edges, na, nb, [0, 39])
    f2 = pool.entropy()
    for k, c in enumerate((0, 39)):
        assert abs((f2[c] - f1[c]) - (pool.entropy_accum(c) - d0[k])) <= 1e-6 * abs(f1[c])


def test_two_handles_on_two_devices_or_one(host):
    """Function attributes (dynamic shared memory limit) are per device and tracked per handle: a second handle, on
    another GPU when the box has one, runs its first big-shared-memory launch without help from the first."""
    import ctypes as C_
    L = host.load_library()
    import torch
    ndev = torch.cuda.device_count()
    na = nb = 2000
    edges = planted(na, nb, 32, 32, 40000, 3)
    pools = []
    for dev in range(min(ndev, 2) if ndev > 1 else 1):
        for rep in range(2 if ndev == 1 else 1):
            graph = host.Graph(edges, na, nb, device=dev)
            pool = host.ChainPool(graph, np.tile(planted_labels(na, nb, 32, 32), (32, 1)), 32, 32, 1.0)
            seeds = np.arange(32, dtype=np.uint64) + 1
            pool.randomize(seeds)
            pool.anneal("constant", 1.0, 0.0, 2 * (na + nb), 10 ** 9, seeds)
            check_invariants(pool, edges, na, nb, [0, 31])
            pools.append(pool)
    assert len(pools) >= 1


def test_u8_labels_round_trip_and_rebuild_skip(host):
    """The 8-bit label entry points carry the same labels as the 32-bit ones; handing back exactly the labels the handle
    holds keeps its counts (no rebuild), a single changed label rebuilds them."""
    g = load_golden("c2_const_k46")
    na, nb, edges = g["na"], g["nb"], g["edges"]
    graph = host.Graph(edges, na, nb)
    C = 37
    pool = host.ChainPool(graph, np.tile(g["labels0"], (C, 1)), 4, 6, 1.0)
    seeds = np.arange(C, dtype=np.uint64) + 5
    pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 5 * (na + nb), 10 ** 9, seeds)
    l32 = pool.labels()
    l8 = pool.labels(out=np.zeros((C, na + nb), dtype=np.uint8))
    assert l8.dtype == np.uint8 and (l8 == l32).all()
    acc0 = pool.entropy_accum(3)
    pool.set_labels(l8)                      # unchanged: counts kept
    check_invariants(pool, edges, na, nb, [0, 36])
    l8b = l8.copy()
    l8b[36, 999] = 4 + (l8b[36, 999] - 4 + 1) % 6
    pool.set_labels(l8b)                     # one label changed: counts rebuilt
    check_invariants(pool, edges, na, nb, [0, 36])
    assert (pool.labels(36) == l8b[36]).all()
    pool.anneal("constant", 1.0, 0.0, 2 * (na + nb), 10 ** 9, seeds)
    check_invariants(pool, edges, na, nb, [0, 36])
    bad = l8b.copy(); bad[1, 0] = 7          # a type-b block id on a type-a node
    with pytest.raises(host.BisbmError):
        pool.set_labels(bad)


def test_label_arrays_stay_coherent(host):
    """The handle keeps two label arrays (canonical i32, u8 shadow) and refreshes one from the other on demand.  Whatever
    the order of 8-bit / 32-bit imports, parallel sweeps, replay moves and exports, every view shows the same labels and
    the counts equal a rebuild from them.  n is a multiple of 16 (the 16-byte paths of the 8-bit import / export) and
    large enough for the staged count builder."""
    na = nb = 2560
    ka, kb = 6, 9
    edges = planted(na, nb, ka, kb, 40000, 3)
    graph = host.Graph(edges, na, nb)
    C = 45
    lab0 = planted_labels(na, nb, ka, kb)
    rng = np.random.default_rng(1)
    labs = np.tile(lab0, (C, 1)).astype(np.uint8)
    for c in range(C):      # every chain different
        idx = rng.integers(0, na, 200)
        labs[c, idx] = rng.integers(0, ka, 200)
        idx = na + rng.integers(0, nb, 200)
        labs[c, idx] = ka + rng.integers(0, kb, 200)
    pool = host.ChainPool(graph, labs.astype(np.uint32), ka, kb, 1.0)
    pool.set_labels(labs)                                    # 8-bit import over a 32-bit state: same labels, counts kept
    assert (pool.labels() == labs).all()
    check_invariants(pool, edges, na, nb, [0, 31, 32, 44])
    labs2 = labs.copy(); labs2[44, na + 5] = ka + (labs2[44, na + 5] - ka + 1) % kb
    pool.set_labels(labs2)                                   # 8-bit import, one label changed: counts rebuilt from the shadow
    check_invariants(pool, edges, na, nb, [0, 44])
    out8 = pool.labels(out=np.zeros((C, na + nb), dtype=np.uint8))
    assert (out8 == labs2).all() and (pool.labels() == labs2).all() and (pool.labels(44) == labs2[44]).all()
    seeds = np.arange(C, dtype=np.uint64) + 9
    pool.anneal("constant", 1.0, 0.0, 3 * (na + nb), 10 ** 9, seeds)     # sweep2: writes the shadow only
    a8 = pool.labels(out=np.zeros((C, na + nb), dtype=np.uint8))
    a32 = pool.labels()
    assert (a8 == a32).all() and not (a32 == labs2).all()
    check_invariants(pool, edges, na, nb, [0, 17, 44])
    pool.replay_init(3, 77)                                  # replay: reads and writes the canonical labels of chain 3
    pool.replay_anneal(3, "constant", 1.0, 0.0, 2 * (na + nb), 10 ** 9)
    b32 = pool.labels()
    assert not (b32[3] == a32[3]).all() and (np.delete(b32, 3, 0) == np.delete(a32, 3, 0)).all()
    pool.anneal("constant", 1.0, 0.0, 2 * (na + nb), 10 ** 9, seeds)     # the shadow must have picked up the replay moves
    check_invariants(pool, edges, na, nb, [3, 4, 44])
    c8 = pool.labels(out=np.zeros((C, na + nb), dtype=np.uint8))
    pool.set_labels(c8)                                      # unchanged 8-bit labels: shortcut
    pool.randomize(seeds)                                    # reads the canonical labels
    check_invariants(pool, edges, na, nb, [0, 3, 44])
    assert (np.sort(pool.labels(7)[:na]) == np.sort(c8[7, :na])).all()   # a permutation within the type
    bad = c8.copy(); bad[2, na] = 0                          # a type-a block id on a type-b node
    with pytest.raises(host.BisbmError):
        pool.set_labels(bad)


def test_grid_search_driver_finds_the_planted_k(host):
    """BASELINE configs[3] through the in-process (Ka, Kb) search driver (bisbm_grid_search): a grid around the planted
    (4, 6) of bisbm-1000 plus large-K points (other K classes: separate pools over the shared graph -- (20, 24) staged at
    32 + 32, (40, 44) counts in L2, (48, 4) and (3, 64) staged with asymmetric strides), 4 restarts each, abrupt_cool annealing; the description-length minimum must land on or next to the planted point, and the
    returned best partition must score the reported minimum."""
    g = load_golden("c2_const_k46")
    na, nb, edges = g["na"], g["nb"], g["edges"]
    n = na + nb
    graph = host.Graph(edges, na, nb)
    points = [(a, b) for a in (2, 3, 4, 5, 6, 8) for b in (3, 4, 6, 8, 12)] + [(20, 24), (40, 44), (48, 4), (3, 64)]
    ent, acc, best, lab, stats = host.grid_search(graph, points, 4, 1.0, "abrupt_cool", 60.0 * n, 0.0, 120 * n, 10 ** 9, seed=3)
    assert ent.shape == (len(points), 4) and np.isfinite(ent).all() and stats["buckets"] == 6
    bp = points[best[0]]
    print("grid minimum at", bp, "entropy", ent.min(), "stats", stats)
    assert ent[best] == ent.min() and abs(bp[0] - 4) <= 2 and abs(bp[1] - 6) <= 2
    pool = host.ChainPool(graph, lab, bp[0], bp[1], 1.0)
    assert abs(pool.entropy(0) - ent.min()) <= 1e-9 * abs(ent.min())
    assert stats["moves"] == len(points) * 4 * 120 * n
    # a second call runs in the pools the first one left on the graph handle (same streams of random numbers; the order in
    # which concurrent warps commit is not reproducible, so the numbers agree statistically, not bit for bit)
    ent2, acc2, best2, lab2, st2 = host.grid_search(graph, points, 4, 1.0, "abrupt_cool", 60.0 * n, 0.0, 120 * n, 10 ** 9, seed=3)
    bp2 = points[best2[0]]
    assert np.isfinite(ent2).all() and abs(bp2[0] - 4) <= 2 and abs(bp2[1] - 6) <= 2 and abs(ent2.min() - ent.min()) <= 0.01 * abs(ent.min())
    assert st2["buckets"] == 6 and st2["moves"] == stats["moves"]
    assert abs(host.ChainPool(graph, lab2, bp2[0], bp2[1], 1.0).entropy(0) - ent2.min()) <= 1e-9 * abs(ent2.min())
    host.grid_release(graph)
    ent3 = host.grid_search(graph, points[:4], 4, 1.0, "abrupt_cool", 60.0 * n, 0.0, 120 * n, 10 ** 9, seed=3)[0]
    assert np.isfinite(ent3).all()
    # the buckets behind it (bisbm_grid_k_class) and the per-bucket report
    assert host.grid_k_class(graph, 5, 7) == (8, 8, True) and host.grid_k_class(graph, 20, 24) == (32, 32, True)
    assert host.grid_k_class(graph, 64, 2) == (64, 16, True) and host.grid_k_class(graph, 3, 48) == (24, 48, True)
    assert host.grid_k_class(graph, 40, 44) == (64, 64, False)
    rep = stats["report"]
    assert len(rep) == 6 and sum(r["chains"] for r in rep) == 4 * len(points)
    assert {(r["KA"], r["KB"]): r["kernel"] for r in rep}[(40, 44)] == 5 and all(r["kernel"] in (3, 5) for r in rep)


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_estimate_mode_variable_k(host, precision):
    """README "estimation" mode (vary_k): blocks may empty and re-fill, the K-dependent terms of the description length
    follow the number of occupied blocks.  Strictly sequential chains: the accumulated dS must equal the change of
    entropy() (which counts occupied blocks in this mode) although blocks come and go; counts always equal a rebuild
    from the labels."""
    g = load_golden("c1_seed1")
    _estimate_mode_check(host, g["edges"], g["na"], g["nb"], g["labels0"], precision, 2 if precision == "fp32" else 3)


def test_estimate_mode_hub_round1(host):
    """The same on a graph with a hub (256 parallel edges between the first a-node and the first b-node): degree > 255
    takes the round-1 kernel (0), which must run estimate mode as well -- blocks empty at T = 2 and, for strictly
    sequential chains, the accumulated dS equals the change of entropy() counted with the occupied blocks."""
    g = load_golden("c1_seed1")
    na, nb = g["na"], g["nb"]
    hub = np.tile(np.array([[0, na]], dtype=np.uint32), (256, 1))
    edges = np.concatenate([np.asarray(g["edges"], dtype=np.uint32).reshape(-1, 2), hub])
    _estimate_mode_check(host, edges, na, nb, g["labels0"], "fp64", 0)


def _estimate_mode_check(host, edges, na, nb, labels0, precision, kernel):
    graph = host.Graph(edges, na, nb)
    C = 64
    pool = host.ChainPool(graph, np.tile(labels0, (C, 1)), 5, 5, 1.0)
    pool.set_precision(precision)
    pool.set_option("vary_k", 1)
    seeds = np.arange(C, dtype=np.uint64) + 17
    pool.randomize(seeds)
    e0 = pool.entropy()
    k0 = pool.occupied_blocks()
    assert (k0 == 5).all()
    emptied = 0
    for rnd in range(6):
        acc, sw = pool.anneal("constant", 2.0, 0.0, 30 * (na + nb), 10 ** 9, seeds + np.uint64(1000 * rnd), max_inflight=1)
        assert pool.sweep_info()[0] == kernel
        kk = pool.occupied_blocks()
        emptied += int((kk < 5).any())
        for c in (0, 31, 63):
            lab = pool.labels(c)
            m, e, nr, eta = counts_from_labels(edges, na, nb, lab, 5, 5)
            assert (pool.m(c) == m).all() and (pool.m_r(c) == e).all() and (pool.n_r(c) == nr).all() and (pool.eta(c) == eta).all()
            assert kk[c, 0] == (nr[:5] > 0).sum() and kk[c, 1] == (nr[5:] > 0).sum()
    assert emptied > 0       # at T = 2 on 32 nodes blocks do empty
    e1 = pool.entropy()
    tol = 1e-7 if precision == "fp64" else 2e-4
    for c in (0, 31, 63):
        assert abs((e1[c] - e0[c]) - pool.entropy_accum(c)) <= tol * abs(e0[c]), (c, e1[c] - e0[c], pool.entropy_accum(c))
    # concurrent moves keep the counts consistent as well
    pool.anneal("constant", 2.0, 0.0, 50 * (na + nb), 10 ** 9, seeds)
    lab = pool.labels(5)
    m, e, nr, eta = counts_from_labels(edges, na, nb, lab, 5, 5)
    assert (pool.m(5) == m).all() and (pool.n_r(5) == nr).all() and (nr >= 0).all()


def test_edge_list_text_is_parsed_on_the_device(host):
    """load_edge_list (reference src/graph_utilities.cc:20-34) on the device: the file's text goes in, the CSR that comes
    out equals the one built from the parsed arrays -- rows in file order, multi-edges kept -- for plain "a b" lines, for
    tabs / runs of blanks / CRLF / a missing final newline / skipped non-edge lines, and for a text that spans many 4 KB
    chunks with lines of every length straddling the chunk borders."""
    g = load_golden("c2_const_k46")
    na, nb, edges = g["na"], g["nb"], np.asarray(g["edges"], dtype=np.uint32).reshape(-1, 2)
    ref = host.Graph(edges, na, nb)
    rp0, col0 = ref.csr()
    plain = "".join("%d %d\n" % (a, b) for a, b in edges)
    rng = np.random.default_rng(5)
    seps = [" ", "\t", "   ", " \t ", "\t\t"]
    ends = ["\n", "\r\n", " \n", "\t\r\n"]
    messy = ["# a comment line\n", "\n", "   \n"]
    for i, (a, b) in enumerate(edges):
        messy.append("%s%d%s%d%s" % (["", " ", "\t"][i % 3], a, seps[int(rng.integers(len(seps)))], b, ends[int(rng.integers(len(ends)))]))
        if i % 97 == 0:
            messy.append(["\n", "nodes follow\n", "\t\n"][i % 3])
    messy = "".join(messy)
    messy = messy[:-1] if messy.endswith("\n") else messy          # no newline at the end of the file
    assert len(plain) > 3 * 4096
    for text in (plain, messy, messy.encode()):
        gt = host.Graph(text, na, nb)
        assert gt.n_edges == len(edges)
        rp, col = gt.csr()
        assert (rp == rp0).all() and (col == col0).all()
    # the same chains on both graphs score the same description length
    lab = np.tile(g["labels0"], (2, 1))
    assert (host.ChainPool(host.Graph(messy, na, nb), lab, 4, 6, 1.0).entropy() == host.ChainPool(ref, lab, 4, 6, 1.0).entropy()).all()
    # a missing second number reads as 0; ids that do not fit 32 bits, out-of-range ids and same-type edges are refused
    for bad in ("0 99999999999\n", "0 %d\n" % (na + nb), "0 1\n"):
        with pytest.raises(host.BisbmError):
            host.Graph(bad, na, nb)
    empty = host.Graph("", na, nb)
    assert empty.n_edges == 0


def test_grid_search_initial_partitions_equal_the_two_step_form(host):
    """bisbm_grid_search writes its initial partitions (equal-size blocks in node order -- the reference's `-n` with equal
    sizes -- then --randomize with the chain's seed) in ONE pass straight into the 8-bit label shadow.  With duration 0 the
    scores it returns are those of the initial partitions: they must be the scores of the same partitions made the long way
    (labels from the host, ChainPool.randomize with the same seed)."""
    g = load_golden("c2_const_k46")
    na, nb, edges = g["na"], g["nb"], g["edges"]
    graph = host.Graph(edges, na, nb)
    points, restarts, seed = [(4, 6), (3, 5), (7, 2)], 3, 7
    ent, acc, best, lab, stats = host.grid_search(graph, points, restarts, 1.0, "abrupt_cool", 0.0, 0.0, 0, 10 ** 9, seed=seed)
    assert stats["moves"] == 0
    v = np.arange(na + nb)
    for p, (a, b) in enumerate(points):
        lab0 = np.where(v < na, v * a // na, a + (v - na) * b // nb).astype(np.uint32)
        for q in range(restarts):
            s = (seed * 0x9E3779B97F4A7C15 + (p << 20) + q + 1) % (1 << 64)
            pool = host.ChainPool(graph, lab0[None, :], a, b, 1.0)
            pool.randomize(np.array([s], dtype=np.uint64))
            assert abs(pool.entropy(0) - ent[p, q]) <= 1e-12 * abs(ent[p, q]), (p, q, pool.entropy(0), ent[p, q])
            if (p, q) == best:
                assert (pool.labels(0) == lab).all()
