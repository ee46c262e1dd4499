"""Parity of the parallel sweep AT THE BENCHMARKED OPERATING POINT, and of its device arithmetic.

* bisbm_parallel_transition runs ONE forced proposal through the sweep kernel's own device code (sweep2_kernel in
  KAT mode: same staging, same neighbour pass, same dS assembly) and is compared with the reference's
  transition_ratio known answers (tests/golden/*.npz kat_* vectors, generated from the unmodified reference build):
  double 1e-9 relative, float 2e-5 absolute -- including the out-of-range completions (small blocks: exact log q
  table and Stirling form) and, on the mid-size graph, the per-block log q expansions.
* On a mid-size planted graph (40k + 40k nodes, 600k edges, K = 8 + 8: the oracle is still feasible, the GPU already
  takes the SLICED MULTI-CTA plan of the benchmark: 8 chain groups x 18 CTAs, default in-flight bound) 256 GPU chains
  are compared with 128 oracle chains (tests/golden/parity_mid.npz) by two-sample KS tests on the final description
  length, the acceptance ratio and the NMI against the planted partition; max_inflight = 1 (strictly sequential
  chains) is the control.
"""
import hashlib
import json

import numpy as np
import pytest

from conftest import load_golden
from helpers import nmi, planted, planted_labels

pytestmark = pytest.mark.gpu

KAT_GOLDENS = ["c1_seed1", "c1_seed42", "c2_abrupt", "c2_const_k46", "big_blocks", "isolated"]


def _kat_check(pool, chain, kv, ks, kd, ka, lab, precision):
    worst_ds, worst_la, checked = 0.0, 0.0, 0
    for v, s, dS, ar in zip(kv, ks, kd, ka):
        d, la = pool.parallel_transition(chain, int(v), int(s))
        if np.isinf(dS):
            assert np.isinf(d) and d > 0
            continue
        if s == lab[v]:
            assert d == 0.0 and la == 0.0     # r == s: dS = 0, accu_r = 1
            continue
        if precision == "fp64":
            assert abs(d - dS) <= 1e-9 * max(1.0, abs(dS)), (v, s, d, dS)
            assert abs(la - np.log(ar)) <= 1e-9 * max(1.0, abs(np.log(ar))), (v, s, la, np.log(ar))
        else:
            assert abs(d - dS) <= 2e-5 * max(1.0, abs(dS) / 8.0), (v, s, d, dS)
            assert abs(la - np.log(ar)) <= 2e-5 * max(1.0, abs(np.log(ar))), (v, s, la, np.log(ar))
        worst_ds = max(worst_ds, abs(d - dS) / max(1.0, abs(dS)))
        worst_la = max(worst_la, abs(la - np.log(ar)))
        checked += 1
    return worst_ds, worst_la, checked


@pytest.mark.parametrize("counts", ["staged", "l2", "staged_k32"])
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("name", KAT_GOLDENS)
def test_parallel_kernel_transition_kats(host, name, precision, counts):
    g = load_golden(name)
    na, nb = g["na"], g["nb"]
    graph = host.Graph(g["edges"], na, nb)
    C = 35     # the chain under test sits in the second chain group, next to padding lanes
    pool = host.ChainPool(graph, np.tile(g["init_labels"], (C, 1)), int(g["ka"]), int(g["kb"]), float(g["eps"]))
    pool.set_precision(precision)
    if counts == "l2":
        pool.set_option("kernel", 5)      # sweep2_kernel<.., STAGED = false>: the large-K form of the same kernel
    if counts == "staged_k32":
        # count strides of 32 + 32 (the chains keep their K; the extra blocks stay empty): the Ka = Kb = 32 compile-time
        # specialisations sweep2_kernel<R, 32, TYPE> that the benchmark runs
        pool.set_option("reserve_ka", 32)
        pool.set_option("reserve_kb", 32)
        pool.set_labels(np.tile(g["init_labels"], (C, 1)))
    w1, w2, n = _kat_check(pool, 33, g["kat_v"], g["kat_s"], g["kat_dS"], g["kat_accu"], g["init_labels"], precision)
    print("%s %s: %d known answers, worst rel dS error %.2e, worst |log accu error| %.2e" % (name, precision, n, w1, w2))
    assert n > 0
    # nothing was committed
    assert (pool.labels(33) == g["init_labels"]).all()
    assert (pool.m(33) == g["init_m"]).all() and (pool.n_r(33) == g["init_n_r"]).all()


def _mid():
    fx = load_golden("parity_mid")
    na, nb, ka, kb = int(fx["na"]), int(fx["nb"]), int(fx["ka"]), int(fx["kb"])
    edges = planted(na, nb, ka, kb, int(fx["n_edges"]), int(fx["graph_seed"]))
    assert hashlib.sha1(np.ascontiguousarray(edges).tobytes()).hexdigest() == str(fx["edges_sha1"])
    return fx, na, nb, ka, kb, edges


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_parallel_kernel_transition_kats_large_blocks(host, precision):
    """Blocks with e_r = 75 000, n_r = 5 000: log q takes the asymptotic branch in the reference
    (src/support/int_part.cc:73-98) and the per-block second-order expansion in the kernel."""
    fx, na, nb, ka, kb, edges = _mid()
    lab = planted_labels(na, nb, ka, kb)
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(lab, (33, 1)), ka, kb, 1.0)
    pool.set_precision(precision)
    assert abs(pool.entropy(32) - float(fx["init_entropy"])) <= 1e-9 * float(fx["init_entropy"])
    w1, w2, n = _kat_check(pool, 32, fx["kat_v"], fx["kat_s"], fx["kat_dS"], fx["kat_accu"], lab, precision)
    print("mid graph %s: %d known answers, worst rel dS error %.2e, worst |log accu error| %.2e" % (precision, n, w1, w2))
    assert n > 100


def _run_mid(host, proto, inflight, C, precision="fp64", inflight_div=None):
    fx, na, nb, ka, kb, edges = _mid()
    n = na + nb
    lab = planted_labels(na, nb, ka, kb)
    graph = host.Graph(edges, na, nb)
    pool = host.ChainPool(graph, np.tile(lab, (C, 1)), ka, kb, 1.0)
    pool.set_precision(precision)
    if inflight_div:
        pool.set_option("inflight_div", inflight_div)
    seeds = np.arange(C, dtype=np.uint64) + 31337
    if proto in ("tr", "qu"):
        pool.randomize(seeds)
    sweeps = int(fx["sweeps_%s" % proto[:2]])
    if proto == "qu":       # abrupt_cool: hot_qu sweeps at T = 1, then greedy sweeps
        acc, sw = pool.anneal("abrupt_cool", float(int(fx["hot_qu"]) * n), 0.0, sweeps * n, 10 ** 18, seeds, max_inflight=inflight)
    else:
        acc, sw = pool.anneal("constant", 1.0, 0.0, sweeps * n, 10 ** 18, seeds, max_inflight=inflight)
    assert (sw == sweeps).all()
    ent = pool.entropy()
    labs = pool.labels()
    nm = np.array([nmi(labs[c], lab) for c in range(0, C, max(1, C // 64))])
    return fx, pool, ent, acc, nm


def _report(tag, fx, proto, ent, acc, nm, info):
    from scipy.stats import ks_2samp
    p_ent = ks_2samp(fx["%s_entropy" % proto], ent).pvalue
    p_acc = ks_2samp(fx["%s_accept" % proto], acc).pvalue
    p_nmi = ks_2samp(fx["%s_nmi" % proto], nm).pvalue
    rec = {"test": tag, "protocol": proto, "plan": {"kernel": info[0], "warps_per_cta": info[1], "ctas_per_group": info[2], "slice": info[3]},
           "oracle": {"entropy_mean": float(np.mean(fx["%s_entropy" % proto])), "entropy_sd": float(np.std(fx["%s_entropy" % proto])),
                      "accept_mean": float(np.mean(fx["%s_accept" % proto])), "nmi_mean": float(np.mean(fx["%s_nmi" % proto])), "chains": int(len(fx["%s_entropy" % proto]))},
           "gpu": {"entropy_mean": float(ent.mean()), "entropy_sd": float(ent.std()), "accept_mean": float(acc.mean()), "nmi_mean": float(nm.mean()), "chains": int(len(ent))},
           "ks_p": {"entropy": float(p_ent), "accept": float(p_acc), "nmi": float(p_nmi)}}
    print(json.dumps(rec))
    return p_ent, p_acc, p_nmi


def _accept_close(fx, proto, acc):
    """|mean acceptance - oracle mean| in units of the oracle's chain-to-chain spread."""
    return abs(float(np.mean(acc)) - float(np.mean(fx["%s_accept" % proto]))) / float(np.std(fx["%s_accept" % proto]))


def test_parity_with_oracle_at_the_benchmarked_plan_stationary(host):
    """Protocol "eq" (planted start, 30 sweeps at T = 1: samples of the STATIONARY distribution, sd of the description
    length 70 out of 5.15e6) with 256 chains = 8 chain groups x 18 CTAs x 16 warps at the default in-flight bound -- the
    plan bench.py times.  KS on description length, acceptance and NMI against 128 oracle chains, p > 0.01 each."""
    fx, pool, ent, acc, nm = _run_mid(host, "eq", 0, 256)
    info = pool.sweep_info()
    assert info[0] == 3 and info[2] > 1 and info[3] < int(fx["na"])       # staged double kernel, several CTAs per group, sliced
    p_ent, p_acc, p_nmi = _report("default_plan", fx, "eq", ent, acc, nm, info)
    assert p_ent > 0.01 and p_acc > 0.01 and p_nmi > 0.01


def test_parity_with_oracle_sequential_control_stationary(host):
    """The same comparison with max_inflight = 1 (strictly sequential chains: no stale reads at all)."""
    fx, pool, ent, acc, nm = _run_mid(host, "eq", 1, 128)
    info = pool.sweep_info()
    assert info[2] == 1
    p_ent, p_acc, p_nmi = _report("sequential_control", fx, "eq", ent, acc, nm, info)
    assert p_ent > 0.01 and p_acc > 0.01 and p_nmi > 0.01


def test_parity_with_oracle_burn_in_transient(host):
    """Protocol "tr" (randomised start, 40 sweeps at T = 1: the burn-in transient of the staleness study).  A transient
    depends on the ORDER in which a sweep visits the vertices: the reference shuffles all vertices together, parallel mode
    alternates the two types (DESIGN.md 4, known deviation).  The observable that shows it is the acceptance ratio
    averaged over the transient (0.7937 reference order, 0.7906 type-alternating order, oracle both times).  So: (i) the
    acceptance must agree (KS p > 0.01) with oracle chains run in the type-alternating order (tr_alt_*:
    ora_anneal_alternating, everything else the reference's anneal), for the benchmarked sliced plan AND for strictly
    sequential chains; (ii) benchmarked plan vs sequential chains of the same sampler must agree on acceptance and
    description length (the staleness check proper); (iii) description length and NMI agree with the reference's own
    order (p > 0.01) and the mean acceptance stays within one standard deviation of it.  Every comparison is printed as one
    JSON line (profiles/r02_kat_parity.txt)."""
    from scipy.stats import ks_2samp
    fx, pool, ent, acc, nm = _run_mid(host, "tr", 0, 256)
    info = pool.sweep_info()
    assert info[0] == 3 and info[2] > 1 and info[3] < int(fx["na"])
    p_ent, p_acc, p_nmi = _report("default_plan", fx, "tr", ent, acc, nm, info)
    a_ent, a_acc, a_nmi = _report("default_plan", fx, "tr_alt", ent, acc, nm, info)
    fx2, pool2, ent2, acc2, nm2 = _run_mid(host, "tr", 1, 128)
    assert pool2.sweep_info()[2] == 1
    q_ent, q_acc, q_nmi = _report("sequential_control", fx, "tr", ent2, acc2, nm2, pool2.sweep_info())
    b_ent, b_acc, b_nmi = _report("sequential_control", fx, "tr_alt", ent2, acc2, nm2, pool2.sweep_info())
    p_self_acc = ks_2samp(acc, acc2).pvalue
    p_self_ent = ks_2samp(ent, ent2).pvalue
    print("burn-in: plan vs sequential chains of the same sampler: KS p acceptance %.3f, description length %.3f; "
          "mean acceptance vs reference-order oracle: plan %.2f sd, sequential %.2f sd" % (
              p_self_acc, p_self_ent, _accept_close(fx, "tr", acc), _accept_close(fx, "tr", acc2)))
    assert a_acc > 0.01 and b_acc > 0.01                                                                             # (i)
    assert p_self_acc > 0.01 and p_self_ent > 0.01                                                                   # (ii)
    assert p_ent > 0.01 and p_nmi > 0.01 and q_ent > 0.01 and q_nmi > 0.01                                           # (iii)
    assert _accept_close(fx, "tr", acc) < 1.0 and _accept_close(fx, "tr", acc2) < 1.0


def test_parity_with_oracle_quench(host):
    """Protocol "qu" (randomised start, abrupt_cool: 10 sweeps at T = 1, then 10 greedy sweeps at T = 0 -- the reference's
    default schedule, src/metropolis_hasting.cc:33-37) at the benchmarked sliced plan.  This is the regime where blocks change
    by more than the validity range of their log q expansion within one half sweep (lazy refresh between slices, DESIGN.md
    3.2) and where half sweeps run as constant T = 0.  As for the burn-in transient, the path depends on the visiting order,
    so: (i) description length, NMI and acceptance agree (KS p > 0.01) with oracle chains run in the type-alternating order
    (qu_alt_*), for the sliced plan and for strictly sequential chains; (ii) sliced plan vs sequential chains of the same
    sampler agree; (iii) the mean description length stays within one oracle standard deviation of the reference-order
    oracle's."""
    from scipy.stats import ks_2samp
    if "qu_entropy" not in load_golden("parity_mid"):
        pytest.skip("fixture without the quench protocol")
    fx, pool, ent, acc, nm = _run_mid(host, "qu", 0, 256)
    info = pool.sweep_info()
    assert info[0] == 3 and info[2] > 1 and info[3] < int(fx["na"])
    p_ent, p_acc, p_nmi = _report("default_plan", fx, "qu", ent, acc, nm, info)
    a_ent, a_acc, a_nmi = _report("default_plan", fx, "qu_alt", ent, acc, nm, info)
    fx2, pool2, ent2, acc2, nm2 = _run_mid(host, "qu", 1, 128)
    assert pool2.sweep_info()[2] == 1
    _report("sequential_control", fx, "qu", ent2, acc2, nm2, pool2.sweep_info())
    b_ent, b_acc, b_nmi = _report("sequential_control", fx, "qu_alt", ent2, acc2, nm2, pool2.sweep_info())
    p_self_ent, p_self_acc = ks_2samp(ent, ent2).pvalue, ks_2samp(acc, acc2).pvalue
    off = abs(float(ent.mean()) - float(np.mean(fx["qu_entropy"]))) / float(np.std(fx["qu_entropy"]))
    print("quench: plan vs sequential chains: KS p description length %.3f, acceptance %.3f; mean description length vs "
          "reference-order oracle: %.2f sd" % (p_self_ent, p_self_acc, off))
    assert a_ent > 0.01 and a_nmi > 0.01 and a_acc > 0.01 and b_ent > 0.01 and b_nmi > 0.01 and b_acc > 0.01        # (i)
    assert p_self_ent > 0.01 and p_self_acc > 0.01                                                                   # (ii)
    assert off < 1.0                                                                                                 # (iii)
