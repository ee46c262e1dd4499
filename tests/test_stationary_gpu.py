"""Every one-CTA sweep plan against the exact stationary distribution of small enumerable models (tests/stationary_models.py).

32768 chains start from exact draws of pi ~ exp(-S/T) over the labelings of their mode (fixed K: no empty block; estimate
mode, vary_k: any labeling, S with the occupied block counts), take 50 strictly sequential sweeps (max_inflight=1: exact
Metropolis-Hastings, and a one-CTA plan is deterministic, so every p-value is reproducible), and the histogram of their
final STATES must pass a chi-square test against pi.  Starting from pi makes the test independent of mixing: a kernel with
a wrong proposal draw, Hastings factor or prior term drifts towards its own fixed point.  Unlike an energy-level histogram,
the state histogram also sees a bias that keeps S but favours some labelings (a categorical scan that prefers one block)."""
import numpy as np
import pytest
from scipy.stats import chisquare

import stationary_models as sm
from helpers import counts_from_labels

pytestmark = pytest.mark.gpu

N_CHAINS = 32768
SWEEPS = 50
BIG = 2 ** 62           # steps_await that never stops the run early
P_MIN = 1e-4

# plan -> (precision, forced kernel (-1: the planner's choice), Ka = Kb = 32 count strides, kernel id that must run)
PLANS = {"staged_f64": ("fp64", -1, False, 3), "staged_f32": ("fp32", -1, False, 2),
         "k32_f64": ("fp64", -1, True, 3), "k32_f32": ("fp32", -1, True, 2),
         "l2_f64": ("fp64", 5, False, 5), "l2_f32": ("fp32", 5, False, 4),
         "round1": ("fp64", 0, False, 0), "planner": ("fp64", -1, False, None)}
SWEEP2 = ["staged_f64", "staged_f32", "k32_f64", "k32_f32", "l2_f64", "l2_f32"]

# (model, eps, T (None: from the S range), plans); every case runs in fixed-K and in estimate mode
CASES = [("A", 1.0, 1.0, SWEEP2 + ["round1"]),
         ("A", 0.1, 1.0, ["staged_f64", "round1"]),
         ("B", 1.0, None, SWEEP2 + ["round1"]),
         ("B256", 1.0, None, ["planner"])]
PARAMS = [pytest.param(m, e, T, p, vk, id="%s-eps%g-%s-%s" % (m, e, p, "vary_k" if vk else "fixed_k"))
          for m, e, T, plans in CASES for p in plans for vk in (False, True)]


def make(name):
    return sm.model_a() if name == "A" else sm.model_b(256 if name == "B256" else 255)


def k_of_chains(name):
    """per-chain (Ka, Kb): model A mixes (2, 3) and (3, 2) inside every 32-chain group, model B has Ka = Kb = 2"""
    c = np.arange(N_CHAINS)
    if name == "A":
        return np.where(c % 2 == 0, 2, 3).astype(np.uint32), np.where(c % 2 == 0, 3, 2).astype(np.uint32)
    return np.full(N_CHAINS, 2, dtype=np.uint32), np.full(N_CHAINS, 2, dtype=np.uint32)


def choose_T(S):
    """the smallest multiple of 1/4 (exact in float) at which at least 3/4 of the states expect >= 20 of the chains"""
    for T in np.arange(0.25, 1000.0, 0.25):
        if (N_CHAINS * sm.target(S, T) >= 20).mean() >= 0.75:
            return float(T)
    raise AssertionError("no temperature found")


def chi2_states(obs, exp_, ddof):
    """chi-square p-value of state counts against expected counts; states are pooled in order of increasing expectation
    until every bin expects >= 5"""
    order = np.argsort(exp_, kind="stable")
    bo, be, co, ce = [], [], 0.0, 0.0
    for o, e in zip(obs[order], exp_[order]):
        co += o
        ce += e
        if ce >= 5:
            bo.append(co); be.append(ce); co = ce = 0.0
    if ce > 0:
        bo[-1] += co; be[-1] += ce
    return chisquare(bo, be, ddof=ddof).pvalue, len(bo)


def check_invariants(pool, model, chains):
    for c in chains:
        ka, kb = int(pool.ka[c]), int(pool.kb[c])
        lab = pool.labels(c)
        assert (lab[:model.na] < ka).all() and (lab[model.na:] >= ka).all() and (lab[model.na:] < ka + kb).all()
        m, e, nr, eta = counts_from_labels(model.edges, model.na, model.nb, lab, ka, kb)
        assert (pool.m(c) == m).all() and (pool.m_r(c) == e).all() and (pool.n_r(c) == nr).all()
        assert (pool.eta(c) == eta).all()


@pytest.mark.parametrize("name,eps,T,plan,vary_k", PARAMS)
def test_stationary_distribution(host, name, eps, T, plan, vary_k):
    model = make(name)
    prec, kernel, k32, kid = PLANS[plan]
    ka, kb = k_of_chains(name)
    groups = []                                  # (ka, kb, chains, states, codes, pi)
    for a, b in sorted(set(zip(ka.tolist(), kb.tolist()))):
        X = sm.states(model, a, b, vary_k)
        S = np.array([sm.entropy(model, x, a, b, vary_k) for x in X])
        groups.append([a, b, np.flatnonzero((ka == a) & (kb == b)), X, sm.state_codes(X, 8), S])
    if T is None:
        T = choose_T(np.concatenate([g[5] for g in groups]))
    rng = np.random.default_rng(2024)
    labels = np.zeros((N_CHAINS, model.n), dtype=np.uint32)
    for g in groups:
        g[5] = sm.target(g[5], T)
        labels[g[2]] = g[3][rng.choice(len(g[3]), size=len(g[2]), p=g[5])]

    graph = host.Graph(model.edges, model.na, model.nb)
    if k32:
        graph.set_option("reserve_ka", 32)       # count strides of 32 + 32: the sweep2_kernel<R, 32, TYPE> specialisations
        graph.set_option("reserve_kb", 32)
    pool = host.ChainPool(graph, labels, ka, kb, eps)
    pool.set_precision(prec)
    pool.set_option("kernel", kernel)
    pool.set_option("vary_k", int(vary_k))
    seeds = np.arange(N_CHAINS, dtype=np.uint64) * 2654435761 + 99
    pool.anneal("constant", T, 0.0, SWEEPS * model.n, BIG, seeds, max_inflight=1)
    info = pool.sweep_info()
    assert info[0] == (0 if name == "B256" else kid), info
    assert info[2] == 1                          # one CTA per chain group

    out = pool.labels()
    obs, exp_ = [], []
    for a, b, chains, X, codes, pi in groups:
        srt = np.argsort(codes)
        idx = np.searchsorted(codes[srt], sm.state_codes(out[chains], 8))
        idx = np.minimum(idx, len(codes) - 1)
        assert (codes[srt][idx] == sm.state_codes(out[chains], 8)).all(), "a chain left the state space of its mode"
        obs.append(np.bincount(srt[idx], minlength=len(X)).astype(np.float64))
        exp_.append(len(chains) * pi)
    p, bins = chi2_states(np.concatenate(obs), np.concatenate(exp_), len(groups) - 1)
    moved = (out != labels).any(1).mean()
    print("stationary %s eps %g T %g %s vary_k %d: kernel %d, p %.4g (%d bins), %.3f of the chains moved" % (
        name, eps, T, plan, vary_k, info[0], p, bins, moved))
    check_invariants(pool, model, [0, 1, 33, N_CHAINS - 1])
    assert moved > 0.1                           # (a kernel that never moves would pass the chi-square)
    assert p > P_MIN


@pytest.mark.parametrize("vary_k", [False, True])
@pytest.mark.parametrize("name,k", [("A", (2, 3)), ("A", (3, 2)), ("B", (2, 2)), ("B256", (2, 2))])
def test_entropy_kernel_on_every_labeling(host, name, k, vary_k):
    """entropy_kernel on a pool holding every labeling of the mode equals the host restatement of S to 1e-12 relative
    (estimate mode: the prior terms with the occupied block counts)"""
    model = make(name)
    X = sm.states(model, k[0], k[1], vary_k)
    pool = host.ChainPool(host.Graph(model.edges, model.na, model.nb), X, k[0], k[1], 1.0)
    pool.set_option("vary_k", int(vary_k))
    got = pool.entropy()
    want = np.array([sm.entropy(model, x, k[0], k[1], vary_k) for x in X])
    assert (np.abs(got - want) <= 1e-12 * np.abs(want)).all(), np.abs(got - want).max()
    if vary_k:
        occ = np.array([sm.occupied(model, x, k[0]) for x in X])
        assert (pool.occupied_blocks() == occ).all()
