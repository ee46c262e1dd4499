"""The host restatement of what the sweep kernels sample (tests/stationary_models.py) against the oracle, on every labeling
of the enumerable models: S equals ora_entropy, the proposal rule's q(y->x) / q(x->y) equals transition_ratio's accu_r
and the kernels' one-pass Hastings factor, and the Metropolis-Hastings rule with these factors is in detailed balance with
pi ~ exp(-S/T) -- in fixed-K and in estimate mode (vary_k), whose parity the reference leaves unpinned.  No GPU."""
import math

import numpy as np
import pytest

import stationary_models as sm
from oracle import port

CONFIGS = [("A", (2, 3)), ("A", (3, 2)), ("B", (2, 2)), ("B256", (2, 2))]


def make(name):
    return sm.model_a() if name == "A" else sm.model_b(256 if name == "B256" else 255)


def oracle_chain(model, lab, ka, kb, eps=1.0):
    c = port.PortChain(model.n, model.na, model.nb, model.edges, lab, ka, kb, eps, 1)
    c.init(False)
    return c


def compact(model, lab, ka):
    """relabel the occupied blocks of each type to 0 .. k-1 (in order) -> (labels, k_a, k_b)"""
    lab = np.asarray(lab, dtype=np.int64)
    ua, ub = sorted(set(lab[:model.na].tolist())), sorted(set(lab[model.na:].tolist()))
    mp = {b: i for i, b in enumerate(ua)}
    mp.update({b: len(ua) + i for i, b in enumerate(ub)})
    return np.array([mp[int(x)] for x in lab], dtype=np.uint32), len(ua), len(ub)


def test_enumeration_sizes():
    a, b = sm.model_a(), sm.model_b()
    assert len(sm.states(a, 2, 3)) == len(sm.states(a, 3, 2)) == 504
    assert len(sm.states(a, 2, 3, True)) == len(sm.states(a, 3, 2, True)) == 1296
    assert len(sm.states(b, 2, 2)) == 84 and len(sm.states(b, 2, 2, True)) == 128
    assert (a.deg[[3, 7]] == 0).all() and a.E == 12 and len(a.mult) == 8
    assert list(b.deg[:3]) == [255, 33, 1] and b.deg[3:].max() <= 255
    assert list(sm.model_b(256).deg[:3]) == [256, 33, 1] and sm.model_b(256).deg[3:].max() <= 255
    # the reference's q table in exact integers, against the oracle's log-domain table
    tab = port.log_q_table(300, 8)
    for n in range(1, 301):
        for k in range(1, 9):
            want = tab[n, k]
            assert (sm.partitions(n, k) == 0) if np.isinf(want) else abs(math.log(sm.partitions(n, k)) - want) <= 1e-12 * max(1.0, want)
    assert sm.partitions(12, 3) == 14 and sm.partitions(289, 1) == 1 and sm.partitions(5, 0) == 0


@pytest.mark.parametrize("name,k", CONFIGS)
def test_entropy_equals_oracle(name, k):
    """fixed K: S of every labeling equals ora_entropy to 1e-12 relative; estimate mode: S of every labeling (empty blocks
    allowed) equals ora_entropy of the compacted labeling with K = the occupied blocks"""
    model = make(name)
    ka, kb = k
    for lab in sm.states(model, ka, kb):
        S, So = sm.entropy(model, lab, ka, kb), oracle_chain(model, lab, ka, kb).entropy()
        assert abs(S - So) <= 1e-12 * abs(So), (name, lab, S, So)
    n_empty = 0
    for lab in sm.states(model, ka, kb, vary_k=True):
        cl, ca, cb = compact(model, lab, ka)
        n_empty += (ca, cb) != (ka, kb)
        S, So = sm.entropy(model, lab, ka, kb, vary_k=True), oracle_chain(model, cl, ca, cb).entropy()
        assert abs(S - So) <= 1e-12 * abs(So), (name, lab, S, So)
        if (ca, cb) == (ka, kb):
            assert S == sm.entropy(model, lab, ka, kb)
    assert n_empty > 0


@pytest.mark.parametrize("eps", [1.0, 0.1])
@pytest.mark.parametrize("name,k", CONFIGS)
def test_hastings_factor_is_the_proposal_ratio(name, k, eps):
    """fixed K, every single move x -> y: log(q(y->x) / q(x->y)) of the proposal rule equals transition_ratio's log accu_r
    (oracle) and the kernels' one-pass restatement, and the oracle's dS equals S(y) - S(x)"""
    model = make(name)
    ka, kb = k
    n = 0
    for x in sm.states(model, ka, kb):
        ora = oracle_chain(model, x, ka, kb, eps)
        Sx = sm.entropy(model, x, ka, kb)
        _, _, nr, _ = sm.counts(model, x, ka, kb)
        for v, s in sm.single_moves(model, x, ka, kb):
            if nr[x[v]] == 1:
                continue                       # y has an empty block: outside the fixed-K state space
            y = x.copy()
            y[v] = s
            lq = math.log(sm.proposal_prob(model, y, ka, kb, v, int(x[v]), eps) / sm.proposal_prob(model, x, ka, kb, v, s, eps))
            dS, accu = ora.transition(v, s)
            assert abs(lq - math.log(accu)) <= 1e-12 * max(1.0, abs(lq)), (name, x, v, s, lq, math.log(accu))
            assert abs(lq - sm.kernel_hastings(model, x, ka, kb, v, s, eps)) <= 1e-12 * max(1.0, abs(lq))
            assert abs(dS - (sm.entropy(model, y, ka, kb) - Sx)) <= 1e-11 * max(1.0, abs(Sx))
            n += 1
    assert n > 0


def kernel_dS(model, ora, x, ka, kb, v, s, vary_k):
    """dS as a sweep kernel computes it: transition_ratio's terms, plus in estimate mode the prior delta when the move
    empties its block and / or opens an empty one"""
    dS, _ = ora.transition(v, s)
    if vary_k:
        _, _, nr, _ = sm.counts(model, x, ka, kb)
        dk = int(nr[s] == 0) - int(nr[x[v]] == 1)
        if dk:
            oa, ob = sm.occupied(model, x, ka)
            tb = v >= model.na
            dS += sm.prior_k_delta(model, tb, ob if tb else oa, oa if tb else ob, int(dk))
    return dS


@pytest.mark.parametrize("vary_k", [False, True])
@pytest.mark.parametrize("eps,T", [(1.0, 1.0), (0.1, 1.0), (1.0, 7.0)])
@pytest.mark.parametrize("name,k", CONFIGS)
def test_detailed_balance(name, k, eps, T, vary_k):
    """pi(x) P(x, y) = pi(y) P(y, x) (in logs, to 1e-12 relative) for every pair of labelings one move apart, with P(x, y) = q(x->y)
    min(1, exp(-dS / T) accu_r) built from the kernels' dS and Hastings factor and pi from the restated S"""
    model = make(name)
    ka, kb = k
    X = sm.states(model, ka, kb, vary_k)
    S = {int(c): sm.entropy(model, x, ka, kb, vary_k) for c, x in zip(sm.state_codes(X, ka + kb), X)}
    worst, n = 0.0, 0
    for x in X:
        ora_x = oracle_chain(model, x, ka, kb, eps)
        cx = int(sm.state_codes(x, ka + kb))
        for v, s in sm.single_moves(model, x, ka, kb):
            y = x.copy()
            y[v] = s
            cy = int(sm.state_codes(y, ka + kb))
            if cy not in S or cy < cx:
                continue                       # outside the state space (fixed K), or the pair was seen from y
            r = int(x[v])
            ora_y = oracle_chain(model, y, ka, kb, eps)
            dxy = kernel_dS(model, ora_x, x, ka, kb, v, s, vary_k)
            dyx = kernel_dS(model, ora_y, y, ka, kb, v, r, vary_k)
            assert abs(dxy + dyx) <= 1e-11 * max(1.0, abs(S[cx]))
            assert abs(dxy - (S[cy] - S[cx])) <= 1e-11 * max(1.0, abs(S[cx])), (name, x, v, s, dxy, S[cy] - S[cx])
            hxy = sm.kernel_hastings(model, x, ka, kb, v, s, eps)
            hyx = sm.kernel_hastings(model, y, ka, kb, v, r, eps)
            lhs = -S[cx] / T + math.log(sm.proposal_prob(model, x, ka, kb, v, s, eps)) + min(0.0, -dxy / T + hxy)
            rhs = -S[cy] / T + math.log(sm.proposal_prob(model, y, ka, kb, v, r, eps)) + min(0.0, -dyx / T + hyx)
            worst = max(worst, abs(lhs - rhs) / max(1.0, abs(lhs)))   # relative to the size of the log terms
            n += 1
    print("%s %s eps %g T %g vary_k %d: %d pairs, worst relative error of log pi(x)P(x,y) = log pi(y)P(y,x): %.2e" % (
        name, k, eps, T, vary_k, n, worst))
    assert n > 0 and worst <= 1e-12
