"""Small models whose labelings can all be enumerated, and a plain-Python restatement of what a sweep kernel samples: the
description length S (blockmodel_t::entropy, reference src/blockmodel.cc:753-787), the proposal rule (single_vertex_change,
src/blockmodel.cc:613-637) and the Hastings factor (transition_ratio, src/metropolis_hasting.cc:103-192).  The target of a
chain at temperature T is pi(x) ~ exp(-S(x) / T) over the labelings of its mode: every block occupied (fixed K), or any
labeling with S counting the occupied blocks (estimate mode, vary_k).  Test infrastructure only (not product code)."""
import itertools
import math
from functools import lru_cache

import numpy as np


class Model:
    """na + nb nodes (type a first), an edge list with multiplicities, and the label-independent parts of S."""

    def __init__(self, name, na, nb, pairs):
        self.name, self.na, self.nb = name, na, nb
        self.n = na + nb
        rows = []
        for (a, b), mult in pairs:
            assert 0 <= a < na and na <= b < self.n
            rows += [(a, b)] * mult
        self.edges = np.array(rows, dtype=np.uint32).reshape(-1, 2)
        self.E = len(rows)
        self.deg = np.bincount(self.edges.ravel(), minlength=self.n).astype(np.int64)
        self.mult = [mult for _, mult in pairs]
        # -sum_v log d_v! + sum over distinct pairs log A_ij!   (the multi-edge term of entropy())
        self.base = -sum(math.lgamma(int(d) + 1) for d in self.deg) + sum(math.lgamma(m + 1) for m in self.mult if m > 1)
        self.adj = [[] for _ in range(self.n)]       # with multiplicity
        for a, b in rows:
            self.adj[a].append(b)
            self.adj[b].append(a)


def model_a():
    """4 + 4 nodes, 8 distinct edges (12 with multiplicities); a-node 3 and b-node 7 are isolated (d = 0: the uniform
    pick over all K blocks is the whole proposal)"""
    pairs = [((0, 4), 2), ((0, 5), 1), ((0, 6), 1), ((1, 4), 1), ((1, 5), 3), ((1, 6), 1), ((2, 5), 1), ((2, 6), 2)]
    return Model("A", 4, 4, pairs)


def model_b(hub=255):
    """3 + 4 nodes, Ka = Kb = 2.  a-node 0 has degree `hub` ((hub - 3) + 1 + 1 + 1 parallel edges): at 255 its u8
    histogram bin reaches 254 (fixed K) and 255 (estimate mode), at 256 the planner takes the round-1 kernel with u16
    bins.  a-node 1 has degree 33 (one more than the 32-neighbour tile), a-node 2 degree 1.  No b-node exceeds 255."""
    h = hub - 3
    pairs = [((0, 3), h), ((0, 4), 1), ((0, 5), 1), ((0, 6), 1),
             ((1, 3), 1), ((1, 4), 16), ((1, 5), 8), ((1, 6), 8), ((2, 5), 1)]
    return Model("B" if hub == 255 else "B%d" % hub, 3, 4, pairs)


# ---- log q(n, k): the reference's partition table (init_q_cache, src/support/int_part.cc:34-51) in exact integers ----
# q(n, 1) = 1 and q(n, k) = q(n, k - 1) + q(n - k, k) for 2 <= k <= n, where the table holds q(n - k, k) only for
# k <= n - k (its other cells stay log 0 = -inf).  So q(n, k) is not the number of partitions of n into at most k parts for
# every (n, k) (q(12, 3) = 14, not 19), but it is what the oracle, the replay path and the sweep kernels' tables hold, so it
# is part of the target they sample.
@lru_cache(maxsize=None)
def partitions(n, k):
    if k < 1 or k > n:
        return 0
    if k == 1:
        return 1
    return partitions(n, k - 1) + (partitions(n - k, k) if n > k else 0)


def log_q(n, k):
    """log_q<int> (src/support/int_part.hh:27-37): 0 for n <= 0 or k < 1, k clipped to n"""
    if n <= 0 or k < 1:
        return 0.0
    return math.log(partitions(n, min(k, n)))


def lbinom(N, k):
    """lbinom_fast (src/support/util.hh:41-47)"""
    if N == 0 or k == 0 or k > N:
        return 0.0
    return math.lgamma(N + 1) - math.lgamma(k + 1) - math.lgamma(N - k + 1)


def counts(model, lab, ka, kb):
    """m [K][K] (symmetric), e_r [K], n_r [K], eta [K][max d + 1] of a labeling with global block ids"""
    K = ka + kb
    lab = np.asarray(lab, dtype=np.int64)
    ea, eb = model.edges[:, 0].astype(np.int64), model.edges[:, 1].astype(np.int64)
    m = np.zeros((K, K), dtype=np.int64)
    np.add.at(m, (lab[ea], lab[eb]), 1)
    np.add.at(m, (lab[eb], lab[ea]), 1)
    eta = np.zeros((K, int(model.deg.max()) + 1), dtype=np.int64)
    np.add.at(eta, (lab, model.deg), 1)
    return m, m.sum(1), np.bincount(lab, minlength=K), eta


def occupied(model, lab, ka):
    lab = np.asarray(lab)
    return len(set(lab[:model.na].tolist())), len(set(lab[model.na:].tolist()))


def prior(model, ka, kb):
    """the K-dependent terms of entropy() and the constants that follow them"""
    return (lbinom(ka * kb + model.E - 1, model.E) + lbinom(model.na - 1, ka - 1) + lbinom(model.nb - 1, kb - 1) +
            math.log(model.na * model.nb) + math.lgamma(model.na + 1) + math.lgamma(model.nb + 1))


def entropy(model, lab, ka, kb, vary_k=False):
    """S of one labeling; vary_k: the prior terms with the number of OCCUPIED blocks per type"""
    m, e, nr, eta = counts(model, lab, ka, kb)
    S = model.base
    S -= sum(math.lgamma(int(x) + 1) for x in m[:ka, ka:].ravel())
    S -= sum(math.lgamma(int(x) + 1) for x in eta.ravel())
    S += sum(math.lgamma(int(x) + 1) + log_q(int(x), int(y)) for x, y in zip(e, nr))
    if vary_k:
        ka, kb = occupied(model, lab, ka)
    return S + prior(model, ka, kb)


def states(model, ka, kb, vary_k=False):
    """every labeling of the mode, [n_states][n] global block ids (fixed K: no empty block)"""
    def side(n, k):
        return [s for s in itertools.product(range(k), repeat=n) if vary_k or len(set(s)) == k]
    return np.array([list(a) + [ka + x for x in b] for a in side(model.na, ka) for b in side(model.nb, kb)], dtype=np.uint32)


def state_codes(lab, K):
    """one integer per labeling (base-K digits) -- to map sampled labelings to enumerated states"""
    lab = np.asarray(lab, dtype=np.int64)
    return (lab * (K ** np.arange(lab.shape[-1], dtype=np.int64))).sum(-1)


def target(S, T):
    """pi over enumerated states with description lengths S at temperature T"""
    w = np.exp(-(np.asarray(S) - np.min(S)) / T)
    return w / w.sum()


# ---- the proposal and the Hastings factor ----
def proposal_prob(model, lab, ka, kb, v, s, eps):
    """probability that single_vertex_change proposes global block s (own type, != label of v) for node v in labeling lab:
    d = 0 -> 1 / K; else sum over v's edges (to a node in block t) of (1/d) (m_ts + eps) / (e_t + eps K)"""
    K = ka + kb
    d = len(model.adj[v])
    if d == 0:
        return 1.0 / K
    m, e, _, _ = counts(model, lab, ka, kb)
    return sum((m[t, s] + eps) / (e[t] + eps * K) for t in (int(lab[j]) for j in model.adj[v])) / d


def kernel_hastings(model, lab, ka, kb, v, s, eps):
    """log accu_r as the sweep kernels compute it in one pass over v's edges (acc_edge, csrc/sweep.cuh): with c = earlier
    edges of v into the same block t, a0 += (m_st + eps) / (e_t + eps K), a1 += (m_rt - 2c - 1 + eps) / (e_t + eps K)"""
    K = ka + kb
    if not model.adj[v]:
        return 0.0
    m, e, _, _ = counts(model, lab, ka, kb)
    r = int(lab[v])
    a0 = a1 = 0.0
    seen = {}
    for j in model.adj[v]:
        t = int(lab[j])
        c = seen.get(t, 0)
        seen[t] = c + 1
        inv = 1.0 / (e[t] + eps * K)
        a0 += (m[s, t] + eps) * inv
        a1 += (m[r, t] - 2 * c - 1 + eps) * inv
    return math.log(a1 / a0)


def prior_k_delta(model, type_b, k_own, k_opp, dk):
    """the kernels' estimate-mode prior delta (prior_k_delta, csrc/sweep.cuh) for a move of a node of one type"""
    n_own = model.nb if type_b else model.na
    k2 = k_own + dk
    return (lbinom(k2 * k_opp + model.E - 1, model.E) + lbinom(n_own - 1, k2 - 1)) - \
           (lbinom(k_own * k_opp + model.E - 1, model.E) + lbinom(n_own - 1, k_own - 1))


def single_moves(model, lab, ka, kb):
    """(v, s) of every move of one node to another block of its own type"""
    for v in range(model.n):
        lo, hi = (0, ka) if v < model.na else (ka, ka + kb)
        if hi - lo == 1:
            continue
        for s in range(lo, hi):
            if s != int(lab[v]):
                yield v, s
