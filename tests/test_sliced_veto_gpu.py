"""The exact "would empty block r" veto of the staged sweep under a sliced multi-CTA plan.

Blocks small enough to empty within one launch take the exact path: an atomic count of the launch's decrements, checked
against n_r at the launch's start.  Here every chain starts with blocks of one or two nodes, on a graph where a chain group
is cut into several CTAs per launch, at fixed K: after every call no block may be empty, and the device counts must equal a
rebuild from the labels."""
import numpy as np
import pytest

from helpers import counts_from_labels

pytestmark = pytest.mark.gpu

NA = NB = 8192
KA = KB = 32
TINY = 10          # blocks of one or two nodes per type


def random_graph(seed, n_edges=65536):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(0, NA, n_edges), NA + rng.integers(0, NB, n_edges)], 1).astype(np.uint32)


def tiny_block_labels(rng, n_chains):
    out = np.empty((n_chains, NA + NB), dtype=np.uint32)
    for c in range(n_chains):
        for n0, nt, k, off in ((0, NA, KA, 0), (NA, NB, KB, KA)):
            lab = np.empty(nt, dtype=np.int64)
            perm = rng.permutation(nt)
            sizes = rng.integers(1, 3, size=TINY)
            pos = 0
            for b in range(TINY):
                lab[perm[pos:pos + sizes[b]]] = b
                pos += sizes[b]
            rest = perm[pos:]
            lab[rest] = TINY + np.arange(rest.size) % (k - TINY)
            out[c, n0:n0 + nt] = off + lab
    return out


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_sliced_veto_keeps_blocks(host, precision):
    edges = random_graph(5)
    graph = host.Graph(edges, NA, NB)
    n_chains = 64                  # two chain groups: with CTAs left over, the spare-SM CTAs join the groups in turn
    rng = np.random.default_rng(7)
    pool = host.ChainPool(graph, tiny_block_labels(rng, n_chains), KA, KB, 1.0)
    pool.set_precision(precision)
    seeds = np.arange(1, n_chains + 1, dtype=np.uint64) * 977
    smallest = []
    for _ in range(4):
        pool.anneal("constant", 1.0, 0.0, 2 * (NA + NB), 10 ** 18, seeds)
        kernel, _wpc, cpg, slice_ = pool.sweep_info()
        assert kernel == (3 if precision == "fp64" else 2)          # the staged sweep2 kernel
        assert cpg >= 4 and slice_ < NA                             # several CTAs per group, several launches per half sweep
        labels = pool.labels()
        for c in range(n_chains):
            m, e, nr, eta = counts_from_labels(edges, NA, NB, labels[c], KA, KB)
            assert (nr >= 1).all(), "chain %d: a block emptied" % c
            assert (pool.n_r(c) == nr).all()
            assert (pool.m(c) == m).all()
            assert (pool.m_r(c) == e).all()
            assert (pool.eta(c) == eta).all()
            smallest.append(int(nr.min()))
    # the chains stay where the veto decides: blocks far below one launch's slice
    assert min(smallest) <= 2
