"""Chain agreement (bisbm_chain_agreement) on the GPU: exact statistics against a numpy / scipy recomputation from the
labels over every sweep kernel's label array, estimate mode and the multi-pass tables of large K; the reference form;
invariance under block relabelling; no side effects; a known two-mode split; and the command line's --agreement_out."""
import os
import subprocess

import numpy as np
import pytest

from agreement_ref import slots
from conftest import ROOT, load_golden
from helpers import planted

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "bin", "mcmc")
BIG = 10 ** 9
KEYS = ("vi", "nmi", "ari", "overlap")


def _k46():
    g = load_golden("c2_const_k46")
    return g["edges"], g["na"], g["nb"], g["labels0"].astype(np.uint32)


def _close(got, want):
    return abs(got - want) <= 1e-12 * max(1.0, abs(want))


def _check_pairs(res, labs, na, pairs=None):
    """every pair (or the given ones) against agreement_ref, per slot; overlap * n exact"""
    R, n = labs.shape
    ns = [na, n - na, n]
    for key in KEYS:
        a = res[key]
        assert a.shape == (3, R, R)
        assert (a.view(np.uint64) == a.transpose(0, 2, 1).view(np.uint64)).all(), key      # bitwise symmetric
        d = a[:, np.arange(R), np.arange(R)]
        assert (d == (0.0 if key == "vi" else 1.0)).all(), key
    for i, j in (pairs if pairs is not None else [(i, j) for i in range(R) for j in range(i + 1, R)]):
        want = slots(labs[i], labs[j], na)
        for s in range(3):
            for key in ("vi", "nmi", "ari"):
                assert _close(res[key][s, i, j], want[s][key]), (i, j, s, key, res[key][s, i, j], want[s][key])
            assert res["overlap"][s, i, j] == want[s]["matched"] / ns[s], (i, j, s)          # M exact: the same division


def _mixed_pool(host, kernel=None, prec="fp64", vary=False):
    """100 chains (padding lanes in the last group, two chunks of row chains), (4, 6) and (5, 5) blocks mixed, randomised
    starts and a few sweeps at T = 1"""
    edges, na, nb, mb = _k46()
    R = 100
    graph = host.Graph(edges, na, nb)
    n = na + nb
    if vary:
        kas, kbs = np.full(R, 6), np.full(R, 8)
        lab = np.concatenate([mb[:na], mb[na:] + 2]).astype(np.uint32)
        labels = np.tile(lab, (R, 1))
    else:
        kas = np.where(np.arange(R) % 3 == 0, 5, 4)
        kbs = 10 - kas
        v = np.arange(n)[None, :]
        labels = np.where(v < na, v % kas[:, None], kas[:, None] + v % kbs[:, None]).astype(np.uint32)
    pool = host.ChainPool(graph, labels, kas, kbs, 1.0)
    pool.set_precision(prec)
    if kernel is not None:
        pool.set_option("kernel", kernel)
    seeds = np.arange(R, dtype=np.uint64) + 23
    if vary:
        pool.set_option("vary_k", 1)
    else:
        pool.randomize(seeds)
    pool.anneal("constant", 1.0, 0.0, 3 * n, BIG, seeds)
    return pool, na, seeds


# case -> (precision, forced kernel, kernel id that must run)
CASES = {"staged_f64": ("fp64", None, 3), "staged_f32": ("fp32", None, 2), "l2": ("fp64", 5, 5), "round1_i32": ("fp64", 0, 0)}


@pytest.mark.parametrize("case", list(CASES))
def test_pairs_equal_the_host(host, case):
    prec, kernel, kid = CASES[case]
    pool, na, _ = _mixed_pool(host, kernel, prec)
    assert pool.sweep_info()[0] == kid
    labs = pool.labels().astype(np.int64)
    _check_pairs(pool.chain_agreement(), labs, na)


def test_estimate_mode_with_empty_blocks(host):
    pool, na, _ = _mixed_pool(host, vary=True)
    occ = np.asarray(pool.occupied_blocks()).reshape(-1, 2)
    assert (occ < [6, 8]).any()                               # some chains have empty blocks: zero rows
    labs = pool.labels().astype(np.int64)
    _check_pairs(pool.chain_agreement(), labs, na)


def _large_k_pool(host, k, kernel):
    na = nb = 3000
    graph = host.Graph(planted(na, nb, 8, 8, 30000, 3), na, nb)
    R = 36                                                    # padding lanes in the second group
    lab0 = np.concatenate([np.arange(na) % k, k + np.arange(nb) % k]).astype(np.uint32)
    pool = host.ChainPool(graph, np.tile(lab0, (R, 1)), k, k, 1.0)
    pool.set_option("kernel", kernel)
    seeds = np.arange(R, dtype=np.uint64) + 1
    pool.randomize(seeds)
    return pool, na, seeds


@pytest.mark.parametrize("k,kernel", [(128, 5), (300, 0)], ids=["k128_l2", "k300_i32"])
def test_large_k_multi_pass(host, k, kernel):
    pool, na, seeds = _large_k_pool(host, k, kernel)
    pool.anneal("constant", 1.0, 0.0, 2 * 6000, BIG, seeds)
    assert pool.sweep_info()[0] == kernel
    labs = pool.labels().astype(np.int64)
    rng = np.random.default_rng(1)
    R = labs.shape[0]
    pairs = [(i, j) for i in range(R) for j in range(i + 1, R) if rng.random() < 0.25] + [(0, R - 1), (31, 32)]
    _check_pairs(pool.chain_agreement(), labs, na, pairs)


def test_reference_form(host):
    pool, na, _ = _mixed_pool(host, None)
    labs = pool.labels().astype(np.int64)
    R, n = labs.shape
    KA = int(pool.ka.max())
    full = pool.chain_agreement()
    # a reference equal to chain k's labels, renumbered to the pool's (type b from the largest ka on), is column k
    for k in (0, 1, 99):
        ref = np.where(np.arange(n) < na, labs[k], labs[k] - int(pool.ka[k]) + KA)
        r = pool.chain_agreement(ref)
        for key in KEYS:
            assert r[key].shape == (3, R)
            assert all(_close(r[key][s, c], full[key][s, c, k]) for s in range(3) for c in range(R)), (k, key)
    # the planted partition of the graph's golden labels against the numpy values
    ref = np.asarray(load_golden("c2_const_k46")["labels0"], dtype=np.int64)
    refp = np.where(np.arange(n) < na, ref, ref - 4 + KA)
    r = pool.chain_agreement(refp)
    for c in (0, 50, 99):
        want = slots(ref, labs[c], na)
        for s in range(3):
            for key in ("vi", "nmi", "ari"):
                assert _close(r[key][s, c], want[s][key]), (c, s, key)
            assert r["overlap"][s, c] == want[s]["matched"] / [na, n - na, n][s]
    # overlap=False: NaN overlap, the rest unchanged
    r2 = pool.chain_agreement(refp, overlap=False)
    assert np.isnan(r2["overlap"]).all()
    for key in ("vi", "nmi", "ari"):
        assert (r2[key] == r[key]).all()
    # errors
    bad = refp.copy()
    bad[0] = KA                                             # a type-b id on a type-a node
    with pytest.raises(host.BisbmError) as ei:
        pool.chain_agreement(bad)
    assert ei.value.code == 1
    bad = refp.copy()
    bad[-1] = KA + int(pool.kb.max())
    with pytest.raises(host.BisbmError):
        pool.chain_agreement(bad)


def test_relabelling_invariance_and_no_side_effects(host):
    pool, na, seeds = _mixed_pool(host, None)
    labs = pool.labels()
    R, n = labs.shape
    pool.marginals_clear()
    pool.coassign_set(np.arange(0, n, 7))
    pool.marginal_sample()
    a1 = pool.chain_agreement()
    a2 = pool.chain_agreement()
    for key in KEYS:
        assert (a1[key].view(np.uint64) == a2[key].view(np.uint64)).all(), key          # bit-identical
    # nothing any other call sees has moved
    assert (pool.labels() == labs).all()
    hist0, co0 = pool.marginals().copy(), pool.coassign()
    m0 = [pool.m(c).copy() for c in (0, 57, 99)]
    pool.chain_agreement(overlap=False)
    assert (pool.marginals() == hist0).all() and (pool.coassign()[0] == co0[0]).all() and pool.coassign()[1] == co0[1]
    assert all((pool.m(c) == m).all() for c, m in zip((0, 57, 99), m0))
    # an anneal after the call is bit-identical to one without it (a twin pool built the same way, never compared)
    twin, _, _ = _mixed_pool(host, None)
    assert (twin.labels() == labs).all()
    pool.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
    twin.anneal("constant", 1.0, 0.0, 2 * n, BIG, seeds)
    assert (pool.labels() == twin.labels()).all()
    assert all((pool.m(c) == twin.m(c)).all() and pool.entropy(c) == twin.entropy(c) for c in (0, 57, 99))
    # permuting each chain's block ids within its type leaves every metric unchanged
    rng = np.random.default_rng(9)
    perm = labs.astype(np.int64).copy()
    for c in range(R):
        ka, kb = int(pool.ka[c]), int(pool.kb[c])
        pa, pb = rng.permutation(ka), ka + rng.permutation(kb)
        x = labs[c].astype(np.int64)
        perm[c] = np.where(np.arange(n) < na, pa[np.minimum(x, ka - 1)], pb[np.clip(x - ka, 0, kb - 1)])
    pool.set_labels(labs)
    base = pool.chain_agreement()
    pool.set_labels(perm.astype(np.uint32))
    moved = pool.chain_agreement()
    for key in KEYS:
        assert np.allclose(moved[key], base[key], rtol=1e-12, atol=1e-12), key


def test_a_known_two_mode_split(host):
    """half the chains start at one greedy fixed point, half at another; greedy sweeps keep them apart"""
    na = nb = 2000
    graph = host.Graph(planted(na, nb, 6, 6, 40000, 8, ratio=2.0), na, nb)
    n = na + nb
    rnd = np.random.default_rng(2)
    starts = [np.concatenate([rnd.integers(0, 6, na), 6 + rnd.integers(0, 6, nb)]).astype(np.uint32) for _ in range(2)]
    # two local optima of a weakly structured graph: greedy (T = 0) sweeps to convergence from two random partitions
    pre = host.ChainPool(graph, np.stack(starts), 6, 6, 1.0)
    s2 = np.array([1, 2], dtype=np.uint64)
    pre.anneal("abrupt_cool", 0.0, 0.0, 60 * n, BIG, s2)
    fixed = pre.labels()
    R = 64
    start = np.stack([fixed[c % 2] for c in range(R)])        # chains 0, 2, 4 .. at one, 1, 3, 5 .. at the other
    pool = host.ChainPool(graph, start, 6, 6, 1.0)
    seeds = np.arange(R, dtype=np.uint64) + 100
    pool.anneal("abrupt_cool", 0.0, 0.0, 3 * n, BIG, seeds)
    res = pool.chain_agreement()
    modes = host.chain_modes(res["overlap"][2])
    assert modes.tolist() == [c % 2 for c in range(R)]
    o = res["overlap"][2]
    same = (np.arange(R)[:, None] % 2) == (np.arange(R)[None, :] % 2)
    assert o[~same].max() < o[same].min()


def _run_cli(*args):
    p = subprocess.run([str(a) for a in [CLI, *args]], capture_output=True, text=True, timeout=600)
    return p.returncode, p.stdout, p.stderr


@pytest.mark.parametrize("mode", ["chains", "marginalize", "tempering", "estimate"])
def test_cli(pkg, host, tmp_path, mode):
    """bin/mcmc with and without --agreement_out: stdout unchanged; the file's format; its values equal
    bisbm_chain_agreement of a pool that replays the run (plain --marginalize) or are self-consistent"""
    pkg.build.build_all()
    edges, na, nb, mb = _k46()
    path = os.path.join(str(tmp_path), "g.edgelist")
    np.savetxt(path, edges, fmt="%d", delimiter="\t")
    out = os.path.join(str(tmp_path), "agree.txt")
    R = 40
    common = ["-e", path, "-y", 500, 500, "-n", 125, 125, 125, 125, 83, 83, 83, 83, 84, 84, "-z", 4, 6, "--randomize",
              "--chains", R, "--seed", 5]
    extra = {"chains": ["-c", "abrupt_cool", "-a", 2000, "-t", 3000, "-x", 1000],
             "marginalize": ["--marginalize", "-b", 10, "-t", 8, "-f", 4],
             "tempering": ["--marginalize", "-b", 10, "-t", 8, "-f", 4, "--tempering", 1, 1.5],
             "estimate": ["--estimate", "-b", 2, "-t", 4, "-f", 2]}[mode]
    rc0, out0, err0 = _run_cli(*common, *extra)
    assert rc0 == 0, err0
    rc, so, se = _run_cli(*common, *extra, "--agreement_out", out)
    assert rc == 0, se
    assert so == out0
    lines = [l for l in se.splitlines() if l.startswith("chain agreement:")]
    assert len(lines) == 1 and "NMI median" in lines[0] and "modes at overlap >= 0.95:" in lines[0], se
    with open(out) as f:
        rows = f.read().splitlines()
    assert rows[0] == str(R) and len(rows) == 1 + R * (R - 1) // 2
    vals = np.array([list(map(float, r.split())) for r in rows[1:]])
    assert vals.shape[1] == 14
    assert (vals[:, 0] < vals[:, 1]).all()
    assert ((vals[:, 2::4] <= 1 + 1e-12) & (vals[:, 2::4] >= -1e-12)).all()          # NMI
    assert ((vals[:, 5::4] > 0) & (vals[:, 5::4] <= 1)).all()                        # overlap
    if mode == "marginalize":
        # the same run through the Python API: same seeds, same labels, same numbers
        graph = host.Graph(edges, na, nb)
        lab0 = np.repeat(np.arange(10), [125, 125, 125, 125, 83, 83, 83, 83, 84, 84]).astype(np.uint32)
        pool = host.ChainPool(graph, np.tile(lab0, (R, 1)), 4, 6, 1.0)
        seeds = np.array([(5 * 0x9E3779B97F4A7C15 + c) % 2 ** 64 for c in range(R)], dtype=np.uint64)
        pool.randomize(seeds)
        pool.marginals_clear()
        pool.marginalize(10, 8, 4, seeds)
        res = pool.chain_agreement()
        i, j = vals[:, 0].astype(int), vals[:, 1].astype(int)
        for s, col in ((2, 2), (0, 6), (1, 10)):
            for k, key in enumerate(("nmi", "vi", "ari", "overlap")):
                assert np.array_equal(vals[:, col + k], res[key][s, i, j]), (s, key)
