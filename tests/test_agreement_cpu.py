"""Chain agreement without a device: chain_modes on synthetic overlap matrices, the numpy / scipy reference against
helpers.nmi and brute force, the Python-side argument checks, the C entry point's answer to a missing handle, and the
command line's --agreement_out rejections (they fire before any device is used)."""
import itertools
import os
import subprocess

import numpy as np
import pytest

from agreement_ref import metrics, slots
from conftest import ROOT
from helpers import nmi

CLI = os.path.join(ROOT, "bin", "mcmc")


def test_chain_modes_components_in_order_of_first_appearance(host):
    o = np.eye(7)
    for i, j in [(0, 3), (3, 5), (1, 6), (2, 4)]:
        o[i, j] = o[j, i] = 0.97
    o[0, 1] = o[1, 0] = 0.949                               # below the threshold: no edge
    assert host.chain_modes(o).tolist() == [0, 1, 2, 0, 2, 0, 1]
    assert host.chain_modes(o, threshold=0.94).tolist() == [0, 0, 1, 0, 1, 0, 0]
    assert host.chain_modes(o, threshold=1.0).tolist() == list(range(7))
    assert host.chain_modes(np.ones((4, 4))).tolist() == [0, 0, 0, 0]
    # an edge given on one side only still joins (a matrix against a threshold need not be symmetric)
    o = np.eye(3)
    o[2, 0] = 0.99
    assert host.chain_modes(o).tolist() == [0, 1, 0]
    with pytest.raises(ValueError):
        host.chain_modes(np.ones((2, 3)))


def test_reference_nmi_equals_helpers_nmi():
    rng = np.random.default_rng(1)
    for _ in range(30):
        n = int(rng.integers(2, 60))
        x = rng.integers(0, rng.integers(1, 6), size=n)
        y = rng.integers(0, rng.integers(1, 6), size=n)
        assert abs(metrics(x, y)["nmi"] - nmi(x, y)) <= 1e-12


def _brute(x, y):
    n = len(x)
    same_x = x[:, None] == x[None, :]
    same_y = y[:, None] == y[None, :]
    iu = np.triu_indices(n, 1)
    a, b, ab = same_x[iu].sum(), same_y[iu].sum(), (same_x & same_y)[iu].sum()
    tot = n * (n - 1) // 2
    exp = a * b / tot
    ari = 1.0 if 0.5 * (a + b) - exp == 0 else (ab - exp) / (0.5 * (a + b) - exp)
    ux, uy = np.unique(x), np.unique(y)
    best = 0
    small, large = (ux, uy) if len(ux) <= len(uy) else (uy, ux)
    for perm in itertools.permutations(large, len(small)):
        m = dict(zip(small, perm))
        src, dst = (x, y) if len(ux) <= len(uy) else (y, x)
        best = max(best, int(sum(m[s] == d for s, d in zip(src, dst))))
    h = lambda p: -(p[p > 0] * np.log(p[p > 0])).sum()
    px = np.bincount(np.unique(x, return_inverse=True)[1]) / n
    py = np.bincount(np.unique(y, return_inverse=True)[1]) / n
    vi = 2 * h(np.bincount(np.unique(x * 100 + y, return_inverse=True)[1]) / n) - h(px) - h(py)
    return ari, best, vi


def test_reference_ari_overlap_vi_against_brute_force():
    rng = np.random.default_rng(2)
    for _ in range(25):
        n = int(rng.integers(2, 25))
        x = rng.integers(0, 4, size=n)
        y = rng.integers(0, 5, size=n)
        ari, best, vi = _brute(x, y)
        m = metrics(x, y)
        assert abs(m["ari"] - ari) <= 1e-12 and m["matched"] == best and abs(m["vi"] - vi) <= 1e-12


def test_reference_slots_and_identity():
    rng = np.random.default_rng(4)
    na, nb = 30, 20
    x = np.concatenate([rng.integers(0, 3, na), 3 + rng.integers(0, 4, nb)])
    s = slots(x, x, na)
    for m in s:
        assert abs(m["vi"]) <= 1e-12 and m["nmi"] == 1.0 and m["ari"] == 1.0 and m["overlap"] == 1.0
    # relabelling the blocks within a type changes nothing
    y = np.concatenate([rng.integers(0, 3, na), 3 + rng.integers(0, 4, nb)])
    perm_a, perm_b = rng.permutation(3), 3 + rng.permutation(4)
    y2 = np.where(np.arange(na + nb) < na, perm_a[np.minimum(y, 2)], perm_b[np.maximum(y - 3, 0)])
    for m1, m2 in zip(slots(x, y, na), slots(x, y2, na)):
        for k in ("vi", "nmi", "ari", "overlap"):
            assert abs(m1[k] - m2[k]) <= 1e-12


class _Pool:
    """just enough of a ChainPool for its argument check, which runs before any library call"""
    n_chains = 3

    class g:
        n = 10


@pytest.mark.parametrize("bad", [np.zeros(9, dtype=np.int64), np.array([1, -2] * 5), np.zeros((2, 5), dtype=np.int64)])
def test_chain_agreement_rejects_what_is_not_a_partition(host, bad):
    with pytest.raises(ValueError):
        host.ChainPool.chain_agreement(_Pool(), bad)


def test_entry_point_without_a_handle(pkg, host):
    pkg.build.build_lib()
    L = host.load_library()
    assert L.bisbm_chain_agreement(None, None, 1, None) == 1
    assert b"null handle" in L.bisbm_last_error()


@pytest.fixture(scope="module")
def cli(pkg):
    pkg.build.build_all()
    return CLI


def _run(cli, *args):
    p = subprocess.run([str(a) for a in [cli, "-e", "x", "-y", 18, 14, "-n", 9, 9, 7, 7, "-z", 2, 2, *args]],
                       capture_output=True, text=True, timeout=60)
    return p.returncode, p.stdout, p.stderr


def test_cli_agreement_rejections(cli, tmp_path):
    out = os.path.join(str(tmp_path), "agree.txt")
    rc, so, se = _run(cli, "--chains", 4, "--agreement_out")
    assert rc == 1 and so == "" and "'--agreement_out' is missing" in se, se
    for extra in ([], ["--chains", 1], ["--marginalize"], ["--estimate", "--chains", 1]):
        rc, so, se = _run(cli, "--agreement_out", out, *extra)
        assert rc == 1 and so == "" and se == "--agreement_out needs --chains >= 2\n", (extra, se)
    rc, so, se = _run(cli, "--agreement_out", out, "--chains", 4, "--gpus", 2, "--marginalize")
    assert rc == 1 and so == "" and se == "--agreement_out compares the chains of one GPU (no --gpus > 1)\n", se
    rc, so, se = _run(cli, "--agreement_out", out, "--chains", 4, "-g")          # the agglomerative path
    assert rc == 1 and so == "" and "the agglomerative paths run one chain" in se, se
    assert not os.path.exists(out)


def test_cli_usage_lists_agreement_out(cli):
    p = subprocess.run([cli, "-h"], capture_output=True, text=True, timeout=60)
    assert p.returncode == 0 and "--agreement_out" in p.stderr
