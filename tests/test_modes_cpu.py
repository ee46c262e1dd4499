"""Marginals by mode without a device: mode_references against a stub pool, the Python-side argument checks, the C entry
points' answer to a missing handle, and the command line's --modes_out rejections (they fire before any device is used)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

CLI = os.path.join(ROOT, "bin", "mcmc")


class _StubPool:
    """what mode_references reads of a ChainPool: the pairwise agreement, the entropies and the labels"""

    def __init__(self, overlap, entropy, labels):
        self.n_chains = len(entropy)
        self._o, self._s, self._l = np.asarray(overlap), np.asarray(entropy), np.asarray(labels)
        self.agreement_calls = 0

    def chain_agreement(self, ref=None, overlap=True):
        assert ref is None and overlap
        self.agreement_calls += 1
        return {"overlap": np.stack([np.zeros_like(self._o), np.zeros_like(self._o), self._o])}

    def entropy(self, chain=None):
        return self._s.copy() if chain is None else self._s[chain]

    def labels(self, chain=None):
        return self._l.copy() if chain is None else self._l[chain].copy()


def _stub():
    # chains 0, 2, 5 | 1, 4 | 3: three components at 0.95
    o = np.eye(6)
    for i, j in [(0, 2), (2, 5), (1, 4)]:
        o[i, j] = o[j, i] = 0.96
    o[0, 3] = o[3, 0] = 0.94
    ent = np.array([5.0, 3.0, 4.0, 9.0, 3.0, 1.0])               # chains 1 and 4 tie: the lower id is the reference
    labels = np.arange(6)[:, None] * 10 + np.arange(8)[None, :]   # row c identifies chain c
    return _StubPool(o, ent, labels), labels


def test_mode_references_take_the_lowest_entropy_member(host):
    pool, labels = _stub()
    refs, mode = host.mode_references(pool)
    assert mode.tolist() == [0, 1, 0, 2, 1, 0]
    assert refs.dtype == np.uint32 and refs.shape == (3, 8)
    assert (refs == labels[[5, 1, 3]]).all()
    assert pool.agreement_calls == 1
    refs, mode = host.mode_references(pool, threshold=0.9)     # 3 joins 0's component
    assert mode.tolist() == [0, 1, 0, 0, 1, 0] and (refs == labels[[5, 1]]).all()


def test_mode_references_restricted_to_candidates(host):
    pool, labels = _stub()
    refs, mode = host.mode_references(pool, chains=[3, 2, 4])
    # the candidates in the order given: 3, 2 and 4 are three modes (2's partners 0 and 5 are not candidates)
    assert mode.tolist() == [-1, -1, 1, 0, 2, -1]
    assert (refs == labels[[3, 2, 4]]).all()
    refs, mode = host.mode_references(pool, chains=np.array([0, 2]))
    assert mode.tolist() == [0, -1, 0, -1, -1, -1] and (refs == labels[[2]]).all()
    for bad in ([], [1, 1], [6], [-1]):
        with pytest.raises(ValueError):
            host.mode_references(pool, chains=bad)


class _Pool:
    """just enough of a ChainPool for its argument check, which runs before any library call"""
    n_chains = 3

    class g:
        n = 10


@pytest.mark.parametrize("bad", [np.zeros(9, dtype=np.int64), np.array([1, -2] * 5), np.zeros((2, 2, 5), dtype=np.int64),
                                 np.zeros((0, 10), dtype=np.int64)])
def test_modes_set_rejects_what_is_not_a_set_of_partitions(host, bad):
    with pytest.raises(ValueError):
        host.ChainPool.marginal_modes_set(_Pool(), bad)


def test_entry_points_without_a_handle(pkg, host):
    pkg.build.build_lib()
    L = host.load_library()
    assert L.bisbm_marginal_modes_set(None, 0, None, 0.0) == 1
    assert b"null handle" in L.bisbm_last_error()
    assert L.bisbm_marginal_modes_get(None, None, None, None, None) == 1
    assert b"null handle" in L.bisbm_last_error()
    assert L.bisbm_marginal_modes_argmax(None, None) == 1
    assert b"null handle" in L.bisbm_last_error()


@pytest.fixture(scope="module")
def cli(pkg):
    pkg.build.build_all()
    return CLI


def _run(cli, *args):
    p = subprocess.run([str(a) for a in [cli, "-e", "x", "-y", 18, 14, "-n", 9, 9, 7, 7, "-z", 2, 2, *args]],
                       capture_output=True, text=True, timeout=60)
    return p.returncode, p.stdout, p.stderr


def test_cli_modes_rejections(cli, tmp_path):
    out = os.path.join(str(tmp_path), "modes.txt")
    rc, so, se = _run(cli, "--chains", 4, "--marginalize", "--modes_out")
    assert rc == 1 and so == "" and "'--modes_out' is missing" in se, se
    for extra in ([], ["--chains", 4], ["--chains", 4, "--estimate"]):
        rc, so, se = _run(cli, "--modes_out", out, *extra)
        assert rc == 1 and so == "" and se == "--modes_out needs --marginalize\n", (extra, se)
    rc, so, se = _run(cli, "--modes_out", out, "--chains", 4, "--gpus", 2, "--marginalize")
    assert rc == 1 and so == "" and se == "--modes_out finds the modes of one GPU's chains (no --gpus > 1)\n", se
    for extra in ([], ["--chains", 1]):
        rc, so, se = _run(cli, "--modes_out", out, "--marginalize", *extra)
        assert rc == 1 and so == "" and se == "--modes_out needs --chains >= 2\n", (extra, se)
    assert not os.path.exists(out)


def test_cli_usage_lists_modes_out(cli):
    p = subprocess.run([cli, "-h"], capture_output=True, text=True, timeout=60)
    assert p.returncode == 0 and "--modes_out" in p.stderr
