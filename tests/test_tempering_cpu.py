"""Parallel tempering without a device: geometric_ladder, the Python-side argument checks, the command line's rejections
(they fire before any handle is made) and the C entry points' answers to a missing handle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

CLI = os.path.join(ROOT, "bin", "mcmc")


def test_geometric_ladder(host):
    t = host.geometric_ladder(1.0, 1.5, 8)
    assert len(t) == 8 and t[0] == 1.0 and t[-1] == 1.5
    assert np.allclose(t[1:] / t[:-1], 1.5 ** (1 / 7)) and (np.diff(t) >= 0).all()
    assert host.geometric_ladder(2.0, 2.0, 3).tolist() == [2.0, 2.0, 2.0]
    assert host.geometric_ladder(1.0, 4.0, 1).tolist() == [1.0]
    assert host.geometric_ladder(1.0, 4.0, 3).tolist() == [1.0, 2.0, 4.0]
    for args in [(1.0, 2.0, 0), (0.0, 2.0, 4), (2.0, 1.0, 4), (1.0, np.inf, 4), (-1.0, 1.0, 2)]:
        with pytest.raises(ValueError):
            host.geometric_ladder(*args)


class _Pool:
    """just enough of a ChainPool for its argument checks, which run before any library call"""
    n_chains = 8


@pytest.mark.parametrize("temps", [[1.0, 2.0, 3.0], [1.0, 0.0], [1.0, -2.0], [1.0, float("nan")], [1.0, float("inf")], [2.0, 1.0]])
def test_tempering_set_rejects_bad_ladders(host, temps):
    with pytest.raises(ValueError):
        host.ChainPool.tempering_set(_Pool(), temps)


def test_tempering_set_rejects_bad_rung_shape(host):
    with pytest.raises(ValueError):
        host.ChainPool.tempering_set(_Pool(), [1.0, 2.0], rung_of_chain=[0, 1, 0])


def test_tempering_run_rejects_zero_swap_interval(host):
    with pytest.raises(ValueError):
        host.ChainPool.tempering_run(_Pool(), 10, 0, np.zeros(8, dtype=np.uint64))


def test_entry_points_without_a_handle(pkg, host):
    """bound with their declared signatures; a null handle is BISBM_ERR_ARG, not a crash.  Without a device no handle can
    exist: every way to make one fails with BISBM_ERR_CUDA (tests/test_capi_cpu.py)."""
    pkg.build.build_lib()
    L = host.load_library()
    t = np.array([1.0, 2.0])
    assert L.bisbm_tempering_set(None, 2, t.ctypes.data_as(C.POINTER(C.c_double)), None) == 1
    assert L.bisbm_tempering_run(None, 1, 1, 0, None, 1, 0, None) == 1
    assert L.bisbm_tempering_stats(None, None, None, None, None, None, None) == 1
    assert b"null handle" in L.bisbm_last_error()


@pytest.fixture(scope="module")
def cli(pkg):
    pkg.build.build_all()
    return CLI


@pytest.mark.parametrize("extra,msg", [
    (["--marginalize", "--estimate"], "--tempering does not combine with --estimate"),
    (["--marginalize", "-g"], "--tempering does not combine with the agglomerative paths (-g / -u)"),
    (["--marginalize", "--gpus", 2], "--tempering runs on one GPU (no --gpus > 1)"),
    ([], "--tempering needs --marginalize"),
    (["--chains", 4], "--tempering needs --marginalize"),
    (["--marginalize", "--chains", 6], "--chains must be a multiple of the number of --tempering temperatures"),
    (["--marginalize", "--swap_every", 0], "bad value for --swap_every"),
])
def test_cli_rejections(cli, extra, msg):
    args = [cli, "-e", "x", "-y", 18, 14, "-n", 9, 9, 7, 7, "-z", 2, 2, "--tempering", 1, 1.5, 2, 3] + extra
    p = subprocess.run([str(a) for a in args], capture_output=True, text=True, timeout=60)
    assert p.returncode == 1 and p.stderr == msg + "\n", p.stderr


def test_cli_usage_lists_the_options(cli):
    p = subprocess.run([cli, "-h"], capture_output=True, text=True, timeout=60)
    assert p.returncode == 0 and "--tempering" in p.stderr and "--swap_every" in p.stderr
