"""Label alignment of the marginals without a device: the Python-side argument check, the C entry points' answers to a
missing handle, and the command line's --align rejection and usage text (they fire before any handle is made)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

CLI = os.path.join(ROOT, "bin", "mcmc")


class _Pool:
    """just enough of a ChainPool for its argument check, which runs before any library call"""
    class g:
        n = 10


def test_marginals_align_rejects_a_reference_of_the_wrong_length(host):
    for bad in (np.zeros(9, dtype=np.uint32), np.zeros((2, 10), dtype=np.uint32)):
        with pytest.raises(ValueError):
            host.ChainPool.marginals_align(_Pool(), bad)


def test_entry_points_without_a_handle(pkg, host):
    pkg.build.build_lib()
    L = host.load_library()
    assert L.bisbm_marginals_align(None, None) == 1
    assert L.bisbm_marginals_alignment(None, None) == 1
    assert b"null handle" in L.bisbm_last_error()


@pytest.fixture(scope="module")
def cli(pkg):
    pkg.build.build_all()
    return CLI


@pytest.mark.parametrize("extra", [[], ["--chains", 4], ["--chains", 4, "--randomize"], ["--estimate"]])
def test_cli_align_needs_marginalize(cli, extra):
    args = [cli, "-e", "x", "-y", 18, 14, "-n", 9, 9, 7, 7, "-z", 2, 2, "--align"] + extra
    p = subprocess.run([str(a) for a in args], capture_output=True, text=True, timeout=60)
    assert p.returncode == 1 and p.stderr == "--align needs --marginalize\n", p.stderr


def test_cli_usage_lists_align(cli):
    p = subprocess.run([cli, "-h"], capture_output=True, text=True, timeout=60)
    assert p.returncode == 0 and "--align" in p.stderr
