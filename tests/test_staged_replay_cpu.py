"""The host model of the staged sweep (tests/staged_model.cc) checked without a GPU: its move arithmetic against the
oracle's transition_ratio, and its visiting order against the rule that every half sweep visits each position once."""
import ctypes as C

import numpy as np
import pytest

from conftest import TRAJECTORIES, load_golden
from helpers import staged_model, sweep_plan
from oracle import port

pu = C.POINTER(C.c_uint32)


@pytest.fixture(scope="module")
def model():
    return staged_model()


def csr(edges, n):
    ea, eb = edges[:, 0].astype(np.int64), edges[:, 1].astype(np.int64)
    src = np.concatenate([ea, eb])
    dst = np.concatenate([eb, ea])
    order = np.argsort(src, kind="stable")
    rp = np.zeros(n + 1, dtype=np.uint32)
    np.add.at(rp, src + 1, 1)
    return np.cumsum(rp).astype(np.uint32), dst[order].astype(np.uint32)


@pytest.mark.parametrize("name", TRAJECTORIES)
def test_model_transition_matches_oracle(model, name):
    """the model's dS and log accu_r of a move equal the oracle's transition_ratio on random states.  dS to 1e-9 relative: the
    oracle sums the two entropies in double before it subtracts them (up to 2e-10 of cancellation on big_blocks)."""
    g = load_golden(name)
    na, nb, ka, kb = g["na"], g["nb"], g["ka"], g["kb"]
    n = na + nb
    edges = g["edges"]
    rp, col = csr(edges, n)
    rng = np.random.default_rng(17)
    checked = 0
    for _ in range(4):
        lab = np.concatenate([rng.integers(0, ka, na), ka + rng.integers(0, kb, nb)]).astype(np.uint32)
        o = port.PortChain(n, na, nb, edges, lab, ka, kb, g["eps"], 1)
        o.init(False)
        for v in rng.integers(0, n, 60):
            v = int(v)
            lo, k = (0, ka) if v < na else (ka, kb)
            if k == 1:
                continue
            s = int(lo + rng.integers(0, k))
            if s == lab[v]:
                continue
            dS_o, accu_o = o.transition(v, s)
            d, lh = C.c_double(), C.c_double()
            assert model.sm_transition(na, nb, len(edges), rp.ctypes.data_as(pu), col.ctypes.data_as(pu),
                                       lab.ctypes.data_as(pu), ka, kb, g["eps"], v, s, C.byref(d), C.byref(lh)) == 0
            assert abs(d.value - dS_o) <= 1e-9 * max(1.0, abs(dS_o)), (name, v, s, d.value, dS_o)
            assert abs(lh.value - np.log(accu_o)) <= 1e-12 * max(1.0, abs(np.log(accu_o))), (name, v, s)
            checked += 1
        o.close()
    assert checked > 20


# (nv, chains, SMs, warps per CTA, inflight_div, max_inflight)
SHAPES = [(16384, 256, 148, 16, 64, 0),       # the benchmark's shape: extras = 148 - 8 x 16 = 20 -> capped at groups - 1
          (16384, 256, 148, 16, 1, 0),        # several rounds per CTA
          (16384, 256, 148, 16, 64, 2048),    # explicit bound: no extras
          (6000, 200, 148, 16, 64, 0),        # nv not a multiple of the slice, 7 groups
          (9001, 96, 148, 8, 64, 0),          # 3 groups, extras = 2 = groups - 1
          (5000, 32, 148, 16, 64, 0),         # one group: no extras
          (1500, 64, 148, 16, 1, 5),          # one CTA
          (100003, 640, 132, 16, 64, 0)]      # 20 groups on a smaller part


@pytest.mark.parametrize("shape", SHAPES)
def test_visiting_order_covers_every_position_once(model, shape):
    nv, chains, sms, wpc, div, mi = shape
    cpg, sl, _wu, extras, _sliced = sweep_plan(nv, chains, sms, wpc, div, mi)
    G = (chains + 31) // 32
    nl, cmax = C.c_uint32(), C.c_uint32()
    assert model.sm_visit_cover(nv, G, cpg, sl, extras, C.byref(nl), C.byref(cmax)) == 0, (shape, cpg, sl, extras)
    assert cmax.value <= cpg + (1 if extras else 0)
    if extras:
        assert cmax.value == cpg + 1            # some group is handed a spare-SM CTA


@pytest.mark.parametrize("extras", [1, 2, 3])
@pytest.mark.parametrize("nv", [997, 1024, 4099])
def test_visiting_order_with_extras_up_to_groups_minus_one(model, nv, extras):
    """extras = 1 .. groups - 1 with 4 groups, 3 CTAs per group and slices that do not divide nv"""
    nl, cmax = C.c_uint32(), C.c_uint32()
    assert model.sm_visit_cover(nv, 4, 3, 3 * 16, extras, C.byref(nl), C.byref(cmax)) == 0
