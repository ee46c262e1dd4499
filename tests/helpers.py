"""numpy restatements used by several tests (not product code)."""
import numpy as np


def counts_from_labels(edges, na, nb, labels, ka, kb):
    """m (K x K symmetric), e_r, n_r, eta rebuilt from scratch like compute_m / compute_m_r /
    compute_n_r / compute_eta_rk (reference src/blockmodel.cc:691-746)."""
    K = ka + kb
    n = na + nb
    labels = np.asarray(labels, dtype=np.int64)
    ea, eb = edges[:, 0].astype(np.int64), edges[:, 1].astype(np.int64)
    m = np.zeros((K, K), dtype=np.int64)
    np.add.at(m, (labels[ea], labels[eb]), 1)
    np.add.at(m, (labels[eb], labels[ea]), 1)
    deg = np.bincount(np.concatenate([ea, eb]), minlength=n)
    eta = np.zeros((K, deg.max() + 1), dtype=np.int64)
    np.add.at(eta, (labels, deg), 1)
    return m, m.sum(1), np.bincount(labels, minlength=K), eta


def planted(na, nb, ka, kb, n_edges, seed, ratio=10.0):
    """Synthetic planted bipartite SBM of SURVEY.md 8(d) (same generator as tests/golden/make_golden.py
    and bench.py)."""
    rng = np.random.default_rng(seed)
    w = np.ones((ka, kb))
    for r in range(ka):
        w[r, r * kb // ka] = ratio
    p = (w / w.sum()).ravel()
    pair = rng.choice(ka * kb, size=n_edges, p=p)
    r, s = pair // kb, pair % kb
    ba = np.arange(na) * ka // na
    bb = np.arange(nb) * kb // nb
    a_start = np.searchsorted(ba, np.arange(ka))
    a_cnt = np.bincount(ba, minlength=ka)
    b_start = np.searchsorted(bb, np.arange(kb))
    b_cnt = np.bincount(bb, minlength=kb)
    ea = a_start[r] + (rng.random(n_edges) * a_cnt[r]).astype(np.int64)
    eb = na + b_start[s] + (rng.random(n_edges) * b_cnt[s]).astype(np.int64)
    return np.stack([ea, eb], 1).astype(np.uint32)


def planted_labels(na, nb, ka, kb):
    return np.concatenate([np.arange(na) * ka // na, ka + np.arange(nb) * kb // nb]).astype(np.uint32)


def nmi(a, b):
    a = np.asarray(a); b = np.asarray(b)
    n = len(a)
    ua, ia = np.unique(a, return_inverse=True)
    ub, ib = np.unique(b, return_inverse=True)
    c = np.zeros((len(ua), len(ub)))
    np.add.at(c, (ia, ib), 1)
    pa, pb = c.sum(1) / n, c.sum(0) / n
    p = c / n
    nz = p > 0
    mi = (p[nz] * np.log(p[nz] / (pa[:, None] * pb[None, :])[nz])).sum()
    ha = -(pa[pa > 0] * np.log(pa[pa > 0])).sum()
    hb = -(pb[pb > 0] * np.log(pb[pb > 0])).sum()
    return 2 * mi / (ha + hb) if ha + hb > 0 else 1.0


def staged_model():
    """ctypes handle of tests/staged_model.cc (the host model of the staged sweep's moves), built on first use."""
    import ctypes as C
    import os
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    lib = os.path.join(here, "libstaged_model.so")
    deps = [os.path.join(here, "staged_model.cc"), os.path.join(root, "oracle", "bisbm_oracle.c"),
            os.path.join(root, "bipartitesbm-mcmc_b200", "csrc", "devmath.cuh")]
    if not os.path.exists(lib) or any(os.path.getmtime(d) > os.path.getmtime(lib) for d in deps):
        tmp = lib + ".%d" % os.getpid()
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-o", tmp,
                               deps[0], "-x", "c", deps[1], "-lm"])
        os.replace(tmp, lib)
    L = C.CDLL(lib)
    pu, pd, pq = C.POINTER(C.c_uint32), C.POINTER(C.c_double), C.POINTER(C.c_uint64)
    L.sm_visit_cover.argtypes = [C.c_uint32] * 5 + [pu, pu]
    L.sm_transition.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, pu, pu, pu, C.c_uint32, C.c_uint32, C.c_double, C.c_uint32,
                                C.c_uint32, pd, pd]
    L.sm_replay_sweep.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, pu, pu, C.c_uint32, pu, pu, pu, C.c_double, pq,
                                  C.c_uint64, C.c_uint64, C.c_int, C.c_float, C.c_float, pu, C.c_int, C.c_int,
                                  pq, pd, pd, pu, pq]
    return L


def replay_sweep(L, na, nb, n_edges, row_ptr, col, labels, ka, kb, eps, seeds, epoch, schedule, p0, p1, plans, vary_k, fp32):
    """One sweep of every chain by the staged model (tests/staged_model.cc) from `labels` [chains][n] (global ids), under
    plans = [plan of type a, plan of type b], each (ctas per group, slice, warps used, extras, sliced).  Returns a dict of
    per-chain arrays: labels, accepted, dS (sum over the accepted moves), tol (sum of their tie tolerances), flags, moves."""
    import ctypes as C
    P = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    n_chains = labels.shape[0]
    lab = np.ascontiguousarray(labels, dtype=np.uint32).copy()
    ka = np.ascontiguousarray(np.broadcast_to(ka, (n_chains,)), dtype=np.uint32)
    kb = np.ascontiguousarray(np.broadcast_to(kb, (n_chains,)), dtype=np.uint32)
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
    rp = np.ascontiguousarray(row_ptr, dtype=np.uint32)
    cl = np.ascontiguousarray(col, dtype=np.uint32)
    plan = np.ascontiguousarray(np.asarray(plans, dtype=np.uint32).reshape(10))
    out = {"labels": lab, "accepted": np.zeros(n_chains, np.uint64), "dS": np.zeros(n_chains), "tol": np.zeros(n_chains),
           "flags": np.zeros(n_chains, np.uint32), "moves": np.zeros(n_chains, np.uint64)}
    rc = L.sm_replay_sweep(na, nb, n_edges, P(rp, C.c_uint32), P(cl, C.c_uint32), n_chains, P(lab, C.c_uint32),
                           P(ka, C.c_uint32), P(kb, C.c_uint32), eps, P(seeds, C.c_uint64), epoch, 0, schedule, p0, p1,
                           P(plan, C.c_uint32), int(vary_k), int(fp32), P(out["accepted"], C.c_uint64),
                           P(out["dS"], C.c_double), P(out["tol"], C.c_double), P(out["flags"], C.c_uint32),
                           P(out["moves"], C.c_uint64))
    assert rc == 0, "visiting order does not cover the half sweep (%d)" % rc
    return out


def sweep_plan(nv, n_chains, sm_count, wpc, inflight_div=64, max_inflight=0, spare_sms=True):
    """(ctas per group, slice, warps used, extras, sliced) of one staged half sweep: plan_sweep and launch_full_sweep
    (csrc/capi.cu) restated."""
    G = (n_chains + 31) // 32
    inflight = max_inflight if max_inflight else max(1, nv // max(1, inflight_div))
    cpg = max(1, sm_count // G)
    cpg = min(cpg, max(1, inflight // wpc))
    cpg = min(cpg, max(1, nv // (wpc * 4)))
    warps_used = max(1, min(wpc, min(inflight, max(nv, 1)))) if cpg == 1 else wpc
    if cpg > 1:
        sl = max(cpg * wpc, min(inflight, nv))
        sl = max(cpg * wpc, sl // (cpg * wpc) * (cpg * wpc))
    else:
        sl = max(nv, 1)
    sliced = cpg > 1
    extras = min(sm_count - G * cpg, G - 1) if sliced and spare_sms and max_inflight == 0 and sm_count > G * cpg else 0
    return (cpg, sl, warps_used, extras, int(sliced))
