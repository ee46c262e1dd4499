"""Python mirror of the reference's in-process interface for the MH sweep, over libbisbm.so.

The reference is C++ with no bindings; this module gives its classes and call shapes a
Python face so tests read like calls into the reference:

    adj   = edge_to_adj(load_edge_list(path), N)            # src/graph_utilities.cc:20-49
    bm    = blockmodel_t(memberships, types, K, KA, KB, epsilon, adj)   # src/blockmodel.cc:15-75
    bm.shuffle_bisbm(engine, NA, NB) | bm.init_bisbm()                  # src/blockmodel.cc:672-688
    rate  = metropolis_hasting().anneal(bm, exponential_schedule, [10, 0.1], 1000, 100, engine)
    bm.get_memberships(), bm.get_m(), bm.get_m_r(), bm.get_n_r(), bm.entropy()

plus ChainPool, the many-chains-per-launch interface the reference does not have.  All
compute happens in the CUDA library; if libbisbm.so is missing or no GPU is present every
compute call raises -- there is no CPU fallback.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbisbm.so")

EXPONENTIAL, LINEAR, LOGARITHMIC, CONSTANT, ABRUPT_COOL = range(5)
SCHEDULES = {"exponential": 0, "linear": 1, "logarithmic": 2, "constant": 3, "abrupt_cool": 4}

# names of the reference's schedule functions (src/metropolis_hasting.cc:10-37)
exponential_schedule = EXPONENTIAL
linear_schedule = LINEAR
logarithmic_schedule = LOGARITHMIC
constant_schedule = CONSTANT
abrupt_cool_schedule = ABRUPT_COOL


class BisbmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libbisbm error %d: %s" % (code, msg))
        self.code = code


_lib = None
_u32p = C.POINTER(C.c_uint32)
_i32p = C.POINTER(C.c_int32)
_u64p = C.POINTER(C.c_uint64)
_dp = C.POINTER(C.c_double)

# every symbol include/bisbm.h declares, with its ctypes signature
SIGNATURES = {
    "bisbm_last_error": (C.c_char_p, []),
    "bisbm_version": (C.c_char_p, []),
    "bisbm_create": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint64, _u32p, _u32p, C.c_int, C.POINTER(C.c_void_p)]),
    "bisbm_create_csr": (C.c_int, [C.c_uint32, C.c_uint32, _u32p, _u32p, C.c_int, C.POINTER(C.c_void_p)]),
    "bisbm_destroy": (C.c_int, [C.c_void_p]),
    "bisbm_share_graph": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "bisbm_grid_search": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _u32p, C.c_uint32, C.c_double, C.c_int, C.c_float, C.c_float,
                                    C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, _dp, _dp, _u32p, _u32p, _dp]),
    "bisbm_create_from_text": (C.c_int, [C.c_uint32, C.c_uint32, C.c_char_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]),
    "bisbm_get_csr": (C.c_int, [C.c_void_p, _u32p, _u32p]),
    "bisbm_grid_release": (C.c_int, [C.c_void_p]),
    "bisbm_grid_k_class": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _u32p, _u32p, C.POINTER(C.c_int)]),
    "bisbm_grid_search_report": (C.c_int, [C.c_void_p, C.c_uint32, _dp, _u32p]),
    "bisbm_set_chains": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _u32p, C.c_void_p, C.c_double]),
    "bisbm_set_chains_u8": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _u32p, C.c_void_p, C.c_double]),
    "bisbm_randomize": (C.c_int, [C.c_void_p, _u64p]),
    "bisbm_replay_init": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int]),
    "bisbm_replay_anneal": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_float, C.c_float, C.c_uint64, C.c_uint64,
                                      _dp, _u64p]),
    "bisbm_replay_step": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_double, C.POINTER(C.c_int)]),
    "bisbm_replay_transition": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, _dp, _dp]),
    "bisbm_replay_get_vlist": (C.c_int, [C.c_void_p, C.c_uint32, _u32p]),
    "bisbm_replay_rng_words": (C.c_int, [C.c_void_p, C.c_uint32, _u64p, _u64p]),
    "bisbm_replay_agg_merge": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_uint32]),
    "bisbm_replay_agg_merge_total": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_uint32]),
    "bisbm_chain_k": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _u32p]),
    "bisbm_anneal": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_uint64, C.c_uint64, _u64p, C.c_uint32,
                               _dp, _u64p]),
    "bisbm_marginalize": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, _u64p, C.c_uint32]),
    "bisbm_marginals_clear": (C.c_int, [C.c_void_p]),
    "bisbm_marginal_sample": (C.c_int, [C.c_void_p]),
    "bisbm_marginals_align": (C.c_int, [C.c_void_p, _u32p]),
    "bisbm_marginals_alignment": (C.c_int, [C.c_void_p, _u32p]),
    "bisbm_tempering_set": (C.c_int, [C.c_void_p, C.c_uint32, _dp, _u32p]),
    "bisbm_tempering_run": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, _u64p, C.c_uint64, C.c_uint32, _dp]),
    "bisbm_tempering_stats": (C.c_int, [C.c_void_p, _u32p, _u64p, _u64p, _u64p, _u64p, _u64p]),
    "bisbm_set_precision": (C.c_int, [C.c_void_p, C.c_int]),
    "bisbm_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "bisbm_parallel_transition": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, _dp, _dp]),
    "bisbm_sweep_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                   C.POINTER(C.c_uint32)]),
    "bisbm_nccl_get_unique_id": (C.c_int, [C.c_void_p]),
    "bisbm_nccl_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bisbm_marginals_allreduce": (C.c_int, [C.c_void_p]),
    "bisbm_marginals_allreduce_local": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "bisbm_marginals_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), _u64p, _u32p]),
    "bisbm_get_marginals": (C.c_int, [C.c_void_p, _u32p]),
    "bisbm_marginal_argmax": (C.c_int, [C.c_void_p, _u32p]),
    "bisbm_last_timing": (C.c_int, [C.c_void_p, _dp, _u64p, _u64p]),
    "bisbm_sweep_launches": (C.c_int, [C.c_void_p, _u64p]),
    "bisbm_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "bisbm_info": (C.c_int, [C.c_void_p, _u32p, _u64p, _u32p, _u32p]),
    "bisbm_get_labels": (C.c_int, [C.c_void_p, C.c_uint32, _u32p]),
    "bisbm_get_all_labels": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bisbm_get_all_labels_u8": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bisbm_get_m": (C.c_int, [C.c_void_p, C.c_uint32, _i32p]),
    "bisbm_get_m_r": (C.c_int, [C.c_void_p, C.c_uint32, _i32p]),
    "bisbm_get_n_r": (C.c_int, [C.c_void_p, C.c_uint32, _i32p]),
    "bisbm_get_eta": (C.c_int, [C.c_void_p, C.c_uint32, _u32p]),
    "bisbm_entropy": (C.c_int, [C.c_void_p, C.c_uint32, _dp]),
    "bisbm_entropy_all": (C.c_int, [C.c_void_p, _dp]),
    "bisbm_occupied_blocks": (C.c_int, [C.c_void_p, _u32p]),
    "bisbm_entropy_accum": (C.c_int, [C.c_void_p, C.c_uint32, _dp]),
}


def load_library(path=None):
    """dlopen libbisbm.so and bind every entry point; raises if the library is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("BISBM_LIB") or LIB_PATH   # BISBM_LIB: developer knob for A/B builds of the library
    if not os.path.exists(p):
        raise BisbmError(-1, "%s not found: build it with `python -m bipartitesbm-mcmc_b200.build` "
                             "or __graft_entry__.build(); there is no CPU fallback" % p)
    L = C.CDLL(p)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise BisbmError(rc, load_library().bisbm_last_error().decode())


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


# --------------------------------------------------------------------------- I/O helpers
def load_edge_list(path):
    """One edge per line, two whitespace-separated unsigned ints, file order kept
    (reference src/graph_utilities.cc:20-34)."""
    return np.loadtxt(path, dtype=np.uint32, ndmin=2).reshape(-1, 2)


def load_memberships(path):
    """One unsigned label per line (reference src/graph_utilities.cc:5-18)."""
    return np.loadtxt(path, dtype=np.uint32, ndmin=1)


def memberships_from_block_sizes(n):
    """Block r repeated n[r] times (reference src/mcmc_main.cc:310-317)."""
    return np.repeat(np.arange(len(n), dtype=np.uint32), np.asarray(n, dtype=np.int64))


class Graph:
    """Device-resident CSR of a bipartite multigraph (reference edge_to_adj,
    src/graph_utilities.cc:36-49: both directions pushed in file order, multi-edges kept)."""

    def __init__(self, edges, na, nb, device=0):
        """edges: [E][2] node ids -- or the TEXT of an edge-list file (bytes / str), parsed on the device
        (bisbm_create_from_text; reference load_edge_list, src/graph_utilities.cc:20-34)."""
        L = load_library()
        h = C.c_void_p()
        if isinstance(edges, (bytes, bytearray, str)):
            text = edges.encode() if isinstance(edges, str) else bytes(edges)
            _check(L.bisbm_create_from_text(na, nb, text, len(text), device, C.byref(h)))
            ne = C.c_uint64()
            _check(L.bisbm_info(h, None, C.byref(ne), None, None))
            n_edges = ne.value
        else:
            edges = np.ascontiguousarray(edges, dtype=np.uint32).reshape(-1, 2)
            ea = np.ascontiguousarray(edges[:, 0])
            eb = np.ascontiguousarray(edges[:, 1])
            _check(L.bisbm_create(na, nb, len(ea), _p(ea, C.c_uint32), _p(eb, C.c_uint32), device, C.byref(h)))
            n_edges = len(ea)
        self.L, self.h = L, h
        self.na, self.nb, self.n = na, nb, na + nb
        self.n_edges = n_edges
        self.device = device
        md = C.c_uint32()
        _check(L.bisbm_info(h, None, None, C.byref(md), None))
        self.max_degree = md.value

    def csr(self):
        """(row_ptr [n+1], col_idx [2E]) as the library holds them"""
        rp = np.zeros(self.n + 1, dtype=np.uint32)
        col = np.zeros(max(1, 2 * self.n_edges), dtype=np.uint32)
        _check(self.L.bisbm_get_csr(self.h, _p(rp, C.c_uint32), _p(col, C.c_uint32)))
        return rp, col[:2 * self.n_edges]

    def set_option(self, name, value):
        """handle options that matter before the chains exist ('reserve_ka' / 'reserve_kb', include/bisbm.h)"""
        _check(self.L.bisbm_set_option(self.h, name.encode(), int(value)))

    def close(self):
        if getattr(self, "h", None):
            self.L.bisbm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def nccl_unique_id():
    """128 bytes identifying a new NCCL communicator (rank 0 calls this, every rank passes it to ChainPool.nccl_init)."""
    buf = (C.c_uint8 * 128)()
    _check(load_library().bisbm_nccl_get_unique_id(buf))
    return bytes(buf)


def grid_search(graph, points, restarts, epsilon, schedule, p0, p1, duration, steps_await, seed=1, max_inflight=0):
    """det_k_bisbm-style (Ka, Kb) search over the C ABI (bisbm_grid_search): returns (entropy [points][restarts],
    acceptance [points][restarts], (best point index, best restart), best labels [n], stats dict)."""
    if isinstance(schedule, str):
        schedule = SCHEDULES[schedule]
    pts = np.asarray(points, dtype=np.uint32).reshape(-1, 2)
    ka = np.ascontiguousarray(pts[:, 0]); kb = np.ascontiguousarray(pts[:, 1])
    ent = np.zeros(len(pts) * restarts, dtype=np.float64)
    acc = np.zeros(len(pts) * restarts, dtype=np.float64)
    best = C.c_uint32()
    lab = np.zeros(graph.n, dtype=np.uint32)
    stats = np.zeros(8, dtype=np.float64)
    _check(graph.L.bisbm_grid_search(graph.h, len(pts), _p(ka, C.c_uint32), _p(kb, C.c_uint32), restarts, float(epsilon),
                                     schedule, p0, p1, duration, steps_await, seed, max_inflight, _p(ent, C.c_double),
                                     _p(acc, C.c_double), C.byref(best), _p(lab, C.c_uint32), _p(stats, C.c_double)))
    rows = np.zeros((64, 8), dtype=np.float64)
    nrows = C.c_uint32()
    _check(graph.L.bisbm_grid_search_report(graph.h, 64, _p(rows, C.c_double), C.byref(nrows)))
    report = [{"KA": int(r[0]), "KB": int(r[1]), "chains": int(r[2]), "kernel": int(r[3]), "setup_ms": r[4], "anneal_device_ms": r[5],
               "anneal_ms": r[6], "score_teardown_ms": r[7]} for r in rows[:min(nrows.value, 64)]]
    return (ent.reshape(len(pts), restarts), acc.reshape(len(pts), restarts), (best.value // restarts, best.value % restarts), lab,
            {"moves": stats[0], "device_ms": stats[1], "buckets": int(stats[2]), "best_entropy": stats[3], "report": report})


def grid_release(graph):
    """free the pools bisbm_grid_search keeps on the graph handle between calls"""
    _check(graph.L.bisbm_grid_release(graph.h))


def grid_k_class(graph, ka, kb):
    """(KA, KB, staged) of the pool bisbm_grid_search runs a (ka, kb) point in."""
    KA, KB, st = C.c_uint32(), C.c_uint32(), C.c_int()
    _check(graph.L.bisbm_grid_k_class(graph.h, int(ka), int(kb), C.byref(KA), C.byref(KB), C.byref(st)))
    return KA.value, KB.value, bool(st.value)


def grid_partition(graph, points, restarts, world, l2_cost=4.5, classify=None):
    """Deal the points of a (Ka, Kb) grid to `world` GPUs: points of one K bucket are kept together in chunks that fill whole
    32-chain groups (a rank given 2 points x 8 restarts of a bucket would run half-empty warps), and the chunks go to the
    least-loaded rank in order of decreasing cost (a chain whose counts stay in L2 costs ~l2_cost staged ones: measured
    1.2e9 against 5.5-6.4e9 moves/s for pools of one or two chain groups, profiles/r02_bench_c4_n8.json).
    Returns `world` lists of indices into `points`.  `classify(ka, kb) -> (KA, KB, staged)` defaults to the library's own
    bucketing (bisbm_grid_k_class)."""
    if classify is None:
        classify = lambda a, b: grid_k_class(graph, a, b)
    per_chunk = max(1, -(-32 // restarts))
    buckets = {}
    for i, (a, b) in enumerate(points):
        buckets.setdefault(tuple(classify(a, b)), []).append(i)
    chunks = []
    for (KA, KB, staged), idx in sorted(buckets.items()):
        w = 1.0 if staged else l2_cost
        for j in range(0, len(idx), per_chunk):
            part = idx[j:j + per_chunk]
            chunks.append((w * max(len(part), 0.6 * per_chunk), part))      # (a partly filled group costs most of a full one)
    chunks.sort(key=lambda x: (-x[0], x[1][0]))
    load = [0.0] * world
    out = [[] for _ in range(world)]
    for w, part in chunks:
        r = min(range(world), key=lambda k: (load[k], k))
        load[r] += w
        out[r].extend(part)
    return [sorted(o) for o in out]


def geometric_ladder(t_min, t_max, n):
    """n temperatures from t_min to t_max in constant ratio (t_min first: rung 0 is the cold one), for
    ChainPool.tempering_set; n = 1 gives [t_min]."""
    n = int(n)
    if n < 1:
        raise ValueError("a ladder needs at least one rung")
    if not (0 < t_min <= t_max < np.inf):
        raise ValueError("need 0 < t_min <= t_max < inf")
    if n == 1:
        return np.array([float(t_min)])
    out = t_min * (t_max / t_min) ** (np.arange(n) / (n - 1))
    out[-1] = t_max
    return np.maximum.accumulate(out)


def edge_to_adj(edge_list, N, na=None, nb=None, device=0):
    """reference src/graph_utilities.cc:36-49.  The bipartition (na, nb) must be given since
    the device graph validates it; N = na + nb."""
    if na is None or nb is None:
        raise ValueError("edge_to_adj needs the type sizes na, nb (reference -y flag)")
    assert N == na + nb
    return Graph(edge_list, na, nb, device)


class ChainPool:
    """Many independent chains over one graph, all resident on the device."""

    def __init__(self, graph, labels, ka, kb, epsilon):
        self.g = graph
        self.L = graph.L
        if not (isinstance(labels, np.ndarray) and labels.dtype == np.uint8):
            labels = np.ascontiguousarray(labels, dtype=np.uint32)
        if labels.ndim == 1:
            labels = labels[None, :]
        labels = np.ascontiguousarray(labels)
        self.n_chains = labels.shape[0]
        assert labels.shape[1] == graph.n
        self.ka = np.array(np.broadcast_to(np.asarray(ka, dtype=np.uint32), (self.n_chains,)))
        self.kb = np.array(np.broadcast_to(np.asarray(kb, dtype=np.uint32), (self.n_chains,)))
        self.epsilon = float(epsilon)
        self.set_labels(labels)

    # -- state in
    def set_labels(self, labels):
        """labels: uint32 or uint8 [n_chains][n], global block ids (numpy array, or a torch tensor of that element size)."""
        ptr = labels.data_ptr() if hasattr(labels, "data_ptr") else labels.ctypes.data
        item = labels.element_size() if hasattr(labels, "element_size") else labels.dtype.itemsize
        fn = self.L.bisbm_set_chains_u8 if item == 1 else self.L.bisbm_set_chains
        _check(fn(self.g.h, self.n_chains, _p(self.ka, C.c_uint32), _p(self.kb, C.c_uint32), C.c_void_p(ptr), self.epsilon))

    def randomize(self, seeds):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        assert seeds.size == self.n_chains
        _check(self.L.bisbm_randomize(self.g.h, _p(seeds, C.c_uint64)))

    # -- parallel mode
    def anneal(self, schedule, p0, p1, duration, steps_await, seeds, max_inflight=0):
        if isinstance(schedule, str):
            schedule = SCHEDULES[schedule]
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        acc = np.zeros(self.n_chains, dtype=np.float64)
        sw = np.zeros(self.n_chains, dtype=np.uint64)
        _check(self.L.bisbm_anneal(self.g.h, schedule, p0, p1, duration, steps_await, _p(seeds, C.c_uint64),
                                   max_inflight, _p(acc, C.c_double), _p(sw, C.c_uint64)))
        return acc, sw

    def marginalize(self, burn_in, sweeps, every, seeds, max_inflight=0):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        _check(self.L.bisbm_marginalize(self.g.h, burn_in, sweeps, every, _p(seeds, C.c_uint64), max_inflight))

    # -- parallel tempering (include/bisbm.h)
    def tempering_set(self, temps, rung_of_chain=None):
        """Ladder of len(temps) non-decreasing temperatures over the pool (rung 0 = temps[0], the cold one): chains l R .. l R + R - 1
        form ladder l.  rung_of_chain [n_chains] (optional) resumes a saved rung assignment.  temps = [] clears the ladder."""
        t = np.ascontiguousarray(temps, dtype=np.float64).ravel()
        if len(t) and self.n_chains % len(t):
            raise ValueError("%d rungs do not divide %d chains" % (len(t), self.n_chains))
        if not np.all(np.isfinite(t) & (t > 0)) or np.any(np.diff(t) < 0):
            raise ValueError("temperatures must be finite, > 0 and non-decreasing")
        rp = None
        if rung_of_chain is not None:
            rung_of_chain = np.ascontiguousarray(rung_of_chain, dtype=np.uint32)
            if rung_of_chain.shape != (self.n_chains,):
                raise ValueError("rung_of_chain must have one entry per chain")
            rp = _p(rung_of_chain, C.c_uint32)
        _check(self.L.bisbm_tempering_set(self.g.h, len(t), _p(t, C.c_double) if len(t) else None, rp))

    def tempering_run(self, sweeps, swap_every, seeds, swap_seed=1, sample_every=0, max_inflight=0):
        """sweeps full sweeps at each chain's rung temperature, a swap round every swap_every sweeps, a marginal sample of the
        rung-0 chains every sample_every sweeps (0: none).  Returns the per-chain acceptance of this run."""
        if int(swap_every) < 1:
            raise ValueError("swap_every must be >= 1")
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        assert seeds.size == self.n_chains
        acc = np.zeros(self.n_chains, dtype=np.float64)
        _check(self.L.bisbm_tempering_run(self.g.h, int(sweeps), int(swap_every), int(sample_every), _p(seeds, C.c_uint64),
                                          int(swap_seed), int(max_inflight), _p(acc, C.c_double)))
        return acc

    def tempering_stats(self):
        """dict of numpy arrays: rung_of_chain [n_chains], swaps_tried / swaps_accepted [R-1] per adjacent pair, moves_tried /
        moves_accepted [R] per rung, round_trips [n_ladders]."""
        rung = np.zeros(self.n_chains, dtype=np.uint32)
        _check(self.L.bisbm_tempering_stats(self.g.h, _p(rung, C.c_uint32), None, None, None, None, None))
        R = int(rung.max()) + 1     # the library holds the ladder (however it was set): every ladder is a permutation of 0..R-1
        out = {"rung_of_chain": rung,
               "swaps_tried": np.zeros(R - 1, dtype=np.uint64), "swaps_accepted": np.zeros(R - 1, dtype=np.uint64),
               "moves_tried": np.zeros(R, dtype=np.uint64), "moves_accepted": np.zeros(R, dtype=np.uint64),
               "round_trips": np.zeros(self.n_chains // R, dtype=np.uint64)}
        u64 = lambda k: _p(out[k], C.c_uint64) if out[k].size else None
        _check(self.L.bisbm_tempering_stats(self.g.h, None, u64("swaps_tried"), u64("swaps_accepted"),
                                            u64("moves_tried"), u64("moves_accepted"), u64("round_trips")))
        return out

    def set_precision(self, mode):
        """'fp64' (default: the move is evaluated in double like the reference) or 'fp32'."""
        _check(self.L.bisbm_set_precision(self.g.h, {"fp32": 0, "fp64": 1}.get(mode, mode)))

    def set_option(self, name, value):
        """Tuning options of the parallel sweep: 'inflight_div', 'kernel', 'generic' (include/bisbm.h)."""
        _check(self.L.bisbm_set_option(self.g.h, name.encode(), int(value)))

    def parallel_transition(self, chain, v, s):
        """(dS, log accu_r) of moving v to global block s, by the parallel sweep kernel's own device code."""
        dS, la = C.c_double(), C.c_double()
        _check(self.L.bisbm_parallel_transition(self.g.h, chain, v, s, C.byref(dS), C.byref(la)))
        return dS.value, la.value

    def sweep_info(self):
        """(kernel, warps per CTA, CTAs per chain group, slice) of the last parallel call; kernel 3 = sweep2<double>,
        2 = sweep2<float>, 5 / 4 = sweep2<double / float> with counts in L2, 0 = round-1 kernel, counts in L2."""
        k, w, c, sl = C.c_int(), C.c_uint32(), C.c_uint32(), C.c_uint32()
        _check(self.L.bisbm_sweep_info(self.g.h, C.byref(k), C.byref(w), C.byref(c), C.byref(sl)))
        return k.value, w.value, c.value, sl.value

    def marginals_clear(self):
        _check(self.L.bisbm_marginals_clear(self.g.h))

    def nccl_init(self, nranks, rank, unique_id):
        """Collective: join the NCCL communicator of the marginal all-reduce (unique_id: the 128 bytes rank 0 got from
        nccl_unique_id(), passed to the other ranks by the caller)."""
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        _check(self.L.bisbm_nccl_init(self.g.h, nranks, rank, buf))

    def marginals_allreduce(self):
        """Collective: in-place NCCL all-reduce (sum) of the device-resident marginal histogram."""
        _check(self.L.bisbm_marginals_allreduce(self.g.h))

    def marginal_sample(self):
        _check(self.L.bisbm_marginal_sample(self.g.h))

    def marginals_align(self, labels):
        """Align every later marginal sample to the partition `labels` [n] (global block ids, e.g. labels(c) or
        marginal_argmax()): each chain's blocks are permuted within each type to agree with it on as many nodes as
        possible before they are counted.  None clears the reference.  Needs one (ka, kb) for the whole pool."""
        if labels is None:
            _check(self.L.bisbm_marginals_align(self.g.h, None))
            return
        ref = np.ascontiguousarray(labels, dtype=np.uint32)
        if ref.shape != (self.g.n,):
            raise ValueError("the reference needs one label per node")
        _check(self.L.bisbm_marginals_align(self.g.h, _p(ref, C.c_uint32)))

    def marginals_alignment(self):
        """[n_chains][ka + kb]: the global id each chain's block was counted as in the last aligned sample."""
        # sized from the library, not from self.ka / self.kb: while maps exist, the histogram is exactly ka + kb wide (without
        # a histogram there is no aligned sample, and the call fails without writing)
        ptr, ne, w = C.c_void_p(), C.c_uint64(), C.c_uint32()
        width = w.value if self.L.bisbm_marginals_device(self.g.h, C.byref(ptr), C.byref(ne), C.byref(w)) == 0 else 0
        out = np.zeros((self.n_chains, width), dtype=np.uint32)
        _check(self.L.bisbm_marginals_alignment(self.g.h, _p(out, C.c_uint32)))
        return out

    def stream(self):
        """cudaStream_t (as int) the handle launches on."""
        st = C.c_void_p()
        _check(self.L.bisbm_stream(self.g.h, C.byref(st)))
        return st.value or 0

    def marginals(self):
        ptr, ne, w = C.c_void_p(), C.c_uint64(), C.c_uint32()
        _check(self.L.bisbm_marginals_device(self.g.h, C.byref(ptr), C.byref(ne), C.byref(w)))
        out = np.zeros((self.g.n, w.value), dtype=np.uint32)
        _check(self.L.bisbm_get_marginals(self.g.h, _p(out, C.c_uint32)))
        return out

    def marginals_device(self):
        ptr, ne, w = C.c_void_p(), C.c_uint64(), C.c_uint32()
        _check(self.L.bisbm_marginals_device(self.g.h, C.byref(ptr), C.byref(ne), C.byref(w)))
        return ptr.value, ne.value, w.value

    def marginal_argmax(self):
        out = np.zeros(self.g.n, dtype=np.uint32)
        _check(self.L.bisbm_marginal_argmax(self.g.h, _p(out, C.c_uint32)))
        return out

    def last_timing(self):
        ms, la, mv = C.c_double(), C.c_uint64(), C.c_uint64()
        _check(self.L.bisbm_last_timing(self.g.h, C.byref(ms), C.byref(la), C.byref(mv)))
        return ms.value, la.value, mv.value

    def sweep_launches(self):
        x = C.c_uint64()
        _check(self.L.bisbm_sweep_launches(self.g.h, C.byref(x)))
        return x.value

    # -- replay mode
    def replay_init(self, chain, engine_seed, gen_seed=12345, randomize=False):
        _check(self.L.bisbm_replay_init(self.g.h, chain, engine_seed, gen_seed, 1 if randomize else 0))

    def replay_anneal(self, chain, schedule, p0, p1, duration, steps_await):
        if isinstance(schedule, str):
            schedule = SCHEDULES[schedule]
        acc, sw = C.c_double(), C.c_uint64()
        _check(self.L.bisbm_replay_anneal(self.g.h, chain, schedule, p0, p1, duration, steps_await, C.byref(acc),
                                          C.byref(sw)))
        return acc.value, sw.value

    def replay_step(self, chain, v, T):
        a = C.c_int()
        _check(self.L.bisbm_replay_step(self.g.h, chain, v, T, C.byref(a)))
        return bool(a.value)

    def replay_transition(self, chain, v, s):
        dS, ar = C.c_double(), C.c_double()
        _check(self.L.bisbm_replay_transition(self.g.h, chain, v, s, C.byref(dS), C.byref(ar)))
        return dS.value, ar.value

    def replay_vlist(self, chain):
        out = np.zeros(self.g.n, dtype=np.uint32)
        _check(self.L.bisbm_replay_get_vlist(self.g.h, chain, _p(out, C.c_uint32)))
        return out

    def replay_rng_words(self, chain):
        a, b = C.c_uint64(), C.c_uint64()
        _check(self.L.bisbm_replay_rng_words(self.g.h, chain, C.byref(a), C.byref(b)))
        return a.value, b.value

    def chain_k(self, chain):
        a, b = C.c_uint32(), C.c_uint32()
        _check(self.L.bisbm_chain_k(self.g.h, chain, C.byref(a), C.byref(b)))
        self.ka[chain], self.kb[chain] = a.value, b.value
        return a.value, b.value

    def replay_agg_merge(self, chain, diff_a, diff_b=None, nm=10):
        """blockmodel_t::agg_merge (src/blockmodel.cc:109-256) on a replay chain: (diff_a, diff_b) blocks fewer per type
        (negative: agg_split), or -- diff_b None -- diff_a merges of any type (the -u / --nature form).  Returns the new
        (ka, kb)."""
        if diff_b is None:
            _check(self.L.bisbm_replay_agg_merge_total(self.g.h, chain, diff_a, nm))
        else:
            _check(self.L.bisbm_replay_agg_merge(self.g.h, chain, diff_a, diff_b, nm))
        return self.chain_k(chain)

    # -- state out
    def labels(self, chain=None, out=None):
        if chain is None:
            if out is None:
                out = np.zeros((self.n_chains, self.g.n), dtype=np.uint32)
            ptr = out.data_ptr() if hasattr(out, "data_ptr") else out.ctypes.data
            item = out.element_size() if hasattr(out, "element_size") else out.dtype.itemsize
            fn = self.L.bisbm_get_all_labels_u8 if item == 1 else self.L.bisbm_get_all_labels
            _check(fn(self.g.h, C.c_void_p(ptr)))
            return out
        o = np.zeros(self.g.n, dtype=np.uint32)
        _check(self.L.bisbm_get_labels(self.g.h, chain, _p(o, C.c_uint32)))
        return o

    def K(self, chain):
        return int(self.ka[chain]) + int(self.kb[chain])

    def m(self, chain):
        K = self.K(chain)
        out = np.zeros((K, K), dtype=np.int32)
        _check(self.L.bisbm_get_m(self.g.h, chain, _p(out, C.c_int32)))
        return out

    def m_r(self, chain):
        out = np.zeros(self.K(chain), dtype=np.int32)
        _check(self.L.bisbm_get_m_r(self.g.h, chain, _p(out, C.c_int32)))
        return out

    def n_r(self, chain):
        out = np.zeros(self.K(chain), dtype=np.int32)
        _check(self.L.bisbm_get_n_r(self.g.h, chain, _p(out, C.c_int32)))
        return out

    def eta(self, chain):
        out = np.zeros((self.K(chain), self.g.max_degree + 1), dtype=np.uint32)
        _check(self.L.bisbm_get_eta(self.g.h, chain, _p(out, C.c_uint32)))
        return out

    def entropy(self, chain=None):
        if chain is None:
            out = np.zeros(self.n_chains, dtype=np.float64)
            _check(self.L.bisbm_entropy_all(self.g.h, _p(out, C.c_double)))
            return out
        e = C.c_double()
        _check(self.L.bisbm_entropy(self.g.h, chain, C.byref(e)))
        return e.value

    def occupied_blocks(self):
        """[n_chains][2]: non-empty blocks per type (estimate mode's Ka, Kb)."""
        out = np.zeros((self.n_chains, 2), dtype=np.uint32)
        _check(self.L.bisbm_occupied_blocks(self.g.h, _p(out, C.c_uint32)))
        return out

    def entropy_accum(self, chain):
        e = C.c_double()
        _check(self.L.bisbm_entropy_accum(self.g.h, chain, C.byref(e)))
        return e.value


# --------------------------------------------------------------------------- reference-shaped classes
class mt19937:
    """Stand-in for the caller-owned std::mt19937 `engine` (reference src/mcmc_main.cc:242).
    Only its seed crosses the boundary; the stream itself is generated on the device."""

    def __init__(self, seed):
        self.seed = int(seed) & 0xFFFFFFFF
        self.bound = False


class blockmodel_t:
    """One chain with the reference's constructor and getters (src/blockmodel.hh:20-89).
    `gen_seed` stands for the reference's std::random_device draw (src/blockmodel.hh:17-18)."""

    def __init__(self, memberships, types, g, KA, KB, epsilon, adj_list_ptr, gen_seed=12345):
        assert g == KA + KB
        self.graph = adj_list_ptr
        types = np.asarray(types)
        na = int((types == 0).sum())
        assert na == self.graph.na and len(types) == self.graph.n, "types must list type-a nodes first"
        self.KA, self.KB, self.K = KA, KB, KA + KB
        self.epsilon = epsilon
        self.gen_seed = gen_seed
        self.pool = ChainPool(self.graph, np.asarray(memberships, dtype=np.uint32), KA, KB, epsilon)
        self._engine = None

    def _bind(self, engine, randomize):
        if self._engine is not engine or not engine.bound:
            self.pool.replay_init(0, engine.seed, self.gen_seed, randomize)
            engine.bound = True
            self._engine = engine
        elif randomize:
            raise BisbmError(BISBM_ERR_STATE, "shuffle_bisbm after the engine was already used")

    def shuffle_bisbm(self, engine, NA, NB):
        assert NA == self.graph.na and NB == self.graph.nb
        self._bind(engine, True)

    def init_bisbm(self):
        pass  # counts are built by the constructor (set_chains)

    def get_memberships(self):
        return self.pool.labels(0)

    def get_m(self):
        return self.pool.m(0)

    def get_m_r(self):
        return self.pool.m_r(0)

    def get_n_r(self):
        return self.pool.n_r(0)

    def get_eta_rk_(self):
        return self.pool.eta(0)

    def get_vlist(self):
        return self.pool.replay_vlist(0)

    def get_entropy(self):
        return self.pool.entropy_accum(0)

    def get_KA(self):
        return self.KA

    def get_KB(self):
        return self.KB

    def agg_merge(self, engine, diff_a, diff_b=None, nm=10):
        """src/blockmodel.cc:109-256 (both overloads: agg_merge(engine, diff_a, diff_b, nm) / agg_merge(engine, diff, nm))"""
        self._bind(engine, False)
        self.KA, self.KB = self.pool.replay_agg_merge(0, diff_a, diff_b, nm)
        self.K = self.KA + self.KB

    def get_epsilon(self):
        return self.epsilon

    def entropy(self):
        return self.pool.entropy(0)


BISBM_ERR_STATE = 3


class metropolis_hasting:
    """reference src/metropolis_hasting.hh:33-53"""

    def __init__(self):
        self.accu_r_ = 0.0

    def anneal(self, blockmodel, cooling_schedule, cooling_schedule_kwargs, duration, steps_await, engine):
        kw = list(cooling_schedule_kwargs) + [0.0, 0.0]
        blockmodel._bind(engine, False)
        acc, _ = blockmodel.pool.replay_anneal(0, cooling_schedule, kw[0], kw[1], duration, steps_await)
        return acc

    def step(self, blockmodel, vtx, temperature, engine):
        blockmodel._bind(engine, False)
        return blockmodel.pool.replay_step(0, vtx, temperature)

    def transition_ratio(self, blockmodel, moves):
        """moves: [(vertex, source, target)]; returns dS and leaves accu_r_ like the reference."""
        v, _r, s = moves[0]
        if blockmodel._engine is None:
            blockmodel._bind(mt19937(0), False)
        dS, ar = blockmodel.pool.replay_transition(0, v, s)
        self.accu_r_ = ar
        return dS


def marginals_tensor(pool):
    """The device-resident marginal histogram as a torch tensor (int32 view, no copy), for the one
    collective of the path: torch.distributed.all_reduce over NCCL."""
    import torch
    ptr, ne, _w = pool.marginals_device()

    class _Wrap:
        pass

    w = _Wrap()
    w.__cuda_array_interface__ = {"shape": (int(ne),), "typestr": "<i4", "data": (int(ptr), False), "version": 2}
    return torch.as_tensor(w, device=torch.device("cuda", pool.g.device))
