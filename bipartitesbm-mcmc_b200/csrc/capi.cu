// capi.cu -- C ABI of libbisbm.so (include/bisbm.h): handle, device state management, launches.
//
// Host side of the B200-native Metropolis-Hastings sweep.  Everything that computes runs on
// the device (kernels in replay.cuh / sweep.cuh); the host builds the exact glibc tables
// the replay mode needs, owns the device buffers and sequences the launches on one stream.
// There is no CPU execution path for any compute entry point.
#include "../../include/bisbm.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>     // types and prototypes only: libnccl.so.2 is loaded on first use (dlopen), not linked

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <set>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <vector>

#include "ingest.cuh"
#include "replay.cuh"
#include "merge.cuh"
#include "gltable.h"
#include "sweep_aux.cuh"
#include "align.cuh"
#include "sweep2.cuh"
#include "tempering.cuh"

using namespace bisbm;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(BISBM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

struct ReplaySlot {
    ReplayState* d_rs = nullptr;
    uint32_t* d_vlist = nullptr;
    int32_t* d_kh = nullptr;
};

}  // namespace

// device-resident graph + exact log q table: read-only after creation, shared (ref-counted) by every handle made
// from the same graph with bisbm_share_graph
struct GraphDev {
    int device = 0;
    uint32_t *row_ptr = nullptr, *col = nullptr, *degidx = nullptr;
    double* qtab = nullptr;
    ~GraphDev() {
        cudaSetDevice(device);
        if (row_ptr) cudaFree(row_ptr);
        if (col) cudaFree(col);
        if (degidx) cudaFree(degidx);
        if (qtab) cudaFree(qtab);
    }
};

struct bisbm_handle {
    int device = 0;
    std::shared_ptr<GraphDev> gdev;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int sm_count = 148;
    // graph
    uint32_t n = 0, na = 0, nb = 0, W = 0, max_degree = 0;
    uint64_t n_edges = 0;
    std::vector<uint32_t> h_row_ptr, h_degvals;
    uint32_t *d_row_ptr = nullptr, *d_col = nullptr, *d_degidx = nullptr;
    double ent_base = 0.0;  // label-independent entropy terms
    // tables
    double* d_qtab = nullptr;
    GlNode* d_gl = nullptr;             // tabulated g(u), lf(u) of the asymptotic log q (inside d_qtab's allocation)
    uint32_t gl_n = 0;
    uint32_t qn = 0, qk = 0;
    double* d_lg = nullptr;
    uint64_t lg_n = 0;
    // chains
    uint32_t n_chains = 0, C = 0, KA = 0, KB = 0;
    std::vector<uint32_t> h_ka, h_kb;
    uint32_t *d_ka = nullptr, *d_kb = nullptr;
    int32_t *d_labels = nullptr, *d_labels_tmp = nullptr, *d_m = nullptr, *d_e = nullptr, *d_nr = nullptr,
            *d_eta = nullptr;
    // sliced staged sweep (launch_full_sweep): the base counts rotate through three buffer sets.  A launch reads d_m / d_e / d_nr,
    // publishes into the *2 set, which is zero whenever no sliced launch is running, and zeroes the *3 set for the launch after it
    int32_t *d_m2 = nullptr, *d_e2 = nullptr, *d_nr2 = nullptr, *d_m3 = nullptr, *d_e3 = nullptr, *d_nr3 = nullptr;
    int32_t* d_nr_live[2] = {nullptr, nullptr};   // per-block decrements of n_r within one sliced launch (the exact veto);
    uint64_t nr_live_pos = 0;                     // d_nr_live[nr_live_pos & 1], zero between launches, is the next launch's
    // eta of the sliced launches: three buffers of C x KK x W, all zero between half sweeps (launch_full_sweep)
    int32_t* d_eta_ring = nullptr;
    double* d_kat_out = nullptr;               // {dS, log accu_r} of bisbm_parallel_transition
    ncclComm_t comm = nullptr;                 // bisbm_nccl_init: communicator of the marginal-histogram all-reduce
    uint8_t* d_lab8 = nullptr;                 // u8 shadow of the labels for the shared-memory sweep
    double eps = 1.0;
    LogqExp* d_lq = nullptr;
    uint64_t* d_seeds = nullptr;
    uint8_t* d_active = nullptr;
    unsigned long long *d_accepted = nullptr, *d_u = nullptr, *d_sweeps = nullptr;
    double *d_dS = nullptr, *d_entmin = nullptr, *d_ent_out = nullptr;
    uint32_t* d_nactive = nullptr;
    uint64_t sweep_epoch = 0;
    std::map<uint32_t, ReplaySlot> replay;
    // marginals
    uint32_t* d_hist = nullptr;
    uint32_t hist_width = 0;
    // label alignment of the marginal samples (bisbm_marginals_align, align.cuh): a reference is set while al_segments > 0
    uint32_t al_ka = 0, al_kb = 0, al_segments = 0;
    uint32_t *d_al_order = nullptr, *d_al_seg = nullptr, *d_al_overlap = nullptr, *d_al_map = nullptr;
    bool al_sampled = false;                   // d_al_map holds the permutations of an aligned sample
    // timing of the last parallel call
    double last_ms = 0.0;
    uint64_t last_launches = 0, last_moves = 0;
    // move arithmetic of the parallel sweep: double like the reference (default) or fp32 (sweep2.cuh)
    int precision = BISBM_PRECISION_FP64;
    // bisbm_set_option
    int opt_kernel = -1;               // -1: automatic; KERN_L2 forces the round-1 kernel, KERN_S2L_F64 sweep2 with counts in L2
    uint32_t opt_inflight_div = 64;    // default in-flight bound = half sweep / this
    int opt_generic = 0;               // 1: never take the Ka = Kb = 32 specialisation
    int opt_vary_k = 0;                // estimate mode: blocks may empty, K-dependent prior terms in dS
    uint32_t opt_warps = 16;           // warps per CTA of the staged sweep2 kernel (experiment builds: 20, 24)
    uint32_t opt_logq_every = 8;       // sliced launches between lazy refreshes of the log q expansions (0x7fffffff: only per half sweep)
    int opt_spare_sms = 1;             // 1: sliced launches hand the SMs that n_groups x ctas_per_group leaves idle to the groups in turn
    uint32_t opt_reserve_ka = 0, opt_reserve_kb = 0;   // minimum strides of the next bisbm_set_chains (room for agg_split)
    std::set<const void*> attr_done;   // kernels whose shared-memory limit is raised on this handle's device
    std::vector<double> grid_report;   // bisbm_grid_search_report: 8 numbers per K bucket of the last bisbm_grid_search
    std::map<uint64_t, bisbm_handle*> grid_pools;   // bisbm_grid_search: one pool per K bucket, kept between calls (cudaFree of GBs is slow and erratic)
    uint64_t last_sweep_launches = 0, last_marginal_launches = 0;
    uint32_t last_wpc = 0, last_cpg = 0, last_slice = 0;   // launch plan of the last half sweep
    int last_kernel = -1;                                   // KERN_* of the last parallel call
    // two label arrays, refreshed from each other on demand: the canonical i32 labels (replay, round-1 kernel, 32-bit
    // import / export) and the u8 shadow (sweep2 kernels, 8-bit import / export, marginals).  At most one is stale.
    bool lab32_stale = false;
    bool lab8_stale = true;
    // parallel tempering (bisbm_tempering_set): a ladder of tp_rungs temperatures over the pool, device-resident (LadderView)
    uint32_t tp_rungs = 0;
    uint64_t tp_round = 0;                     // swap rounds since bisbm_tempering_set: the parity and the draw of the next one
    double* d_tp_rung_beta = nullptr;
    double* d_tp_beta = nullptr;
    uint32_t *d_tp_rung_of = nullptr, *d_tp_chain_at = nullptr;
    uint8_t* d_tp_trip = nullptr;
    unsigned long long *d_tp_acc_prev = nullptr, *d_tp_stats = nullptr;
};

namespace {

template <typename T>
void dfree(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}

void free_ladder(bisbm_handle* h) {
    dfree(h->d_tp_rung_beta); dfree(h->d_tp_beta); dfree(h->d_tp_rung_of); dfree(h->d_tp_chain_at); dfree(h->d_tp_trip);
    dfree(h->d_tp_acc_prev); dfree(h->d_tp_stats);
    h->tp_rungs = 0;
    h->tp_round = 0;
}

void free_align(bisbm_handle* h) {
    dfree(h->d_al_order); dfree(h->d_al_seg); dfree(h->d_al_overlap); dfree(h->d_al_map);
    h->al_ka = h->al_kb = h->al_segments = 0;
    h->al_sampled = false;
}

void free_chains(bisbm_handle* h) {
    free_ladder(h);
    free_align(h);
    dfree(h->d_ka); dfree(h->d_kb); dfree(h->d_labels); dfree(h->d_labels_tmp);
    dfree(h->d_m); dfree(h->d_e); dfree(h->d_nr); dfree(h->d_eta); dfree(h->d_lq); dfree(h->d_m2); dfree(h->d_e2); dfree(h->d_nr2); dfree(h->d_m3); dfree(h->d_e3); dfree(h->d_nr3);
    dfree(h->d_nr_live[0]); dfree(h->d_nr_live[1]); dfree(h->d_eta_ring); dfree(h->d_kat_out); dfree(h->d_lab8);
    dfree(h->d_seeds); dfree(h->d_active); dfree(h->d_accepted); dfree(h->d_u); dfree(h->d_sweeps);
    dfree(h->d_dS); dfree(h->d_entmin); dfree(h->d_ent_out); dfree(h->d_nactive); dfree(h->d_hist);
    for (auto& kv : h->replay) { dfree(kv.second.d_rs); dfree(kv.second.d_vlist); dfree(kv.second.d_kh); }
    h->replay.clear();
    h->n_chains = 0;
}

GraphView gview(const bisbm_handle* h) {
    GraphView g;
    g.n = h->n; g.na = h->na; g.nb = h->nb; g.n_edges = h->n_edges;
    g.row_ptr = h->d_row_ptr; g.col = h->d_col; g.degidx = h->d_degidx;
    g.W = h->W; g.max_degree = h->max_degree;
    return g;
}

StateView sview(const bisbm_handle* h) {
    StateView s;
    s.C = h->C; s.KA = h->KA; s.KB = h->KB; s.W = h->W;
    s.labels = h->d_labels; s.m = h->d_m; s.e = h->d_e; s.nr = h->d_nr; s.eta = h->d_eta;
    s.ka = h->d_ka; s.kb = h->d_kb; s.eps = h->eps;
    return s;
}

// g(u), lf(u) of log_q_approx (devmath.cuh logq_gl) at u_i = exp(kGlT0 + i / kGlInvH), i < n: computed once per process with
// the reference's own fixed-point iteration and glibc, uploaded with every graph's exact table.  u = k / sqrt(n) lies in
// [n^(-1/4), sqrt(n)] for the arguments that reach the asymptotic branch (10001 <= n <= 2^32).
const double kGlT0 = -2.0, kGlInvH = 1024.0, kGlT1 = 11.6;       // u from 0.135 to 1.1e5 (a block of degree sum e <= 255 n, e >= 10001,
                                                                 // has u = n / sqrt(e) >= 0.39; smaller u takes the formula itself)
const std::vector<GlNode>& gl_table() {
    static std::vector<GlNode> tab;
    static std::once_flag once;
    std::call_once(once, []() { build_gl_table(tab, kGlT0, kGlInvH, kGlT1); });
    return tab;
}

Tables tview(const bisbm_handle* h, bool with_lgamma) {
    Tables t;
    t.lg = with_lgamma ? h->d_lg : nullptr;
    t.lg_n = with_lgamma ? h->lg_n : 0;
    t.qtab = h->d_qtab; t.qn = h->qn; t.qk = h->qk;
    t.gl = h->d_gl; t.gl_t0 = kGlT0; t.gl_inv_h = kGlInvH; t.gl_n = h->gl_n;
    return t;
}

// exact log q table, the recurrence of init_q_cache in log space (reference
// src/support/int_part.cc:30-51) restricted to rows n <= qn and columns k <= qk; cells the
// reference never writes stay -inf.  Host glibc log1p/exp so the values equal the reference's.
void build_qtab(std::vector<double>& q, uint32_t qn, uint32_t qk) {
    const size_t W = (size_t)qk + 1;
    q.assign(((size_t)qn + 1) * W, -INFINITY);
    auto lsum = [](double a, double b) {
        double mx = a > b ? a : b;
        return mx + std::log1p(std::exp(-std::fabs(a - b)));
    };
    for (size_t n = 1; n <= qn; ++n) {
        double* row = q.data() + n * W;
        row[1] = 0.0;
        const size_t kend = std::min<size_t>(n, qk);
        for (size_t k = 2; k <= kend; ++k) {
            double v = lsum(row[k], row[k - 1]);
            if (n > k) v = lsum(v, q[(n - k) * W + k]);
            row[k] = v;
        }
    }
}

int ensure_lgamma_table(bisbm_handle* h) {
    if (h->d_lg) return BISBM_OK;
    // lgamma_fast table of init_cache(E): indices 0..2E (reference src/support/cache.cc:64-91);
    // capped at 2^26 entries, beyond which the device falls back to its own lgamma
    uint64_t want = 2 * h->n_edges + 2 + h->max_degree;
    want = std::min<uint64_t>(want, 1ull << 26);
    std::vector<double> lg(want);
    lg[0] = INFINITY;
    for (uint64_t i = 1; i < want; ++i) lg[i] = std::lgamma((double)i);
    CU(cudaMalloc(&h->d_lg, want * sizeof(double)));
    CU(cudaMemcpy(h->d_lg, lg.data(), want * sizeof(double), cudaMemcpyHostToDevice));
    h->lg_n = want;
    return BISBM_OK;
}

// degree statistics shared by both creation paths: distinct degrees (compressed eta columns), the degree -> column
// table, and -sum_v lgamma(d_v + 1) from the degree histogram (fixed summation order)
void degree_stats(bisbm_handle* h, const std::vector<uint32_t>& deg, std::vector<uint32_t>& table, double* base) {
    h->max_degree = 0;
    for (uint32_t d : deg) h->max_degree = std::max(h->max_degree, d);
    std::vector<uint64_t> cnt((size_t)h->max_degree + 1, 0);
    for (uint32_t d : deg) cnt[d]++;
    h->h_degvals.clear();
    table.assign((size_t)h->max_degree + 1, 0);
    *base = 0.0;
    for (uint32_t d = 0; d <= h->max_degree; ++d)
        if (cnt[d]) {
            table[d] = (uint32_t)h->h_degvals.size();
            h->h_degvals.push_back(d);
            *base -= (double)cnt[d] * std::lgamma((double)d + 1.0);
        }
    h->W = (uint32_t)h->h_degvals.size();
}

// stream, events, exact log q table, shared graph object (after row_ptr / col / degidx are on the device)
int finish_tables(bisbm_handle* h) {
    CU(cudaSetDevice(h->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, h->device));
    h->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreate(&h->stream));
    CU(cudaEventCreate(&h->ev0));
    CU(cudaEventCreate(&h->ev1));
    // exact log q table for every (n, k) this graph can look up below the 10001 threshold
    h->qn = (uint32_t)std::min<uint64_t>(h->n_edges, 10000);
    h->qk = std::max<uint32_t>(1, std::min<uint32_t>(std::max(h->na, h->nb), h->qn));
    {
        std::vector<double> q;
        build_qtab(q, h->qn, h->qk);
        const std::vector<GlNode>& gl = gl_table();
        const size_t qpad = (q.size() + 1) / 2 * 2;       // keep the node table 16-byte aligned
        CU(cudaMalloc(&h->d_qtab, qpad * sizeof(double) + gl.size() * sizeof(GlNode)));
        CU(cudaMemcpy(h->d_qtab, q.data(), q.size() * sizeof(double), cudaMemcpyHostToDevice));
        h->d_gl = reinterpret_cast<GlNode*>(h->d_qtab + qpad);
        h->gl_n = (uint32_t)gl.size();
        CU(cudaMemcpy(h->d_gl, gl.data(), gl.size() * sizeof(GlNode), cudaMemcpyHostToDevice));
    }
    h->gdev = std::make_shared<GraphDev>();
    h->gdev->device = h->device;
    h->gdev->row_ptr = h->d_row_ptr; h->gdev->col = h->d_col; h->gdev->degidx = h->d_degidx; h->gdev->qtab = h->d_qtab;
    return BISBM_OK;
}

// ready CSR from the host (bisbm_create_csr): statistics on the host, arrays uploaded as they are
int finish_graph(bisbm_handle* h, std::vector<uint32_t>& col) {
    const uint32_t n = h->n;
    std::vector<uint32_t> deg(n), table;
    for (uint32_t v = 0; v < n; ++v) deg[v] = h->h_row_ptr[v + 1] - h->h_row_ptr[v];
    double base = 0.0;
    degree_stats(h, deg, table, &base);
    std::vector<uint32_t> degidx(n);
    for (uint32_t v = 0; v < n; ++v) degidx[v] = table[deg[v]];
    // multi-edge term of entropy() (reference src/blockmodel.cc:772-779)
    {
        std::vector<uint32_t> row;
        for (uint32_t v = 0; v < n; ++v) {
            if (deg[v] < 2) continue;
            row.assign(col.begin() + h->h_row_ptr[v], col.begin() + h->h_row_ptr[v + 1]);
            std::sort(row.begin(), row.end());
            size_t i = 0;
            while (i < row.size()) {
                size_t j = i;
                while (j < row.size() && row[j] == row[i]) ++j;
                if (j - i > 1 && v > row[i]) base += std::lgamma((double)(j - i) + 1.0);
                i = j;
            }
        }
    }
    h->ent_base = base;
    CU(cudaSetDevice(h->device));
    CU(cudaMalloc(&h->d_row_ptr, ((size_t)n + 1) * sizeof(uint32_t)));
    CU(cudaMalloc(&h->d_col, std::max<size_t>(col.size(), 1) * sizeof(uint32_t)));
    CU(cudaMalloc(&h->d_degidx, std::max<size_t>(n, 1) * sizeof(uint32_t)));
    CU(cudaMemcpy(h->d_row_ptr, h->h_row_ptr.data(), ((size_t)n + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (!col.empty()) CU(cudaMemcpy(h->d_col, col.data(), col.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (n) CU(cudaMemcpy(h->d_degidx, degidx.data(), (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return finish_tables(h);
}

// edge list -> CSR ON THE DEVICE (ingest.cuh): edge_to_adj of the reference, src/graph_utilities.cc:36-49
// on_device: ea / eb are device arrays (the text parser's output) that this function takes over and frees
int ingest_edges_device(bisbm_handle* h, const uint32_t* ea, const uint32_t* eb, bool on_device = false) {
    const uint32_t n = h->n;
    const uint64_t E = h->n_edges, E2 = 2 * E;
    CU(cudaSetDevice(h->device));
    uint32_t *d_ea = nullptr, *d_eb = nullptr, *d_keys = nullptr, *d_vals = nullptr, *d_keys2 = nullptr, *d_deg = nullptr, *d_table = nullptr;
    unsigned long long *d_bad = nullptr, *d_pk = nullptr, *d_pk2 = nullptr, *d_mult = nullptr;
    void* d_tmp = nullptr;
    if (on_device) { d_ea = const_cast<uint32_t*>(ea); d_eb = const_cast<uint32_t*>(eb); }
    auto cleanup = [&]() {
        for (void* p : {(void*)d_ea, (void*)d_eb, (void*)d_keys, (void*)d_vals, (void*)d_keys2, (void*)d_deg, (void*)d_table, (void*)d_bad,
                        (void*)d_pk, (void*)d_pk2, (void*)d_mult, d_tmp})
            if (p) cudaFree(p);
    };
#define CUI(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return fail(BISBM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } } while (0)
    CUI(cudaMalloc(&h->d_row_ptr, ((size_t)n + 1) * sizeof(uint32_t)));
    CUI(cudaMalloc(&h->d_col, std::max<uint64_t>(E2, 1) * sizeof(uint32_t)));
    CUI(cudaMalloc(&h->d_degidx, std::max<size_t>(n, 1) * sizeof(uint32_t)));
    CUI(cudaMalloc(&d_deg, ((size_t)n + 1) * sizeof(uint32_t)));
    CUI(cudaMemset(d_deg, 0, ((size_t)n + 1) * sizeof(uint32_t)));
    CUI(cudaMalloc(&d_bad, sizeof(unsigned long long)));
    CUI(cudaMemset(d_bad, 0xff, sizeof(unsigned long long)));
    std::vector<unsigned long long> mult(INGEST_MULT_BINS, 0);
    if (E) {
        if (!on_device) {
            CUI(cudaMalloc(&d_ea, E * sizeof(uint32_t)));
            CUI(cudaMalloc(&d_eb, E * sizeof(uint32_t)));
            CUI(cudaMemcpy(d_ea, ea, E * sizeof(uint32_t), cudaMemcpyHostToDevice));
            CUI(cudaMemcpy(d_eb, eb, E * sizeof(uint32_t), cudaMemcpyHostToDevice));
        }
        CUI(cudaMalloc(&d_keys, E2 * sizeof(uint32_t)));
        CUI(cudaMalloc(&d_vals, E2 * sizeof(uint32_t)));
        CUI(cudaMalloc(&d_keys2, E2 * sizeof(uint32_t)));
        const unsigned gb = (unsigned)((E + 255) / 256);
        ingest_expand_kernel<<<gb, 256>>>(d_ea, d_eb, E, n, h->na, d_keys, d_vals, d_bad);
        CUI(cudaGetLastError());
        unsigned long long bad = 0;
        CUI(cudaMemcpy(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost));
        if (bad != ~0ull) {
            const unsigned long long i = bad / 4;
            if ((bad & 3) == INGEST_BAD_RANGE) { cleanup(); return fail(BISBM_ERR_ARG, "edge %llu: node id out of range", i); }
            uint32_t xa = 0, xb = 0;
            if (on_device) { cudaMemcpy(&xa, d_ea + i, 4, cudaMemcpyDeviceToHost); cudaMemcpy(&xb, d_eb + i, 4, cudaMemcpyDeviceToHost); }
            else { xa = ea[i]; xb = eb[i]; }
            cleanup();
            return fail(BISBM_ERR_ARG, "edge %u-%u joins two nodes of the same type", xa, xb);
        }
        // stable sort of the directed entries by source node: rows in file order
        int bits = 1;
        while (bits < 32 && (1ull << bits) < (uint64_t)n) ++bits;
        size_t tmp_bytes = 0;
        CUI(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys2, d_vals, h->d_col, E2, 0, bits));
        CUI(cudaMalloc(&d_tmp, std::max<size_t>(tmp_bytes, 16)));
        CUI(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys2, d_vals, h->d_col, E2, 0, bits));
        ingest_degree_kernel<<<(unsigned)((E2 + 255) / 256), 256>>>(d_keys2, E2, d_deg);
        CUI(cudaGetLastError());
        cudaFree(d_tmp); d_tmp = nullptr;
        cudaFree(d_keys); d_keys = nullptr; cudaFree(d_vals); d_vals = nullptr; cudaFree(d_keys2); d_keys2 = nullptr;
        // multi-edge multiplicities: sort one 64-bit key per undirected edge, count runs
        CUI(cudaMalloc(&d_pk, E * sizeof(unsigned long long)));
        CUI(cudaMalloc(&d_pk2, E * sizeof(unsigned long long)));
        CUI(cudaMalloc(&d_mult, INGEST_MULT_BINS * sizeof(unsigned long long)));
        CUI(cudaMemset(d_mult, 0, INGEST_MULT_BINS * sizeof(unsigned long long)));
        ingest_pair_keys_kernel<<<gb, 256>>>(d_ea, d_eb, E, d_pk);
        CUI(cudaGetLastError());
        tmp_bytes = 0;
        CUI(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, d_pk, d_pk2, E, 0, 32 + bits));
        CUI(cudaMalloc(&d_tmp, std::max<size_t>(tmp_bytes, 16)));
        CUI(cub::DeviceRadixSort::SortKeys(d_tmp, tmp_bytes, d_pk, d_pk2, E, 0, 32 + bits));
        ingest_multiplicity_kernel<<<gb, 256>>>(d_pk2, E, d_mult);
        CUI(cudaGetLastError());
        CUI(cudaMemcpy(mult.data(), d_mult, INGEST_MULT_BINS * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        if (mult[INGEST_MULT_BINS - 1]) { cleanup(); return fail(BISBM_ERR_ARG, "an edge is repeated %d times or more", INGEST_MULT_BINS - 1); }
    }
    // row offsets = exclusive scan of the degrees
    {
        size_t tmp_bytes = 0;
        if (d_tmp) { cudaFree(d_tmp); d_tmp = nullptr; }
        CUI(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_deg, h->d_row_ptr, (int)(n + 1)));
        CUI(cudaMalloc(&d_tmp, std::max<size_t>(tmp_bytes, 16)));
        CUI(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_deg, h->d_row_ptr, (int)(n + 1)));
    }
    h->h_row_ptr.resize((size_t)n + 1);
    CUI(cudaMemcpy(h->h_row_ptr.data(), h->d_row_ptr, ((size_t)n + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    std::vector<uint32_t> deg(n), table;
    for (uint32_t v = 0; v < n; ++v) deg[v] = h->h_row_ptr[v + 1] - h->h_row_ptr[v];
    double base = 0.0;
    degree_stats(h, deg, table, &base);
    for (int L = 2; L < INGEST_MULT_BINS; ++L)
        if (mult[L]) base += (double)mult[L] * std::lgamma((double)L + 1.0);
    h->ent_base = base;
    CUI(cudaMalloc(&d_table, table.size() * sizeof(uint32_t)));
    CUI(cudaMemcpy(d_table, table.data(), table.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if (n) {
        ingest_degidx_kernel<<<(n + 255) / 256, 256>>>(d_deg, n, d_table, h->d_degidx);
        CUI(cudaGetLastError());
    }
    CUI(cudaDeviceSynchronize());
#undef CUI
    cleanup();
    return finish_tables(h);
}

int need_chains(bisbm_handle* h) {
    if (!h) return fail(BISBM_ERR_ARG, "null handle");
    if (h->n_chains == 0) return fail(BISBM_ERR_STATE, "no chains: call bisbm_set_chains first");
    CU(cudaSetDevice(h->device));
    return BISBM_OK;
}

// cudaFuncSetAttribute is per DEVICE and a handle lives on one device: remember per handle which kernels have
// their dynamic shared memory limit raised
int ensure_smem_attr(bisbm_handle* h, const void* fn, int bytes) {
    if (h->attr_done.count(fn)) return BISBM_OK;
    CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    h->attr_done.insert(fn);
    return BISBM_OK;
}

int sync_labels8(bisbm_handle* h);
int sync_labels32(bisbm_handle* h);
void wrote_labels32(bisbm_handle* h);
void wrote_labels8(bisbm_handle* h);

int rebuild_counts(bisbm_handle* h) {
    const size_t KK = (size_t)h->KA + h->KB;
    const bool from8 = h->lab32_stale;      // the u8 shadow holds the current labels (8-bit import, sweep2 kernels)
    CU(cudaMemsetAsync(h->d_m, 0, (size_t)h->C * h->KA * h->KB * sizeof(int32_t), h->stream));
    CU(cudaMemsetAsync(h->d_e, 0, (size_t)h->C * KK * sizeof(int32_t), h->stream));
    CU(cudaMemsetAsync(h->d_nr, 0, (size_t)h->C * KK * sizeof(int32_t), h->stream));
    CU(cudaMemsetAsync(h->d_eta, 0, (size_t)h->C * KK * h->W * sizeof(int32_t), h->stream));
    const size_t staged_bytes = ((size_t)h->KA * h->KB + KK) * 128;
    if (staged_bytes <= 200 * 1024 && h->n >= 4096) {
        // m_rs / n_r accumulated per CTA in shared memory (the 2E * C atomics of compute_m stay on chip)
        int rc = from8 ? ensure_smem_attr(h, (const void*)build_counts_staged_kernel<uint8_t>, 200 * 1024)
                       : ensure_smem_attr(h, (const void*)build_counts_staged_kernel<int32_t>, 200 * 1024);
        if (rc) return rc;
        const uint32_t n_groups = h->C / 32;
        const uint32_t cpg = std::max<uint32_t>(1, (uint32_t)h->sm_count / n_groups);
        if (from8) build_counts_staged_kernel<uint8_t><<<n_groups * cpg, 1024, staged_bytes, h->stream>>>(gview(h), sview(h), h->d_lab8, h->n_chains, cpg);
        else build_counts_staged_kernel<int32_t><<<n_groups * cpg, 1024, staged_bytes, h->stream>>>(gview(h), sview(h), h->d_labels, h->n_chains, cpg);
        const uint32_t tot = h->n_chains * (uint32_t)KK;
        build_e_kernel<<<(tot + 255) / 256, 256, 0, h->stream>>>(sview(h), h->n_chains);
        CU(cudaGetLastError());
        return BISBM_OK;
    }
    const uint32_t wpc = 8;
    const uint64_t warps = (uint64_t)h->n * (h->C / 32);
    if (warps) {
        const uint64_t blocks = (warps + wpc - 1) / wpc;
        if (blocks > 0x7fffffffull) return fail(BISBM_ERR_ARG, "n * chains too large for one launch");
        if (from8) build_counts_kernel<uint8_t><<<(unsigned)blocks, wpc * 32, 0, h->stream>>>(gview(h), sview(h), h->d_lab8, h->n_chains);
        else build_counts_kernel<int32_t><<<(unsigned)blocks, wpc * 32, 0, h->stream>>>(gview(h), sview(h), h->d_labels, h->n_chains);
    }
    const uint32_t tot = h->n_chains * (uint32_t)KK;
    build_e_kernel<<<(tot + 255) / 256, 256, 0, h->stream>>>(sview(h), h->n_chains);
    CU(cudaGetLastError());
    return BISBM_OK;
}

ReplayCtx rctx(bisbm_handle* h, uint32_t chain, const ReplaySlot& sl) {
    ReplayCtx x;
    x.g = gview(h);
    x.c = chain_ref(sview(h), chain, h->h_ka[chain], h->h_kb[chain]);
    x.tb = tview(h, true);
    x.rs = sl.d_rs;
    x.vlist = sl.d_vlist;
    x.kh = sl.d_kh;
    x.kt = reinterpret_cast<uint32_t*>(sl.d_kh + std::max(h->KA, h->KB));
    x.eps = h->eps;
    return x;
}

int need_replay(bisbm_handle* h, uint32_t chain, ReplaySlot** out) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    auto it = h->replay.find(chain);
    if (it == h->replay.end()) return fail(BISBM_ERR_STATE, "chain %u: call bisbm_replay_init first", chain);
    *out = &it->second;
    rc = sync_labels32(h);      // replay reads and writes the canonical labels
    if (rc) return rc;
    wrote_labels32(h);
    return BISBM_OK;
}

// host-side reference schedules (glibc pow / log), for the replay temperature arrays and
// the cold-step bookkeeping; same expressions as reference src/metropolis_hasting.cc:10-37
double host_schedule(int schedule, float p0, float p1, uint64_t t) {
    switch (schedule) {
        case BISBM_EXPONENTIAL: return (double)p0 * std::pow((double)p1, (double)t);
        case BISBM_LINEAR: { volatile float pr = p1 * (float)t; volatile float r = p0 - pr; return (double)r; }
        case BISBM_LOGARITHMIC: {
            float x = (float)t + p1;
            uint64_t i = (uint64_t)x;
            double l = (i == 0) ? 0.0 : std::log((double)i);
            return (double)p0 / l;
        }
        case BISBM_CONSTANT: return (double)p0;
        default: return ((float)t < p0) ? 1.0 : 0.0;
    }
}

// number of steps t in [t0, t1) with T(t) < 1; every schedule is non-increasing in t
uint64_t cold_steps(int schedule, float p0, float p1, uint64_t t0, uint64_t t1) {
    if (t1 <= t0) return 0;
    if (host_schedule(schedule, p0, p1, t0) < 1.0) return t1 - t0;
    if (!(host_schedule(schedule, p0, p1, t1 - 1) < 1.0)) return 0;
    uint64_t lo = t0, hi = t1 - 1;  // T(lo) >= 1, T(hi) < 1
    while (hi - lo > 1) {
        uint64_t mid = lo + (hi - lo) / 2;
        if (host_schedule(schedule, p0, p1, mid) < 1.0) hi = mid; else lo = mid;
    }
    return t1 - hi;
}

// The reference validates the schedule parameters in main() (src/mcmc_main.cc:134-218); anneal() itself trusts
// them.  The library rejects what would make a temperature negative or NaN anywhere in the call (a negative T turns
// the accept rule of step() upside down and lets cross-type proposals through).
int validate_schedule(int schedule, float p0, float p1, uint64_t duration) {
    if (schedule < 0 || schedule > 4) return fail(BISBM_ERR_ARG, "unknown cooling schedule %d", schedule);
    if (!std::isfinite(p0) || !std::isfinite(p1)) return fail(BISBM_ERR_ARG, "cooling schedule parameters must be finite");
    const uint64_t last = duration ? duration - 1 : 0;
    switch (schedule) {
        case BISBM_EXPONENTIAL:
            if (p0 < 0.f || p1 < 0.f) return fail(BISBM_ERR_ARG, "exponential schedule: T_0 and alpha must be >= 0");
            break;
        case BISBM_LINEAR:
            if (p1 < 0.f || host_schedule(schedule, p0, p1, last) < 0.0 || p0 < 0.f)
                return fail(BISBM_ERR_ARG, "linear schedule: T_0 - eta * t must stay >= 0 over the call");
            break;
        case BISBM_LOGARITHMIC:
            if (p0 < 0.f || p1 < 0.f) return fail(BISBM_ERR_ARG, "logarithmic schedule: c and d must be >= 0");
            break;
        case BISBM_CONSTANT:
            if (p0 < 0.f) return fail(BISBM_ERR_ARG, "constant schedule: temperature must be >= 0");
            break;
        default: break;
    }
    return BISBM_OK;
}

// kernels of the parallel sweep (bisbm_sweep_info reports which one ran; ids 1, 6 and 7 are retired and not reused)
enum { KERN_L2 = 0, KERN_S2_F32 = 2, KERN_S2_F64 = 3, KERN_S2L_F32 = 4, KERN_S2L_F64 = 5 };
static inline bool kern_is_s2(int k) { return k >= KERN_S2_F32; }
static inline bool kern_is_s2_staged(int k) { return k == KERN_S2_F32 || k == KERN_S2_F64; }
static inline bool kern_is_f32(int k) { return k == KERN_S2_F32 || k == KERN_S2L_F32; }

struct LaunchPlan {
    int kernel;               // KERN_*
    bool smem;                // counts staged in shared memory (KERN_S2_F32 / KERN_S2_F64)
    int hist_bytes;           // 1, 2 or 4
    uint32_t wpc;             // warps per CTA (blockDim / 32)
    uint32_t warps_used;      // of which take vertices
    uint32_t ctas_per_group;
    uint32_t slice;           // positions of the visiting order per launch
    size_t smem_bytes;
};

const size_t kSmemMax = 227 * 1024;

// Which kernel a parallel call uses -- decided ONCE for both half sweeps (the kernels keep different label
// arrays current: the staged ones the u8 shadow, the L2 one the i32 labels), so asymmetric K can never mix them.
int plan_kernel(const bisbm_handle* h, uint32_t* wpc_out) {
    const uint32_t hb = h->max_degree <= 255u ? 1 : (h->max_degree <= 65535u ? 2 : 4);
    *wpc_out = 32;
    if (h->opt_kernel == KERN_L2) return KERN_L2;
    const bool k8 = h->KA <= 256 && h->KB <= 256;
    if (hb == 1 && k8) {
        const uint32_t rs = h->precision == BISBM_PRECISION_FP32 ? 4u : 8u;
        if (h->opt_kernel != KERN_S2L_F64)
            for (uint32_t w : {h->opt_warps, 16u, 8u, 4u})
                if (sweep2_layout(h->KA, h->KB, 0, w, rs).total <= kSmemMax && sweep2_layout(h->KA, h->KB, 1, w, rs).total <= kSmemMax) {
                    *wpc_out = w;
                    return rs == 4 ? KERN_S2_F32 : KERN_S2_F64;
                }
        // larger still: the same kernel with m_rs / e_r / n_r in L2
        for (uint32_t w : {16u, 8u, 4u})
            if (sweep2_layout(h->KA, h->KB, 0, w, rs, false).total <= kSmemMax && sweep2_layout(h->KA, h->KB, 1, w, rs, false).total <= kSmemMax) {
                *wpc_out = w;
                return rs == 4 ? KERN_S2L_F32 : KERN_S2L_F64;
            }
    }
    return KERN_L2;
}

// How one half sweep is cut into launches.  `max_inflight` bounds the number of moves of one
// chain that may be evaluated against counts that do not yet include each other:
//   one CTA per chain group  -> warps_used concurrent moves (shared-memory counts are exact)
//   several CTAs per group   -> one slice of the visiting order per launch (a CTA sees the other
//                               CTAs' moves of the same slice only in the next launch)
int plan_sweep(bisbm_handle* h, uint32_t type, uint32_t max_inflight, int kernel, uint32_t wpc, LaunchPlan* lp) {
    const uint32_t nv = type ? h->nb : h->na;
    const uint32_t n_groups = h->C / 32;
    const uint32_t hb = h->max_degree <= 255u ? 1 : (h->max_degree <= 65535u ? 2 : 4);
    lp->hist_bytes = (int)hb;
    lp->kernel = kernel;
    lp->smem = kern_is_s2_staged(kernel);
    if (kernel == KERN_L2) {
        wpc = 32;
        if (sweep_smem_bytes(h->KA, h->KB, type, wpc, hb) > 220 * 1024) wpc = 16;
        if (sweep_smem_bytes(h->KA, h->KB, type, wpc, hb) > 220 * 1024)
            return fail(BISBM_ERR_ARG, "K too large for the shared-memory histogram");
    }
    // default bound: 1/inflight_div of the half sweep (DESIGN.md 4) -- also on small graphs, where it means
    // fewer busy warps rather than a looser bound
    const uint32_t inflight = max_inflight ? max_inflight : std::max<uint32_t>(1, nv / std::max<uint32_t>(1, h->opt_inflight_div));
    // CTAs per group: fill the SMs, but never more warps than the in-flight bound or the work allows
    uint32_t cpg = std::max<uint32_t>(1, (uint32_t)h->sm_count / n_groups);
    cpg = std::min<uint32_t>(cpg, std::max<uint32_t>(1, inflight / wpc));
    cpg = std::min<uint32_t>(cpg, std::max<uint32_t>(1, nv / (wpc * 4)));
    lp->ctas_per_group = cpg;
    lp->wpc = wpc;
    lp->warps_used = (cpg == 1) ? std::max<uint32_t>(1, std::min<uint32_t>(wpc, std::min<uint32_t>(inflight, std::max<uint32_t>(nv, 1)))) : wpc;
    // slices only exist for staged counts shared by several CTAs; global counts are live for everybody.
    // A whole number of vertices per warp keeps the CTAs' shares equal.
    if (lp->smem && cpg > 1) {
        lp->slice = std::max<uint32_t>(cpg * wpc, std::min<uint32_t>(inflight, nv));
        lp->slice = std::max<uint32_t>(cpg * wpc, lp->slice / (cpg * wpc) * (cpg * wpc));
    }
    else lp->slice = std::max<uint32_t>(nv, 1);
    if (kern_is_s2(kernel))
        lp->smem_bytes = sweep2_layout(h->KA, h->KB, type, wpc, kern_is_f32(kernel) ? 4u : 8u, lp->smem).total;
    else
        lp->smem_bytes = sweep_smem_bytes(h->KA, h->KB, type, wpc, hb);
    return BISBM_OK;
}

template <typename HistT, int NT>
int launch_sweep_t(bisbm_handle* h, const SweepParams& P, const LaunchPlan& lp) {
    int rc = ensure_smem_attr(h, (const void*)sweep_kernel<HistT, NT>, 220 * 1024);
    if (rc) return rc;
    const unsigned grid = P.n_groups * lp.ctas_per_group;
    sweep_kernel<HistT, NT><<<grid, NT, lp.smem_bytes, h->stream>>>(P);
    {
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess)
            return fail(BISBM_ERR_CUDA, "sweep_kernel launch failed: %s (kernel %d, grid %u, %d threads, %zu bytes of shared memory)",
                        cudaGetErrorString(e), lp.kernel, grid, NT, lp.smem_bytes);
    }
    return BISBM_OK;
}

template <typename HistT>
int launch_sweep_nt(bisbm_handle* h, const SweepParams& P, const LaunchPlan& lp) {
    if (lp.wpc == 32) return launch_sweep_t<HistT, 1024>(h, P, lp);
    return launch_sweep_t<HistT, 512>(h, P, lp);
}

int launch_sweep_h(bisbm_handle* h, const SweepParams& P, const LaunchPlan& lp) {
    if (lp.hist_bytes == 1) return launch_sweep_nt<uint8_t>(h, P, lp);
    if (lp.hist_bytes == 2) return launch_sweep_nt<uint16_t>(h, P, lp);
    return launch_sweep_nt<uint32_t>(h, P, lp);
}

template <typename R, int KF, int TYPE, bool STAGED = true, int NT = 512>
int launch_sweep2_t(bisbm_handle* h, const SweepParams& P, const LaunchPlan& lp, unsigned grid) {
    int rc = ensure_smem_attr(h, (const void*)sweep2_kernel<R, KF, TYPE, STAGED, NT>, (int)kSmemMax);
    if (rc) return rc;
    cudaError_t launched = cudaSuccess;
    if (STAGED && !P.exclusive) {
        // sliced: programmatic dependent launch, so the launch's blocks start (up to griddepcontrol.wait) while the one before
        // finishes
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(lp.wpc * 32); cfg.dynamicSmemBytes = lp.smem_bytes; cfg.stream = h->stream;
        cfg.attrs = at; cfg.numAttrs = 1;
        launched = cudaLaunchKernelEx(&cfg, sweep2_kernel<R, KF, TYPE, STAGED, NT>, P);
    } else {
        sweep2_kernel<R, KF, TYPE, STAGED, NT><<<grid, lp.wpc * 32, lp.smem_bytes, h->stream>>>(P);
    }
    {
        const cudaError_t le = cudaGetLastError(), e = launched != cudaSuccess ? launched : le;
        if (e != cudaSuccess)
            return fail(BISBM_ERR_CUDA, "sweep2_kernel launch failed: %s (kernel %d, grid %u, %u warps, %zu bytes of shared memory)",
                        cudaGetErrorString(e), lp.kernel, grid, lp.wpc, lp.smem_bytes);
    }
    wrote_labels8(h);         // the sweep2 kernels only write the u8 label shadow
    return BISBM_OK;
}

template <typename R>
int launch_sweep2(bisbm_handle* h, const SweepParams& P, const LaunchPlan& lp, unsigned grid) {
    if (!kern_is_s2(lp.kernel) || lp.wpc > 24) return fail(BISBM_ERR_STATE, "internal: sweep2 launcher with the plan of kernel %d (%u warps)", lp.kernel, lp.wpc);
    if (!lp.smem) return launch_sweep2_t<R, 0, 0, false>(h, P, lp, grid);
    // compile-time strides for the common Ka = Kb = 32 pool (BASELINE configs[2])
    if (h->KA == 32 && h->KB == 32 && !h->opt_generic) {
#ifdef BISBM_WARP_VARIANTS
        if (lp.wpc == 24) return P.type ? launch_sweep2_t<R, 32, 1, true, 768>(h, P, lp, grid) : launch_sweep2_t<R, 32, 0, true, 768>(h, P, lp, grid);
        if (lp.wpc == 20) return P.type ? launch_sweep2_t<R, 32, 1, true, 640>(h, P, lp, grid) : launch_sweep2_t<R, 32, 0, true, 640>(h, P, lp, grid);
#endif
        return P.type ? launch_sweep2_t<R, 32, 1>(h, P, lp, grid) : launch_sweep2_t<R, 32, 0>(h, P, lp, grid);
    }
    return launch_sweep2_t<R, 0, 0>(h, P, lp, grid);
}

// one launch of the planned sweep kernel.  Kept out of line and keyed on the plan alone: launch_full_sweep's loop is cloned
// per kernel family by the optimiser, and a build of it was seen taking the sweep2 launcher with a round-1 plan.
__attribute__((noinline)) int dispatch_sweep(bisbm_handle* h, const SweepParams& P, const LaunchPlan& lp, unsigned grid) {
    switch (lp.kernel) {
        case KERN_S2_F64: case KERN_S2L_F64: return launch_sweep2<double>(h, P, lp, grid);
        case KERN_S2_F32: case KERN_S2L_F32: return launch_sweep2<float>(h, P, lp, grid);
        case KERN_L2: {
            const int rc = launch_sweep_h(h, P, lp);
            wrote_labels32(h);
            return rc;
        }
        default: return fail(BISBM_ERR_STATE, "internal: no launcher for kernel %d", lp.kernel);
    }
}

SweepParams base_params(bisbm_handle* h, uint32_t type) {
    SweepParams P;
    memset(&P, 0, sizeof P);
    P.g = gview(h); P.s = sview(h); P.tb = tview(h, false);
    P.lab8 = h->d_lab8;
    P.eta_read = h->d_eta; P.eta_commit = h->d_eta;
    P.seeds = h->d_seeds; P.active = h->d_active; P.accepted = h->d_accepted; P.dS_accum = h->d_dS;
    P.lq = h->d_lq;
    P.n_chains = h->n_chains; P.type = type; P.n_groups = h->C / 32;
    P.kopp_max = type ? h->KA : h->KB;
    P.half_bits = feistel_half_bits(type ? h->nb : h->na);
    P.kat_out = h->d_kat_out;
    P.vary_k = (uint32_t)h->opt_vary_k;
    return P;
}

// one full sweep = type-a half sweep + type-b half sweep (each preceded by the log q refresh
// of the blocks that half sweep changes)
// beta_chain (device, [C], may be null): per-chain 1/T of parallel tempering, which replaces the schedule
int launch_full_sweep(bisbm_handle* h, int schedule, float p0, float p1, uint64_t sweep_in_call, uint32_t max_inflight,
                      const double* beta_chain = nullptr) {
    uint32_t wpc = 32;
    const int kernel = plan_kernel(h, &wpc);
    if (!kern_is_s2(kernel)) {   // the round-1 kernel reads and writes the canonical labels
        int rc = sync_labels32(h);
        if (rc) return rc;
    }
    {   // the sweep2 kernels read and write the u8 shadow (refreshed for the round-1 kernel too, which does not read it)
        int rc = sync_labels8(h);
        if (rc) return rc;
    }
    for (uint32_t type = 0; type < 2; ++type) {
        const uint32_t nv = type ? h->nb : h->na;
        if (nv == 0) continue;
        LaunchPlan lp;
        int rc = plan_sweep(h, type, max_inflight, kernel, wpc, &lp);
        if (rc) return rc;
        const uint32_t kmax = type ? h->KB : h->KA;
        const uint32_t tot = h->n_chains * kmax;
        logq_refresh_kernel<<<(tot * 16 + 127) / 128, 128, 0, h->stream>>>(sview(h), tview(h, false), h->d_lq, h->n_chains, type);
        h->last_launches += 1;
        const bool sliced = lp.smem && lp.ctas_per_group > 1;   // (only the staged sweep2 kernels are sliced)
        h->last_wpc = lp.wpc; h->last_cpg = lp.ctas_per_group; h->last_slice = lp.slice;
        h->last_kernel = kernel;
        // spare SMs: when the groups' CTAs do not fill the GPU (8 groups x 18 CTAs on 148 SMs), the rest are handed to the groups
        // in turn, one more CTA (and one more CTA's worth of positions) for `extras` groups per launch
        uint32_t extras = 0;
        const uint32_t G = h->C / 32;
        if (sliced && h->opt_spare_sms && max_inflight == 0 && (uint32_t)h->sm_count > G * lp.ctas_per_group)   // (an explicit in-flight bound is kept to the letter)
            extras = std::min<uint32_t>((uint32_t)h->sm_count - G * lp.ctas_per_group, G - 1);
        const uint32_t per_cta = lp.slice / std::max<uint32_t>(1, lp.ctas_per_group);
        const size_t n_eta = (size_t)h->C * (h->KA + h->KB) * h->W;
        int32_t* const eta_S[3] = {h->d_eta_ring, h->d_eta_ring + n_eta, h->d_eta_ring + 2 * n_eta};
        int32_t *last_read = nullptr, *last_commit = nullptr;
        for (uint32_t l = 0;; ++l) {
            // the group that has been handed the fewest extra slots (the last one) decides when the half sweep is over
            const uint64_t pos = extras ? ((uint64_t)l * lp.ctas_per_group + ((uint64_t)l * extras) / G) * per_cta : (uint64_t)l * lp.slice;
            if (pos >= nv) break;
            if (sliced && l != 0 && l % h->opt_logq_every == 0) {
                // the blocks whose (e_r, n_r) have left the inner part of their log q expansion's range are expanded again
                logq_refresh_kernel<<<(tot * 16 + 127) / 128, 128, 0, h->stream>>>(sview(h), tview(h, false), h->d_lq, h->n_chains, type, 1u);
                h->last_launches += 1;
            }
            SweepParams P = base_params(h, type);
            if (sliced) {
                // launch l reads eta as it was at its start, S_l, which no launch writes meanwhile: what other CTAs commit is not
                // seen, so the result does not depend on their timing.  It commits into S_{l+1} (zero at its start) and adds S_l
                // there too, so S_{l+1} ends as eta at the start of launch l + 1; it zeroes S_{l+2}.  S_0 is eta itself, then
                // the three ring buffers take turns.
                P.eta_read = (l == 0) ? h->d_eta : eta_S[(l - 1) % 3];
                P.eta_commit = eta_S[l % 3];
                P.eta_zero = eta_S[(l + 1) % 3];
                // counts: read d_m (base), publish into d_m2 (zero), zero d_m3 (the previous base)
                P.m_next = h->d_m2; P.e_next = h->d_e2; P.nr_next = h->d_nr2;
                P.m_zero = h->d_m3; P.e_zero = h->d_e3; P.nr_zero = h->d_nr3;
                P.nr_live = h->d_nr_live[h->nr_live_pos & 1]; P.nr_live_zero = h->d_nr_live[(h->nr_live_pos + 1) & 1];
                last_read = (l == 0) ? nullptr : eta_S[(l - 1) % 3];
                last_commit = P.eta_commit;
            }
            P.ctas_per_group = lp.ctas_per_group; P.warps_used = lp.warps_used;
            P.pos_begin = (uint32_t)pos; P.pos_end = (uint32_t)std::min<uint64_t>(nv, pos + lp.slice);
            P.exclusive = sliced ? 0 : 1;
            P.sweep = h->sweep_epoch;
            P.step_base = sweep_in_call * (uint64_t)h->n + (type ? h->na : 0);
            P.schedule = schedule; P.p0 = p0; P.p1 = p1; P.beta0 = (p0 == 0.0f) ? -1.0 : 1.0 / (double)p0;     // (beta0 < 0: T == 0)
            if (schedule == BISBM_ABRUPT_COOL) {
                // T(t) = 1 for t < p0, else 0 (src/metropolis_hasting.cc:33-37): a half sweep that lies on one side of the
                // switch runs as constant T (beta0 < 0 means T == 0) -- no per-vertex schedule evaluation
                const uint64_t lo = P.step_base, hi = P.step_base + nv;      // steps of this half sweep: [lo, hi)
                if ((float)(hi - 1) < p0) { P.schedule = BISBM_CONSTANT; P.p0 = 1.0f; P.beta0 = 1.0; }
                else if (!((float)lo < p0)) { P.schedule = BISBM_CONSTANT; P.p0 = 0.0f; P.beta0 = -1.0; }
            }
            P.beta_chain = beta_chain;
            P.extras = extras; P.launch_idx = l; P.per_cta = per_cta;
            const unsigned grid = P.n_groups * lp.ctas_per_group + extras;
            rc = dispatch_sweep(h, P, lp, grid);
            if (rc) return rc;
            h->last_launches += 1;
            h->last_sweep_launches += 1;
            if (sliced) {
                int32_t* t = h->d_m; h->d_m = h->d_m2; h->d_m2 = h->d_m3; h->d_m3 = t;
                t = h->d_e; h->d_e = h->d_e2; h->d_e2 = h->d_e3; h->d_e3 = t;
                t = h->d_nr; h->d_nr = h->d_nr2; h->d_nr2 = h->d_nr3; h->d_nr3 = t;
                h->nr_live_pos += 1;
            }
        }
        if (last_commit) {
            // the live eta (read by the other kernels and the host) := the buffer the last launch committed into
            const uint32_t kown = type ? h->KB : h->KA, tot_eta = G * kown * h->W * 32u;
            eta_publish_kernel<<<(tot_eta + 255) / 256, 256, 0, h->stream>>>(h->d_eta, last_commit, last_read, G, h->KA + h->KB,
                                                                            type ? h->KA : 0u, kown, h->W);
            h->last_launches += 1;
        }
    }
    h->sweep_epoch++;
    h->last_moves += (uint64_t)h->n * h->n_chains;
    return BISBM_OK;
}

// refresh the u8 label shadow from the canonical i32 labels (replay moves, 32-bit set_chains, randomize and the round-1
// kernel only write the canonical array); no-op while the shadow is current
int sync_labels8(bisbm_handle* h) {
    if (!h->lab8_stale) return BISBM_OK;
    const uint64_t total = (uint64_t)h->n * h->C;
    const uint64_t threads = (total + 3) / 4;
    labels8_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, h->stream>>>(h->d_labels, h->d_lab8, total);
    CU(cudaGetLastError());
    h->lab8_stale = false;
    return BISBM_OK;
}

// refresh the canonical i32 labels from the u8 shadow (the sweep2 kernels and the 8-bit import only write the shadow);
// called by whatever reads the canonical array, not eagerly
int sync_labels32(bisbm_handle* h) {
    if (!h->lab32_stale) return BISBM_OK;
    const uint64_t total = (uint64_t)h->n * h->C;
    const uint64_t threads = (total + 3) / 4;
    labels32_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, h->stream>>>(h->d_lab8, h->d_labels, total);
    CU(cudaGetLastError());
    h->lab32_stale = false;
    return BISBM_OK;
}
// after a kernel wrote the canonical labels only / the shadow only
void wrote_labels32(bisbm_handle* h) { h->lab32_stale = false; h->lab8_stale = true; }
void wrote_labels8(bisbm_handle* h) { h->lab8_stale = false; h->lab32_stale = true; }

int upload_seeds(bisbm_handle* h, const uint64_t* seeds) {
    std::vector<uint64_t> s(h->C, 0);
    for (uint32_t c = 0; c < h->n_chains; ++c) s[c] = seeds ? seeds[c] : (0x5851F42D4C957F2Dull * (c + 1));
    CU(cudaMemcpyAsync(h->d_seeds, s.data(), h->C * sizeof(uint64_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}


// ---- NCCL, loaded on first use: the only collective of the path is one all-reduce of the marginal histogram ----
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        // a process that already loaded an NCCL (e.g. through torch) keeps using that one
        api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (api.lib) {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
            api.CommInitAll = (decltype(api.CommInitAll))dlsym(api.lib, "ncclCommInitAll");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
            api.AllReduce = (decltype(api.AllReduce))dlsym(api.lib, "ncclAllReduce");
            api.GroupStart = (decltype(api.GroupStart))dlsym(api.lib, "ncclGroupStart");
            api.GroupEnd = (decltype(api.GroupEnd))dlsym(api.lib, "ncclGroupEnd");
            api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
            if (!api.GetUniqueId || !api.CommInitRank || !api.CommInitAll || !api.CommDestroy || !api.AllReduce || !api.GroupStart ||
                !api.GroupEnd || !api.GetErrorString) { dlclose(api.lib); api.lib = nullptr; }
        }
    }
    return api.lib ? &api : nullptr;
}
#define NC(call)                                                                                   \
    do {                                                                                           \
        ncclResult_t r_ = (call);                                                                  \
        if (r_ != ncclSuccess)                                                                     \
            return fail(BISBM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, nccl_api()->GetErrorString(r_), __FILE__, __LINE__); \
    } while (0)

}  // namespace

extern "C" {

const char* bisbm_last_error(void) { return g_err.c_str(); }
const char* bisbm_version(void) { return "bisbm-b200 0.1 (sm_100a)"; }

int bisbm_create_csr(uint32_t na, uint32_t nb, const uint32_t* row_ptr, const uint32_t* col_idx, int device,
                     bisbm_handle** out) {
    if (!out || !row_ptr) return fail(BISBM_ERR_ARG, "null argument");
    *out = nullptr;
    const uint64_t n64 = (uint64_t)na + nb;
    if (n64 == 0 || n64 > 0xfffffff0ull) return fail(BISBM_ERR_ARG, "bad node count");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(BISBM_ERR_CUDA, "no CUDA device (libbisbm has no CPU path)");
    if (device < 0 || device >= ndev) return fail(BISBM_ERR_ARG, "device %d out of range (%d devices)", device, ndev);
    std::unique_ptr<bisbm_handle> h(new bisbm_handle());
    h->device = device;
    h->n = (uint32_t)n64; h->na = na; h->nb = nb;
    h->h_row_ptr.assign(row_ptr, row_ptr + n64 + 1);
    const uint64_t nnz = row_ptr[n64];
    if (nnz & 1) return fail(BISBM_ERR_ARG, "odd number of adjacency entries");
    h->n_edges = nnz / 2;
    if (nnz && !col_idx) return fail(BISBM_ERR_ARG, "null col_idx");
    std::vector<uint32_t> col(col_idx, col_idx + nnz);
    for (uint32_t v = 0; v < h->n; ++v) {
        if (row_ptr[v + 1] < row_ptr[v]) return fail(BISBM_ERR_ARG, "row_ptr not monotone");
        const bool va = v < na;
        for (uint32_t e = row_ptr[v]; e < row_ptr[v + 1]; ++e) {
            if (col[e] >= h->n) return fail(BISBM_ERR_ARG, "neighbour id out of range");
            if ((col[e] < na) == va) return fail(BISBM_ERR_ARG, "edge %u-%u joins two nodes of the same type", v, col[e]);
        }
    }
    int rc = finish_graph(h.get(), col);
    if (rc) { bisbm_destroy(h.release()); return rc; }
    *out = h.release();
    return BISBM_OK;
}

int bisbm_create(uint32_t na, uint32_t nb, uint64_t n_edges, const uint32_t* ea, const uint32_t* eb, int device,
                 bisbm_handle** out) {
    if (!out) return fail(BISBM_ERR_ARG, "null argument");
    *out = nullptr;
    if (n_edges && (!ea || !eb)) return fail(BISBM_ERR_ARG, "null edge arrays");
    const uint64_t n64 = (uint64_t)na + nb;
    if (n64 == 0 || n64 > 0xfffffff0ull) return fail(BISBM_ERR_ARG, "bad node count");
    if (2 * n_edges >= 0xffffffffull) return fail(BISBM_ERR_ARG, "too many edges for 32-bit row offsets");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(BISBM_ERR_CUDA, "no CUDA device (libbisbm has no CPU path)");
    if (device < 0 || device >= ndev) return fail(BISBM_ERR_ARG, "device %d out of range (%d devices)", device, ndev);
    std::unique_ptr<bisbm_handle> h(new bisbm_handle());
    h->device = device;
    h->n = (uint32_t)n64; h->na = na; h->nb = nb; h->n_edges = n_edges;
    // edge_to_adj on the device: both directions, file order within a row, multi-edges kept (reference
    // src/graph_utilities.cc:36-49); validation (id range, bipartition) included
    int rc = ingest_edges_device(h.get(), ea, eb);
    if (rc) { const std::string err = g_err; bisbm_destroy(h.release()); g_err = err; return rc; }
    *out = h.release();
    return BISBM_OK;
}

// load_edge_list on the device: text (host) -> d_ea / d_eb (device, caller frees), E = edge lines in file order
static int parse_edge_text_device(int device, const char* text, uint64_t bytes, uint32_t** d_ea_out, uint32_t** d_eb_out, uint64_t* E_out) {
    *d_ea_out = nullptr; *d_eb_out = nullptr; *E_out = 0;
    if (bytes == 0) return BISBM_OK;
    CU(cudaSetDevice(device));
    unsigned char* d_text = nullptr;
    unsigned long long *d_lines = nullptr, *d_off = nullptr, *d_bad = nullptr;
    uint32_t *d_ea = nullptr, *d_eb = nullptr;
    void* d_tmp = nullptr;
    auto cleanup = [&]() { for (void* p : {(void*)d_text, (void*)d_lines, (void*)d_off, (void*)d_bad, (void*)d_ea, (void*)d_eb, d_tmp}) if (p) cudaFree(p); };
#define CUP(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { cleanup(); return fail(BISBM_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } } while (0)
    const uint64_t chunks = (bytes + PARSE_CHUNK - 1) / PARSE_CHUNK;
    if (chunks > 0x7fffffffull) return fail(BISBM_ERR_ARG, "edge list text too large");
    CUP(cudaMalloc(&d_text, bytes + 16));
    CUP(cudaMemcpy(d_text, text, bytes, cudaMemcpyHostToDevice));
    CUP(cudaMalloc(&d_lines, (chunks + 1) * sizeof(unsigned long long)));
    CUP(cudaMalloc(&d_off, (chunks + 1) * sizeof(unsigned long long)));
    CUP(cudaMemset(d_lines, 0, (chunks + 1) * sizeof(unsigned long long)));
    CUP(cudaMalloc(&d_bad, sizeof(unsigned long long)));
    CUP(cudaMemset(d_bad, 0xff, sizeof(unsigned long long)));
    parse_edges_kernel<false><<<(unsigned)chunks, PARSE_T>>>(d_text, bytes, d_lines, nullptr, nullptr, d_bad);
    CUP(cudaGetLastError());
    size_t tmp_bytes = 0;
    CUP(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_lines, d_off, (int)(chunks + 1)));
    CUP(cudaMalloc(&d_tmp, std::max<size_t>(tmp_bytes, 16)));
    CUP(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_lines, d_off, (int)(chunks + 1)));
    unsigned long long E = 0;
    CUP(cudaMemcpy(&E, d_off + chunks, sizeof E, cudaMemcpyDeviceToHost));       // (entry `chunks` of the scan = total)
    if (E) {
        CUP(cudaMalloc(&d_ea, E * sizeof(uint32_t)));
        CUP(cudaMalloc(&d_eb, E * sizeof(uint32_t)));
        parse_edges_kernel<true><<<(unsigned)chunks, PARSE_T>>>(d_text, bytes, d_off, d_ea, d_eb, d_bad);
        CUP(cudaGetLastError());
        unsigned long long bad = 0;
        CUP(cudaMemcpy(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost));
        if (bad != ~0ull) { cleanup(); return fail(BISBM_ERR_ARG, "edge line %llu: node id does not fit 32 bits", bad); }
    }
#undef CUP
    *d_ea_out = d_ea; *d_eb_out = d_eb; *E_out = E;
    d_ea = nullptr; d_eb = nullptr;
    cleanup();
    return BISBM_OK;
}

static int check_create_args(uint32_t na, uint32_t nb, int device, bisbm_handle** out) {
    if (!out) return fail(BISBM_ERR_ARG, "null argument");
    *out = nullptr;
    const uint64_t n64 = (uint64_t)na + nb;
    if (n64 == 0 || n64 > 0xfffffff0ull) return fail(BISBM_ERR_ARG, "bad node count");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(BISBM_ERR_CUDA, "no CUDA device (libbisbm has no CPU path)");
    if (device < 0 || device >= ndev) return fail(BISBM_ERR_ARG, "device %d out of range (%d devices)", device, ndev);
    return BISBM_OK;
}

int bisbm_create_from_text(uint32_t na, uint32_t nb, const char* text, uint64_t n_bytes, int device, bisbm_handle** out) {
    int rc = check_create_args(na, nb, device, out);
    if (rc) return rc;
    if (n_bytes && !text) return fail(BISBM_ERR_ARG, "null text");
    uint32_t *d_ea = nullptr, *d_eb = nullptr;
    uint64_t E = 0;
    rc = parse_edge_text_device(device, text, n_bytes, &d_ea, &d_eb, &E);
    if (rc) return rc;
    if (2 * E >= 0xffffffffull) { cudaFree(d_ea); cudaFree(d_eb); return fail(BISBM_ERR_ARG, "too many edges for 32-bit row offsets"); }
    std::unique_ptr<bisbm_handle> h(new bisbm_handle());
    h->device = device;
    h->n = na + nb; h->na = na; h->nb = nb; h->n_edges = E;
    rc = ingest_edges_device(h.get(), d_ea, d_eb, true);         // (takes the two arrays over)
    if (rc) { const std::string err = g_err; bisbm_destroy(h.release()); g_err = err; return rc; }
    *out = h.release();
    return BISBM_OK;
}

int bisbm_get_csr(bisbm_handle* h, uint32_t* row_ptr, uint32_t* col_idx) {
    if (!h || !h->gdev) return fail(BISBM_ERR_ARG, "no graph");
    CU(cudaSetDevice(h->device));
    if (row_ptr) std::copy(h->h_row_ptr.begin(), h->h_row_ptr.end(), row_ptr);
    if (col_idx && h->n_edges) CU(cudaMemcpy(col_idx, h->gdev->col, 2 * h->n_edges * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return BISBM_OK;
}

int bisbm_destroy(bisbm_handle* h) {
    if (!h) return BISBM_OK;
    cudaSetDevice(h->device);
    for (auto& kv : h->grid_pools) bisbm_destroy(kv.second);
    h->grid_pools.clear();
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->comm && nccl_api()) { nccl_api()->CommDestroy(h->comm); h->comm = nullptr; }
    free_chains(h);
    if (h->gdev) h->gdev.reset();          // the last handle sharing the graph frees it
    else { dfree(h->d_row_ptr); dfree(h->d_col); dfree(h->d_degidx); dfree(h->d_qtab); }   // creation failed half way
    dfree(h->d_lg);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return BISBM_OK;
}

}  // extern "C"

// buffers and per-chain constants of a pool of n_chains chains (everything of bisbm_set_chains except the labels);
// *same_model: same shapes, K per chain and epsilon as the pool the handle already holds
static int alloc_chains(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb, double eps, bool* same_model_out) {
    if (!h || !ka || !kb) return fail(BISBM_ERR_ARG, "null argument");
    if (n_chains == 0) return fail(BISBM_ERR_ARG, "n_chains must be > 0");
    if (!(eps > 0.0)) return fail(BISBM_ERR_ARG, "epsilon must be > 0");
    CU(cudaSetDevice(h->device));
    free_ladder(h);      // a new pool has no ladder
    free_align(h);       // and no alignment reference
    uint32_t KA = 0, KB = 0;
    for (uint32_t c = 0; c < n_chains; ++c) {
        if (ka[c] == 0 || kb[c] == 0) return fail(BISBM_ERR_ARG, "chain %u: ka and kb must be >= 1", c);
        KA = std::max(KA, ka[c]); KB = std::max(KB, kb[c]);
    }
    KA = std::max(KA, h->opt_reserve_ka); KB = std::max(KB, h->opt_reserve_kb);
    const uint32_t C = (n_chains + 31) / 32 * 32;
    const uint32_t n = h->n;
    const size_t KK = (size_t)KA + KB;
    bool reuse = h->n_chains == n_chains && h->C == C && h->KA == KA && h->KB == KB && h->d_labels;
    // same K per chain and same epsilon as well: the counts stay valid if the labels turn out to be the ones held already
    bool same_model = reuse && h->eps == eps;
    for (uint32_t c = 0; same_model && c < n_chains; ++c) same_model = h->h_ka[c] == ka[c] && h->h_kb[c] == kb[c];
    if (!reuse) {
        free_chains(h);
        h->n_chains = n_chains; h->C = C; h->KA = KA; h->KB = KB;
        CU(cudaMalloc(&h->d_ka, C * sizeof(uint32_t)));
        CU(cudaMalloc(&h->d_kb, C * sizeof(uint32_t)));
        CU(cudaMalloc(&h->d_labels, (size_t)n * C * sizeof(int32_t)));
        CU(cudaMalloc(&h->d_labels_tmp, (size_t)n * C * sizeof(int32_t)));
        CU(cudaMalloc(&h->d_m, (size_t)C * KA * KB * sizeof(int32_t)));
        CU(cudaMalloc(&h->d_e, (size_t)C * KK * sizeof(int32_t)));
        CU(cudaMalloc(&h->d_lab8, (size_t)n * C));
        CU(cudaMalloc(&h->d_nr, (size_t)C * KK * sizeof(int32_t)));
        for (int32_t** p : {&h->d_m2, &h->d_m3}) CU(cudaMalloc(p, (size_t)C * KA * KB * sizeof(int32_t)));
        for (int32_t** p : {&h->d_e2, &h->d_e3, &h->d_nr2, &h->d_nr3, &h->d_nr_live[0], &h->d_nr_live[1]})
            CU(cudaMalloc(p, (size_t)C * KK * sizeof(int32_t)));
        CU(cudaMalloc(&h->d_kat_out, 2 * sizeof(double)));
        CU(cudaMalloc(&h->d_eta, (size_t)C * KK * h->W * sizeof(int32_t)));
        CU(cudaMalloc(&h->d_eta_ring, 3 * (size_t)C * KK * h->W * sizeof(int32_t)));
        // what must be zero when no sliced launch is running
        CU(cudaMemsetAsync(h->d_m2, 0, (size_t)C * KA * KB * sizeof(int32_t), h->stream));
        for (int32_t* p : {h->d_e2, h->d_nr2, h->d_nr_live[0], h->d_nr_live[1]}) CU(cudaMemsetAsync(p, 0, (size_t)C * KK * sizeof(int32_t), h->stream));
        CU(cudaMemsetAsync(h->d_eta_ring, 0, 3 * (size_t)C * KK * h->W * sizeof(int32_t), h->stream));
        CU(cudaMalloc(&h->d_lq, (size_t)C * KK * sizeof(LogqExp)));
        CU(cudaMalloc(&h->d_seeds, C * sizeof(uint64_t)));
        CU(cudaMalloc(&h->d_active, C));
        CU(cudaMalloc(&h->d_accepted, C * sizeof(unsigned long long)));
        CU(cudaMalloc(&h->d_u, C * sizeof(unsigned long long)));
        CU(cudaMalloc(&h->d_sweeps, C * sizeof(unsigned long long)));
        CU(cudaMalloc(&h->d_dS, C * sizeof(double)));
        CU(cudaMalloc(&h->d_entmin, C * sizeof(double)));
        CU(cudaMalloc(&h->d_ent_out, C * sizeof(double)));
        CU(cudaMalloc(&h->d_nactive, sizeof(uint32_t)));
    } else {
        // same shapes: keep the device buffers, drop per-chain replay state
        for (auto& kv : h->replay) { dfree(kv.second.d_rs); dfree(kv.second.d_vlist); dfree(kv.second.d_kh); }
        h->replay.clear();
    }
    h->eps = eps;
    h->h_ka.assign(C, 1); h->h_kb.assign(C, 1);
    std::copy(ka, ka + n_chains, h->h_ka.begin());
    std::copy(kb, kb + n_chains, h->h_kb.begin());
    CU(cudaMemsetAsync(h->d_lq, 0, (size_t)C * KK * sizeof(LogqExp), h->stream));
    CU(cudaMemsetAsync(h->d_dS, 0, C * sizeof(double), h->stream));
    CU(cudaMemsetAsync(h->d_active, 0, C, h->stream));
    CU(cudaMemsetAsync(h->d_active, 1, n_chains, h->stream));
    CU(cudaMemcpyAsync(h->d_ka, h->h_ka.data(), C * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_kb, h->h_kb.data(), C * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    *same_model_out = same_model;
    return BISBM_OK;
}

template <typename InT>
static int set_chains_impl(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb,
                           const InT* labels, double eps) {
    if (!labels) return fail(BISBM_ERR_ARG, "null argument");
    bool same_model = false;
    const bool had_chains = h->d_labels != nullptr;
    int rc0 = alloc_chains(h, n_chains, ka, kb, eps, &same_model);
    if (rc0) return rc0;
    if (!same_model || !had_chains) { h->lab32_stale = false; h->lab8_stale = true; }   // nothing to compare with
    const uint32_t n = h->n, C = h->C;
    constexpr bool kU8 = sizeof(InT) == 1;
    // host labels [chain][node], global ids  ->  chain-minor, type-local (device transpose).  8-bit labels go straight
    // into the u8 shadow (what the sweep2 kernels read); 32-bit labels into the canonical array.
    {
        InT* stage = reinterpret_cast<InT*>(h->d_labels_tmp);
        CU(cudaMemcpyAsync(stage, labels, (size_t)n_chains * n * sizeof(InT), cudaMemcpyHostToDevice, h->stream));
        unsigned long long* d_bad = reinterpret_cast<unsigned long long*>(h->d_accepted);
        uint32_t* d_changed = reinterpret_cast<uint32_t*>(h->d_accepted + 1);
        CU(cudaMemsetAsync(d_bad, 0xff, sizeof(unsigned long long), h->stream));
        CU(cudaMemsetAsync(d_changed, 0, sizeof(unsigned long long), h->stream));
        if constexpr (kU8) {
            if (same_model) { int rc = sync_labels8(h); if (rc) return rc; }
            dim3 grid((n + L8_NODES - 1) / L8_NODES, C / 32);
            // (in place: every 16-byte piece is read, compared and rewritten by one thread)
            import_labels8_kernel<<<grid, 256, 0, h->stream>>>(reinterpret_cast<const uint8_t*>(stage), h->d_lab8, n, h->na, n_chains, C,
                                                               h->d_ka, h->d_kb, d_bad, same_model ? h->d_lab8 : nullptr, d_changed);
            wrote_labels8(h);
        } else {
            if (same_model) { int rc = sync_labels32(h); if (rc) return rc; }
            dim3 grid((n + 31) / 32, C / 32), block(32, 8);
            import_labels_kernel<InT><<<grid, block, 0, h->stream>>>(stage, h->d_labels, n, h->na, n_chains, C, h->d_ka, h->d_kb, d_bad,
                                                                  same_model ? h->d_labels : nullptr, d_changed);
            wrote_labels32(h);
        }
        CU(cudaGetLastError());
        unsigned long long res[2] = {0, 0};
        CU(cudaMemcpyAsync(res, d_bad, sizeof res, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        const unsigned long long bad = res[0];
        if (same_model && bad == ~0ull && res[1] == 0) {
            // the caller handed back exactly the labels the handle holds (e.g. a checkpoint round trip): the counts
            // built from them are still right
            CU(cudaMemsetAsync(h->d_accepted, 0, 2 * sizeof(unsigned long long), h->stream));
            CU(cudaStreamSynchronize(h->stream));
            return BISBM_OK;
        }
        if (bad != ~0ull) {
            const unsigned long long idx = bad - 1;
            const uint32_t c = (uint32_t)(idx / n), v = (uint32_t)(idx % n);
            const uint32_t g = (uint32_t)labels[idx];
            free_chains(h);
            return fail(BISBM_ERR_ARG, "chain %u node %u: block %u is not a type-%c block (ka=%u kb=%u)", c, v, g,
                        v < h->na ? 'a' : 'b', ka[c], kb[c]);
        }
    }
    int rc = rebuild_counts(h);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

extern "C" {

int bisbm_set_chains(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb,
                     const uint32_t* labels, double eps) {
    return set_chains_impl<uint32_t>(h, n_chains, ka, kb, labels, eps);
}

int bisbm_set_chains_u8(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb,
                        const uint8_t* labels, double eps) {
    if (ka && kb)
        for (uint32_t c = 0; c < n_chains; ++c)
            if ((uint64_t)ka[c] + kb[c] > 256) return fail(BISBM_ERR_ARG, "chain %u: ka + kb > 256 does not fit 8-bit labels", c);
    return set_chains_impl<uint8_t>(h, n_chains, ka, kb, labels, eps);
}

int bisbm_randomize(bisbm_handle* h, const uint64_t* seeds) {
    int rc = need_chains(h);
    if (rc) return rc;
    rc = upload_seeds(h, seeds);
    if (rc) return rc;
    if (!h->d_labels_tmp) CU(cudaMalloc(&h->d_labels_tmp, (size_t)h->n * h->C * sizeof(int32_t)));
    rc = sync_labels32(h);
    if (rc) return rc;
    const uint64_t tot = (uint64_t)h->n * h->C;
    randomize_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(
        gview(h), h->d_labels, h->d_labels_tmp, h->C, h->n_chains, h->d_seeds, feistel_half_bits(h->na),
        feistel_half_bits(h->nb));
    CU(cudaGetLastError());
    std::swap(h->d_labels, h->d_labels_tmp);
    wrote_labels32(h);
    rc = rebuild_counts(h);
    if (rc) return rc;
    CU(cudaMemsetAsync(h->d_dS, 0, h->C * sizeof(double), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

// ---------------------------------------------------------------- replay mode
int bisbm_replay_init(bisbm_handle* h, uint32_t chain, uint32_t engine_seed, uint32_t gen_seed, int randomize) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    rc = ensure_lgamma_table(h);
    if (rc) return rc;
    ReplaySlot& sl = h->replay[chain];
    if (!sl.d_rs) {
        CU(cudaMalloc(&sl.d_rs, sizeof(ReplayState)));
        CU(cudaMalloc(&sl.d_vlist, (size_t)h->n * sizeof(uint32_t)));
        CU(cudaMalloc(&sl.d_kh, ((size_t)std::max(h->KA, h->KB) + 1 + RP_KT_MAX) * sizeof(int32_t)));
    }
    CU(cudaMemsetAsync(sl.d_kh, 0, ((size_t)std::max(h->KA, h->KB) + 1 + RP_KT_MAX) * sizeof(int32_t), h->stream));   // histogram + its (empty) bin list
    rc = sync_labels32(h);
    if (rc) return rc;
    replay_init_kernel<<<1, 32, 0, h->stream>>>(rctx(h, chain, sl), engine_seed, gen_seed, randomize);
    CU(cudaGetLastError());
    wrote_labels32(h);
    if (randomize) {  // compute_n_r / k / m / m_r / eta_rk after the shuffle
        rc = rebuild_counts(h);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

int bisbm_replay_anneal(bisbm_handle* h, uint32_t chain, int schedule, float p0, float p1, uint64_t duration,
                        uint64_t steps_await, double* accept_ratio, uint64_t* sweeps_done) {
    ReplaySlot* sl;
    int rc = need_replay(h, chain, &sl);
    if (rc) return rc;
    rc = validate_schedule(schedule, p0, p1, duration);
    if (rc) return rc;
    const uint64_t N = h->n;
    const uint64_t all_sweeps = duration / N;
    // anneal() resets entropy_min_, the accepted counter and u on entry
    // (reference src/metropolis_hasting.cc:71-75)
    ReplayState hs;
    CU(cudaMemcpy(&hs, sl->d_rs, sizeof hs, cudaMemcpyDeviceToHost));
    hs.entropy_min = INFINITY; hs.accepted = 0; hs.u = 0; hs.sweeps_done = 0; hs.stopped = 0;
    CU(cudaMemcpy(sl->d_rs, &hs, sizeof hs, cudaMemcpyHostToDevice));
    const bool host_temps = (schedule == BISBM_EXPONENTIAL || schedule == BISBM_LOGARITHMIC);
    const uint64_t chunk = std::max<uint64_t>(1, (1ull << 20) / std::max<uint64_t>(N, 1));
    double* d_temps = nullptr;
    std::vector<double> temps;
    if (host_temps) CU(cudaMalloc(&d_temps, chunk * N * sizeof(double)));
    uint64_t done = 0;
    uint32_t stopped = 0;
    while (done < all_sweeps && !stopped) {
        const uint64_t ns = std::min(chunk, all_sweeps - done);
        if (host_temps) {
            temps.resize(ns * N);
            for (uint64_t i = 0; i < ns * N; ++i) temps[i] = host_schedule(schedule, p0, p1, done * N + i);
            CU(cudaMemcpyAsync(d_temps, temps.data(), ns * N * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        }
        replay_anneal_kernel<<<1, 32, 0, h->stream>>>(rctx(h, chain, *sl), schedule, p0, p1, d_temps, done, ns, steps_await);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(h->stream));
        CU(cudaMemcpy(&hs, sl->d_rs, sizeof hs, cudaMemcpyDeviceToHost));
        stopped = hs.stopped;
        done += ns;
    }
    if (d_temps) cudaFree(d_temps);
    if (accept_ratio) {
        if (hs.stopped) *accept_ratio = (double)hs.accepted / (double)(hs.sweeps_done * N);
        else *accept_ratio = (double)hs.accepted / (double)duration;
    }
    if (sweeps_done) *sweeps_done = hs.sweeps_done;
    return BISBM_OK;
}

int bisbm_replay_step(bisbm_handle* h, uint32_t chain, uint32_t v, double T, int* accepted) {
    ReplaySlot* sl;
    int rc = need_replay(h, chain, &sl);
    if (rc) return rc;
    if (v >= h->n) return fail(BISBM_ERR_ARG, "vertex out of range");
    replay_step_kernel<<<1, 32, 0, h->stream>>>(rctx(h, chain, *sl), v, T);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    ReplayState hs;
    CU(cudaMemcpy(&hs, sl->d_rs, sizeof hs, cudaMemcpyDeviceToHost));
    if (accepted) *accepted = hs.last_accept;
    return BISBM_OK;
}

int bisbm_replay_transition(bisbm_handle* h, uint32_t chain, uint32_t v, uint32_t s, double* dS, double* accu_r) {
    ReplaySlot* sl;
    int rc = need_replay(h, chain, &sl);
    if (rc) return rc;
    if (v >= h->n || s >= h->h_ka[chain] + h->h_kb[chain]) return fail(BISBM_ERR_ARG, "vertex or block out of range");
    replay_transition_kernel<<<1, 32, 0, h->stream>>>(rctx(h, chain, *sl), v, s);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    ReplayState hs;
    CU(cudaMemcpy(&hs, sl->d_rs, sizeof hs, cudaMemcpyDeviceToHost));
    if (dS) *dS = hs.last_dS;
    if (accu_r) *accu_r = hs.accu_r;
    return BISBM_OK;
}

int bisbm_replay_get_vlist(bisbm_handle* h, uint32_t chain, uint32_t* vlist) {
    ReplaySlot* sl;
    int rc = need_replay(h, chain, &sl);
    if (rc) return rc;
    CU(cudaMemcpy(vlist, sl->d_vlist, (size_t)h->n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return BISBM_OK;
}

int bisbm_replay_rng_words(bisbm_handle* h, uint32_t chain, uint64_t* engine_words, uint64_t* gen_words) {
    ReplaySlot* sl;
    int rc = need_replay(h, chain, &sl);
    if (rc) return rc;
    ReplayState hs;
    CU(cudaMemcpy(&hs, sl->d_rs, sizeof hs, cudaMemcpyDeviceToHost));
    if (engine_words) *engine_words = ((uint64_t)hs.engine[626] << 32) | hs.engine[625];
    if (gen_words) *gen_words = ((uint64_t)hs.gen[626] << 32) | hs.gen[625];
    return BISBM_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- agglomerative merge / split (replay chains)
namespace {

struct MergeScratch {
    uint32_t *badj = nullptr, *badj_cnt = nullptr, *cand = nullptr, *n_cand = nullptr, *seen = nullptr, *first = nullptr, *map = nullptr;
    double* cand_dS = nullptr;
    ~MergeScratch() {
        cudaFree(badj); cudaFree(badj_cnt); cudaFree(cand); cudaFree(n_cand); cudaFree(seen); cudaFree(first); cudaFree(map); cudaFree(cand_dS);
    }
};

MergeCtx mctx(bisbm_handle* h, uint32_t chain, const ReplaySlot& sl, const MergeScratch& sc) {
    MergeCtx x;
    x.c = chain_ref(sview(h), chain, h->h_ka[chain], h->h_kb[chain]);
    x.tb = tview(h, true);
    x.rs = sl.d_rs;
    x.eps = h->eps;
    x.na = h->na; x.n = h->n;
    x.badj = sc.badj; x.badj_cnt = sc.badj_cnt; x.stride = std::max(h->h_ka[chain], h->h_kb[chain]);
    x.cand = sc.cand; x.cand_dS = sc.cand_dS; x.n_cand = sc.n_cand; x.seen = sc.seen; x.first = sc.first; x.map = sc.map;
    return x;
}

// new block counts of one chain: host copy, device copy, counts rebuilt from the labels (init_bisbm)
int set_chain_k(bisbm_handle* h, uint32_t chain, uint32_t ka, uint32_t kb) {
    if (ka > h->KA || kb > h->KB) return fail(BISBM_ERR_STATE, "chain %u: (%u, %u) blocks exceed the pool's strides (%u, %u)", chain, ka, kb, h->KA, h->KB);
    // an alignment reference and its maps are for the (ka, kb) the pool had: a chain with other block counts drops it
    if (ka != h->h_ka[chain] || kb != h->h_kb[chain]) free_align(h);
    h->h_ka[chain] = ka; h->h_kb[chain] = kb;
    CU(cudaMemcpyAsync(h->d_ka + chain, &h->h_ka[chain], sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_kb + chain, &h->h_kb[chain], sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return rebuild_counts(h);
}

// apply_block_moves (src/blockmodel.cc:505-553): every impacted block becomes the smallest member of its accepted set,
// then the blocks are renumbered in order of first appearance over the nodes and the counts rebuilt (init_bisbm)
int apply_block_moves(bisbm_handle* h, uint32_t chain, const ReplaySlot& sl, MergeScratch& sc, const std::vector<uint32_t>& rep) {
    const uint32_t K = h->h_ka[chain] + h->h_kb[chain];
    CU(cudaMemcpyAsync(sc.map, rep.data(), K * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(sc.first, 0xff, K * sizeof(uint32_t), h->stream));
    MergeCtx x = mctx(h, chain, sl, sc);
    merge_first_kernel<<<(h->n + 255) / 256, 256, 0, h->stream>>>(x);
    CU(cudaGetLastError());
    std::vector<uint32_t> first(K);
    CU(cudaMemcpyAsync(first.data(), sc.first, K * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    std::vector<uint32_t> present;
    for (uint32_t b = 0; b < K; ++b) if (first[b] != 0xffffffffu) present.push_back(b);
    std::sort(present.begin(), present.end(), [&](uint32_t a, uint32_t b) { return first[a] < first[b]; });
    std::vector<uint32_t> newid(K, 0);
    uint32_t new_ka = 0;
    for (uint32_t i = 0; i < present.size(); ++i) { newid[present[i]] = i; if (first[present[i]] < h->na) new_ka = i + 1; }
    const uint32_t new_kb = (uint32_t)present.size() - new_ka;
    // the reference's sanity check (n != K_ -> "[sanity check] inconsistency!"): type-a blocks must come first
    for (uint32_t i = 0; i < new_ka; ++i) if (first[present[i]] >= h->na) return fail(BISBM_ERR_STATE, "agg_merge: blocks mix node types");
    if (new_ka == 0 || new_kb == 0) return fail(BISBM_ERR_STATE, "agg_merge: a node type lost all its blocks");
    std::vector<uint32_t> full(K);
    for (uint32_t b = 0; b < K; ++b) full[b] = newid[rep[b]];
    CU(cudaMemcpyAsync(sc.map, full.data(), K * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    merge_relabel_kernel<<<(h->n + 255) / 256, 256, 0, h->stream>>>(x, new_ka);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    wrote_labels32(h);
    return set_chain_k(h, chain, new_ka, new_kb);
}

// one pass of proposals + description-length changes: candidates in proposal order
int merge_candidates(bisbm_handle* h, uint32_t chain, const ReplaySlot& sl, MergeScratch& sc, uint32_t first_block, uint32_t n_blocks,
                     uint32_t nm, std::vector<uint32_t>& cand, std::vector<double>& dS) {
    const uint32_t K = h->h_ka[chain] + h->h_kb[chain];
    const uint64_t bits = (uint64_t)K * K;
    CU(cudaMemsetAsync(sc.seen, 0, (bits + 31) / 32 * sizeof(uint32_t), h->stream));
    MergeCtx x = mctx(h, chain, sl, sc);
    merge_badj_kernel<<<(K + 127) / 128, 128, 0, h->stream>>>(x);
    const size_t smem = 2 * MT_STATE_WORDS * sizeof(uint32_t) + (size_t)K * sizeof(double);
    if (smem > 200 * 1024) return fail(BISBM_ERR_ARG, "agg_merge: K = %u blocks do not fit the proposal kernel's shared memory", K);
    int rc = ensure_smem_attr(h, (const void*)merge_propose_kernel, 200 * 1024);
    if (rc) return rc;
    merge_propose_kernel<<<1, 32, smem, h->stream>>>(x, first_block, n_blocks, nm);
    CU(cudaGetLastError());
    uint32_t n_cand = 0;
    CU(cudaMemcpyAsync(&n_cand, sc.n_cand, sizeof n_cand, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    cand.assign(2 * (size_t)n_cand, 0); dS.assign(n_cand, 0.0);
    if (n_cand) {
        merge_dS_kernel<<<(n_cand + 127) / 128, 128, 0, h->stream>>>(x, n_cand);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(cand.data(), sc.cand, 2 * (size_t)n_cand * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(dS.data(), sc.cand_dS, (size_t)n_cand * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return BISBM_OK;
}

int alloc_merge_scratch(bisbm_handle* h, uint32_t chain, uint32_t nm, MergeScratch& sc) {
    const uint32_t K = h->h_ka[chain] + h->h_kb[chain];
    const uint32_t stride = std::max(h->h_ka[chain], h->h_kb[chain]);
    const size_t max_cand = (size_t)nm * K;
    CU(cudaMalloc(&sc.badj, (size_t)K * stride * sizeof(uint32_t)));
    CU(cudaMalloc(&sc.badj_cnt, K * sizeof(uint32_t)));
    CU(cudaMalloc(&sc.cand, 2 * max_cand * sizeof(uint32_t)));
    CU(cudaMalloc(&sc.cand_dS, max_cand * sizeof(double)));
    CU(cudaMalloc(&sc.n_cand, sizeof(uint32_t)));
    CU(cudaMalloc(&sc.seen, ((uint64_t)K * K + 31) / 32 * sizeof(uint32_t)));
    CU(cudaMalloc(&sc.first, K * sizeof(uint32_t)));
    CU(cudaMalloc(&sc.map, K * sizeof(uint32_t)));
    return BISBM_OK;
}

// the accepted merges of one selection pass: set_e (impacted blocks) and the partition of set_e into accepted sets,
// kept as "representative = smallest member" per block (src/blockmodel.cc:160-199: a move joins the set that holds its
// source or target, or opens a new one; a move inside set_e is skipped)
struct MergeSets {
    std::vector<int> set_of;                  // block -> set index, -1 outside set_e
    std::vector<std::vector<uint32_t>> sets;
    explicit MergeSets(uint32_t K) : set_of(K, -1) {}
    bool in(uint32_t b) const { return set_of[b] >= 0; }
    bool accept(uint32_t source, uint32_t target) {   // false: both already impacted (skipped by the reference)
        if (in(source) && in(target)) return false;
        if (!in(source) && !in(target)) { sets.push_back({source, target}); set_of[source] = set_of[target] = (int)sets.size() - 1; }
        else {
            const int si = in(source) ? set_of[source] : set_of[target];
            for (uint32_t b : {source, target}) if (!in(b)) { sets[si].push_back(b); set_of[b] = si; }
        }
        return true;
    }
    std::vector<uint32_t> representatives() const {
        std::vector<uint32_t> rep(set_of.size());
        for (uint32_t b = 0; b < rep.size(); ++b) rep[b] = in(b) ? *std::min_element(sets[set_of[b]].begin(), sets[set_of[b]].end()) : b;
        return rep;
    }
};

// agg_split (src/blockmodel.cc:555-611) + apply_split_moves (:433-459): nm random halvings of every block of one type with
// more than one node, the one with the smallest description-length change becomes a new block.  The shuffles consume
// `engine` exactly like std::shuffle over the reference's vector<bool>; see split_dS_kernel for what cannot be pinned.
int agg_split(bisbm_handle* h, uint32_t chain, const ReplaySlot& sl, MergeScratch& sc, bool type_b, uint32_t nm) {
    const uint32_t ka = h->h_ka[chain], kb = h->h_kb[chain], K = ka + kb, n = h->n;
    if ((!type_b && ka + 1 > h->KA) || (type_b && kb + 1 > h->KB))
        return fail(BISBM_ERR_STATE, "agg_split: the pool was created with room for (%u, %u) blocks only", h->KA, h->KB);
    std::vector<int32_t> lab(n);
    CU(cudaMemcpy2D(lab.data(), sizeof(int32_t), h->d_labels + chain, (size_t)h->C * sizeof(int32_t), sizeof(int32_t), n, cudaMemcpyDeviceToHost));
    ReplayState rs;
    CU(cudaMemcpy(&rs, sl.d_rs, sizeof rs, cudaMemcpyDeviceToHost));
    const uint32_t b0 = type_b ? ka : 0, nbk = type_b ? kb : ka;
    std::vector<std::vector<uint32_t>> nodes(nbk);
    for (uint32_t v = type_b ? h->na : 0; v < (type_b ? n : h->na); ++v) nodes[(uint32_t)lab[v]].push_back(v);
    std::vector<SplitCand> cands;
    std::vector<uint32_t> members;
    std::vector<uint8_t> flags;
    std::vector<uint32_t> member_off(nbk, 0);
    for (uint32_t b = 0; b < nbk; ++b) {
        const uint32_t nr = (uint32_t)nodes[b].size();
        if (nr <= 1) continue;
        member_off[b] = (uint32_t)members.size();
        members.insert(members.end(), nodes[b].begin(), nodes[b].end());
        std::vector<uint32_t> splitter(nr, 0);
        for (uint32_t i = nr / 2; i < nr; ++i) splitter[i] = 1;
        mt_shuffle(splitter.data(), nr, 1, rs.engine);
        for (uint32_t rep = 0; rep < nm; ++rep) {
            mt_shuffle(splitter.data(), nr, 1, rs.engine);
            SplitCand cd; cd.block = b0 + b; cd.first_member = member_off[b]; cd.n_members = nr; cd.first_flag = (uint32_t)flags.size();
            for (uint32_t i = 0; i < nr; ++i) flags.push_back((uint8_t)splitter[i]);
            cands.push_back(cd);
        }
    }
    if (cands.empty()) return fail(BISBM_ERR_STATE, "agg_split: no block of type %c has more than one node", type_b ? 'b' : 'a');
    SplitCand* d_c = nullptr; uint32_t* d_m = nullptr; uint8_t* d_f = nullptr; double* d_o = nullptr;
    CU(cudaMalloc(&d_c, cands.size() * sizeof(SplitCand)));
    CU(cudaMalloc(&d_m, members.size() * sizeof(uint32_t)));
    CU(cudaMalloc(&d_f, flags.size()));
    CU(cudaMalloc(&d_o, cands.size() * sizeof(double)));
    CU(cudaMemcpy(d_c, cands.data(), cands.size() * sizeof(SplitCand), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_m, members.data(), members.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_f, flags.data(), flags.size(), cudaMemcpyHostToDevice));
    MergeCtx x = mctx(h, chain, sl, sc);
    const uint32_t kopp = type_b ? ka : kb;
    split_dS_kernel<<<(unsigned)cands.size(), 128, kopp * sizeof(int), h->stream>>>(x, gview(h), d_c, d_m, d_f, d_o);
    cudaError_t e = cudaGetLastError();
    std::vector<double> dS(cands.size());
    if (e == cudaSuccess) e = cudaMemcpyAsync(dS.data(), d_o, dS.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d_c); cudaFree(d_m); cudaFree(d_f); cudaFree(d_o);
    CU(e);
    size_t best = cands.size();
    double ddS = INFINITY;
    for (size_t i = 0; i < cands.size(); ++i) if (dS[i] < ddS) { ddS = dS[i]; best = i; }
    if (best == cands.size()) return fail(BISBM_ERR_STATE, "agg_split: every candidate split has an infinite description-length change");
    const SplitCand& w = cands[best];
    const int32_t new_local = (int32_t)(type_b ? kb : ka);     // the new block takes the next id of its type
    for (uint32_t i = 0; i < w.n_members; ++i)
        if (flags[w.first_flag + i]) lab[members[w.first_member + i]] = new_local;
    CU(cudaMemcpy2D(h->d_labels + chain, (size_t)h->C * sizeof(int32_t), lab.data(), sizeof(int32_t), sizeof(int32_t), n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(sl.d_rs, &rs, sizeof rs, cudaMemcpyHostToDevice));
    wrote_labels32(h);
    (void)K;
    return set_chain_k(h, chain, type_b ? ka : ka + 1, type_b ? kb + 1 : kb);
}

}  // namespace

extern "C" {

int bisbm_replay_agg_merge(bisbm_handle* h, uint32_t chain, int diff_a, int diff_b, uint32_t nm) {
    ReplaySlot* sl;
    int rc = need_replay(h, chain, &sl);
    if (rc) return rc;
    if (nm == 0) return fail(BISBM_ERR_ARG, "nm must be >= 1");
    if (diff_a >= (int)h->h_ka[chain] || diff_b >= (int)h->h_kb[chain]) return fail(BISBM_ERR_ARG, "cannot merge away every block of a type");
    rc = ensure_lgamma_table(h);
    if (rc) return rc;
    for (int guard = 0; guard < 1 << 20; ++guard) {      // each round = one (possibly recursive) call of the reference's agg_merge
        {
            MergeScratch none;       // (agg_split only needs the chain's views)
            while (diff_a < 0) { rc = agg_split(h, chain, *sl, none, false, nm); if (rc) return rc; ++diff_a; }
            while (diff_b < 0) { rc = agg_split(h, chain, *sl, none, true, nm); if (rc) return rc; ++diff_b; }
        }
        if (diff_a + diff_b == 0) return BISBM_OK;       // (also when they cancel: the reference returns here too)
        const uint32_t ka = h->h_ka[chain], kb = h->h_kb[chain], K = ka + kb;
        MergeScratch sc;             // sized for the current K (the splits may have grown it)
        rc = alloc_merge_scratch(h, chain, nm, sc);
        if (rc) return rc;
        uint32_t first_block = 0, n_blocks = K;
        if (diff_a > 0 && diff_b == 0) n_blocks = ka;
        else if (diff_a == 0 && diff_b > 0) { first_block = ka; n_blocks = kb; }
        std::vector<uint32_t> cand;
        std::vector<double> dS;
        rc = merge_candidates(h, chain, *sl, sc, first_block, n_blocks, nm, cand, dS);
        if (rc) return rc;
        // priority_queue<pair<dS, index>, greater<>>: ascending dS, ties by proposal order
        std::vector<uint32_t> order(dS.size());
        std::iota(order.begin(), order.end(), 0u);
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return dS[a] < dS[b] || (dS[a] == dS[b] && a < b); });
        MergeSets ms(K);
        bool recursive = false;
        size_t accepted = 0;
        for (size_t q = 0; q < order.size() && diff_a + diff_b != 0; ++q) {
            const uint32_t i = order[q];
            if (dS[i] == INFINITY) { recursive = true; break; }
            const uint32_t source = cand[2 * i], target = cand[2 * i + 1];
            if (source < ka && diff_a != 0) { if (ms.accept(source, target)) { --diff_a; ++accepted; } }
            else if (source >= ka && diff_b != 0) { if (ms.accept(source, target)) { --diff_b; ++accepted; } }
        }
        rc = apply_block_moves(h, chain, *sl, sc, ms.representatives());
        if (rc) return rc;
        if (!recursive) return BISBM_OK;
        if (accepted == 0 && guard > 64)
            return fail(BISBM_ERR_STATE, "agg_merge: no finite merge candidate left for (%d, %d) more merges", diff_a, diff_b);
    }
    return fail(BISBM_ERR_STATE, "agg_merge did not terminate");
}

int bisbm_replay_agg_merge_total(bisbm_handle* h, uint32_t chain, int diff, uint32_t nm) {
    ReplaySlot* sl;
    int rc = need_replay(h, chain, &sl);
    if (rc) return rc;
    if (nm == 0) return fail(BISBM_ERR_ARG, "nm must be >= 1");
    if (diff == 0) return BISBM_OK;
    if (diff < 0) return fail(BISBM_ERR_ARG, "diff must be >= 0");
    rc = ensure_lgamma_table(h);
    if (rc) return rc;
    const uint32_t ka = h->h_ka[chain], kb = h->h_kb[chain], K = ka + kb;
    MergeScratch sc;
    rc = alloc_merge_scratch(h, chain, nm, sc);
    if (rc) return rc;
    for (int guard = 0; guard < 4096; ++guard) {
        std::vector<uint32_t> cand;
        std::vector<double> dS;
        rc = merge_candidates(h, chain, *sl, sc, 0, K, nm, cand, dS);
        if (rc) return rc;
        std::vector<uint32_t> order(dS.size());
        std::iota(order.begin(), order.end(), 0u);
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return dS[a] < dS[b] || (dS[a] == dS[b] && a < b); });
        MergeSets ms(K);
        int left = diff;
        bool minS = true;     // the reference starts with minS = true; an empty queue leaves it true (and loops forever)
        for (size_t q = 0; q < order.size() && left != 0; ++q) {
            const uint32_t i = order[q];
            if (ms.accept(cand[2 * i], cand[2 * i + 1])) --left;
            minS = dS[i] == INFINITY;     // the round is redone when the LAST popped candidate was infinite
        }
        if (!minS) return apply_block_moves(h, chain, *sl, sc, ms.representatives());
    }
    return fail(BISBM_ERR_STATE, "agg_merge: every round ended on an infinite candidate");
}

int bisbm_chain_k(bisbm_handle* h, uint32_t chain, uint32_t* ka, uint32_t* kb) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    if (ka) *ka = h->h_ka[chain];
    if (kb) *kb = h->h_kb[chain];
    return BISBM_OK;
}

}  // extern "C"

extern "C" {

// ---------------------------------------------------------------- parallel mode
int bisbm_anneal(bisbm_handle* h, int schedule, float p0, float p1, uint64_t duration, uint64_t steps_await,
                 const uint64_t* seeds, uint32_t max_inflight, double* accept_ratio, uint64_t* sweeps_done) {
    int rc = need_chains(h);
    if (rc) return rc;
    rc = validate_schedule(schedule, p0, p1, duration);
    if (rc) return rc;
    rc = upload_seeds(h, seeds);
    if (rc) return rc;
    rc = sync_labels8(h);
    if (rc) return rc;
    const uint64_t N = h->n;
    const uint64_t all_sweeps = duration / N;
    const uint32_t C = h->C;
    {
        std::vector<uint8_t> act(C, 0);
        std::fill(act.begin(), act.begin() + h->n_chains, 1);
        std::vector<double> inf(C, INFINITY);
        CU(cudaMemcpyAsync(h->d_active, act.data(), C, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(h->d_entmin, inf.data(), C * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemsetAsync(h->d_accepted, 0, C * sizeof(unsigned long long), h->stream));
        CU(cudaMemsetAsync(h->d_u, 0, C * sizeof(unsigned long long), h->stream));
        CU(cudaMemsetAsync(h->d_sweeps, 0, C * sizeof(unsigned long long), h->stream));
        uint32_t na_ = h->n_chains;
        CU(cudaMemcpyAsync(h->d_nactive, &na_, sizeof na_, cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    h->last_launches = 0; h->last_sweep_launches = 0; h->last_moves = 0; h->last_ms = 0.0;
    CU(cudaEventRecord(h->ev0, h->stream));
    uint64_t sweep = 0;
    uint32_t n_active = h->n_chains;
    // early stop can only trigger once enough cold steps exist; poll the device counter
    // every `poll` sweeps (each poll is a stream sync)
    const bool can_stop = steps_await < duration;
    for (; sweep < all_sweeps && n_active; ++sweep) {
        rc = launch_full_sweep(h, schedule, p0, p1, sweep, max_inflight);
        if (rc) return rc;
        const uint64_t cold = cold_steps(schedule, p0, p1, sweep * N, (sweep + 1) * N);
        bookkeep_kernel<<<(h->n_chains + 127) / 128, 128, 0, h->stream>>>(
            h->n_chains, h->d_active, h->d_dS, h->d_entmin, h->d_u, h->d_sweeps, sweep, cold, steps_await, h->d_nactive);
        h->last_launches += 1;
        if (can_stop && cold) {
            CU(cudaMemcpyAsync(&n_active, h->d_nactive, sizeof n_active, cudaMemcpyDeviceToHost, h->stream));
            CU(cudaStreamSynchronize(h->stream));
        }
    }
    CU(cudaEventRecord(h->ev1, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->last_ms = ms;
    std::vector<unsigned long long> acc(C), sw(C);
    std::vector<uint8_t> act(C);
    CU(cudaMemcpy(acc.data(), h->d_accepted, C * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(sw.data(), h->d_sweeps, C * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(act.data(), h->d_active, C, cudaMemcpyDeviceToHost));
    for (uint32_t c = 0; c < h->n_chains; ++c) {
        // reference: accepted / ((sweep+1)*N) on early stop, accepted / duration otherwise
        if (accept_ratio) {
            if (!act[c]) accept_ratio[c] = (double)acc[c] / (double)(sw[c] * N);
            else accept_ratio[c] = duration ? (double)acc[c] / (double)duration : 0.0;
        }
        if (sweeps_done) sweeps_done[c] = sw[c];
    }
    return BISBM_OK;
}

// one sample of every chain's current labels into the histogram, straight from the array the sweep kernel keeps
// current: the u8 shadow (sweep2 kernels) or the i32 labels.  rung (device, may be null): only the chains at rung 0.
// With an alignment reference set, every chain's permutations are computed first (align.cuh) and the histogram counts
// the permuted labels; all of it is queued on the stream, nothing waits for the device.
static int launch_marginal(bisbm_handle* h, const uint32_t* rung = nullptr) {
    const uint64_t mw = (uint64_t)h->n * (h->C / 32);
    const unsigned mgrid = (unsigned)((mw * 32 + 255) / 256);
    const uint32_t* map = nullptr;
    if (h->al_segments) {
        const uint32_t ka = h->al_ka, kb = h->al_kb;     // == hist_width (bisbm_marginals_align; K changes drop the reference)
        CU(cudaMemsetAsync(h->d_al_overlap, 0, (size_t)h->C * ((size_t)ka * ka + (size_t)kb * kb) * sizeof(uint32_t), h->stream));
        const dim3 ogrid(h->al_segments, h->C / 32);
        const size_t osmem = (size_t)std::max(ka, kb) * 32 * sizeof(uint32_t);
        const uint32_t *seg_begin = h->d_al_seg, *seg_ref = h->d_al_seg + h->al_segments + 1;
        if (h->lab32_stale)
            align_overlap_kernel<uint8_t><<<ogrid, 256, osmem, h->stream>>>(h->d_lab8, h->C, h->n_chains, ka, kb, h->d_al_order,
                                                                          seg_begin, seg_ref, h->d_al_overlap);
        else
            align_overlap_kernel<int32_t><<<ogrid, 256, osmem, h->stream>>>(h->d_labels, h->C, h->n_chains, ka, kb, h->d_al_order,
                                                                          seg_begin, seg_ref, h->d_al_overlap);
        align_assign_kernel<<<dim3(h->n_chains, 2), 32, align_assign_smem(std::max(ka, kb)), h->stream>>>(h->d_al_overlap, h->C, ka, kb,
                                                                                                     h->d_al_map);
        CU(cudaGetLastError());
        map = h->d_al_map;
        h->al_sampled = true;
    }
    if (h->lab32_stale)
        marginal_kernel<uint8_t><<<mgrid, 256, 0, h->stream>>>(gview(h), h->d_lab8, h->C, h->d_ka, h->n_chains, h->d_hist, h->hist_width, rung, map);
    else
        marginal_kernel<int32_t><<<mgrid, 256, 0, h->stream>>>(gview(h), h->d_labels, h->C, h->d_ka, h->n_chains, h->d_hist, h->hist_width, rung, map);
    CU(cudaGetLastError());
    return BISBM_OK;
}

// kernel launches of one marginal sample (the alignment adds the overlap and assignment kernels)
static uint64_t marginal_launches(const bisbm_handle* h) { return h->al_segments ? 3 : 1; }

int bisbm_marginal_sample(bisbm_handle* h) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!h->d_hist) { rc = bisbm_marginals_clear(h); if (rc) return rc; }
    return launch_marginal(h);
}

int bisbm_marginals_clear(bisbm_handle* h) {
    int rc = need_chains(h);
    if (rc) return rc;
    uint32_t width = 0;
    for (uint32_t c = 0; c < h->n_chains; ++c) width = std::max(width, h->h_ka[c] + h->h_kb[c]);
    if (!h->d_hist || h->hist_width != width) {
        dfree(h->d_hist);
        CU(cudaMalloc(&h->d_hist, (size_t)h->n * width * sizeof(uint32_t)));
        h->hist_width = width;
    }
    CU(cudaMemsetAsync(h->d_hist, 0, (size_t)h->n * width * sizeof(uint32_t), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

int bisbm_marginals_align(bisbm_handle* h, const uint32_t* ref) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!ref) { free_align(h); return BISBM_OK; }
    const uint32_t ka = h->h_ka[0], kb = h->h_kb[0], n = h->n, na = h->na, C = h->C;
    for (uint32_t c = 1; c < h->n_chains; ++c)
        if (h->h_ka[c] != ka || h->h_kb[c] != kb)
            return fail(BISBM_ERR_ARG, "alignment needs one (ka, kb) for the pool: chain %u has (%u, %u), chain 0 (%u, %u)", c,
                        h->h_ka[c], h->h_kb[c], ka, kb);
    for (uint32_t v = 0; v < n; ++v) {
        const uint32_t g = ref[v];
        if (v < na ? g >= ka : (g < ka || g >= ka + kb))
            return fail(BISBM_ERR_ARG, "reference label %u of node %u is not a type-%c block (ka=%u kb=%u)", g, v, v < na ? 'a' : 'b', ka, kb);
    }
    const size_t osmem = (size_t)std::max(ka, kb) * 32 * sizeof(uint32_t), asmem = align_assign_smem(std::max(ka, kb));
    int optin = 0;
    CU(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    if (std::max(osmem, asmem) > (size_t)optin)
        return fail(BISBM_ERR_ARG, "alignment of %u blocks per type needs %zu bytes of shared memory per block (device: %d)",
                    std::max(ka, kb), std::max(osmem, asmem), optin);
    // the histogram a sample adds to must be this pool's width (a pool of other K reusing the buffers keeps the old one)
    if (h->d_hist && h->hist_width != ka + kb)
        return fail(BISBM_ERR_STATE, "the histogram is %u blocks wide, the pool has %u: call bisbm_marginals_clear first", h->hist_width, ka + kb);
    // raised to the device's limit once per handle, so that any later reference fits too
    if (osmem > 48 * 1024) {
        rc = ensure_smem_attr(h, (const void*)align_overlap_kernel<uint8_t>, optin);
        if (!rc) rc = ensure_smem_attr(h, (const void*)align_overlap_kernel<int32_t>, optin);
        if (rc) return rc;
    }
    if (asmem > 48 * 1024 && (rc = ensure_smem_attr(h, (const void*)align_assign_kernel, optin))) return rc;
    // node ids sorted by reference block (counting sort), cut into segments of at most ALIGN_SEG nodes of one block
    std::vector<uint32_t> start(ka + kb + 1, 0), order(n);
    for (uint32_t v = 0; v < n; ++v) ++start[ref[v] + 1];
    for (uint32_t g = 0; g < ka + kb; ++g) start[g + 1] += start[g];
    {
        std::vector<uint32_t> pos(start.begin(), start.end() - 1);
        for (uint32_t v = 0; v < n; ++v) order[pos[ref[v]]++] = v;
    }
    std::vector<uint32_t> seg_begin, seg_ref;
    for (uint32_t g = 0; g < ka + kb; ++g)
        for (uint32_t b = start[g]; b < start[g + 1]; b += ALIGN_SEG) { seg_begin.push_back(b); seg_ref.push_back(g); }
    const uint32_t S = (uint32_t)seg_ref.size();
    seg_begin.push_back(n);
    seg_begin.insert(seg_begin.end(), seg_ref.begin(), seg_ref.end());    // device layout: begin[S + 1], then ref[S]
    free_align(h);
    CU(cudaMalloc(&h->d_al_order, (size_t)n * sizeof(uint32_t)));
    CU(cudaMalloc(&h->d_al_seg, seg_begin.size() * sizeof(uint32_t)));
    CU(cudaMalloc(&h->d_al_overlap, (size_t)C * ((size_t)ka * ka + (size_t)kb * kb) * sizeof(uint32_t)));
    CU(cudaMalloc(&h->d_al_map, (size_t)C * (ka + kb) * sizeof(uint32_t)));
    CU(cudaMemcpyAsync(h->d_al_order, order.data(), (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_al_seg, seg_begin.data(), seg_begin.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->al_ka = ka; h->al_kb = kb; h->al_segments = S;
    return BISBM_OK;
}

int bisbm_marginals_alignment(bisbm_handle* h, uint32_t* map) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!map) return fail(BISBM_ERR_ARG, "null argument");
    if (!h->al_sampled) return fail(BISBM_ERR_STATE, "no aligned marginal sample since the reference was set");
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(map, h->d_al_map, (size_t)h->n_chains * (h->al_ka + h->al_kb) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return BISBM_OK;
}

int bisbm_marginalize(bisbm_handle* h, uint64_t burn_in, uint64_t sweeps, uint64_t every, const uint64_t* seeds,
                      uint32_t max_inflight) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (every == 0) return fail(BISBM_ERR_ARG, "sampling interval must be >= 1");
    if (!h->d_hist) { rc = bisbm_marginals_clear(h); if (rc) return rc; }
    rc = upload_seeds(h, seeds);
    if (rc) return rc;
    rc = sync_labels8(h);
    if (rc) return rc;
    {
        std::vector<uint8_t> act(h->C, 0);
        std::fill(act.begin(), act.begin() + h->n_chains, 1);
        CU(cudaMemcpyAsync(h->d_active, act.data(), h->C, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemsetAsync(h->d_accepted, 0, h->C * sizeof(unsigned long long), h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    h->last_launches = 0; h->last_sweep_launches = 0; h->last_moves = 0; h->last_ms = 0.0;
    CU(cudaEventRecord(h->ev0, h->stream));
    h->last_marginal_launches = 0;
    for (uint64_t sw = 0; sw < burn_in + sweeps; ++sw) {
        rc = launch_full_sweep(h, BISBM_CONSTANT, 1.0f, 0.0f, sw, max_inflight);
        if (rc) return rc;
        if (sw >= burn_in && ((sw - burn_in + 1) % every) == 0) {
            rc = launch_marginal(h);
            if (rc) return rc;
            h->last_marginal_launches += 1;
            h->last_launches += marginal_launches(h);
        }
    }
    CU(cudaEventRecord(h->ev1, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->last_ms = ms;
    return BISBM_OK;
}

// ---------------------------------------------------------------- parallel tempering
static LadderView ladder_view(bisbm_handle* h) {
    LadderView L;
    L.R = h->tp_rungs; L.n_ladders = h->n_chains / h->tp_rungs;
    L.rung_beta = h->d_tp_rung_beta; L.rung_of = h->d_tp_rung_of; L.chain_at = h->d_tp_chain_at; L.beta = h->d_tp_beta;
    L.trip = h->d_tp_trip; L.acc_prev = h->d_tp_acc_prev; L.stats = h->d_tp_stats;
    return L;
}

static size_t ladder_stats_len(uint32_t R, uint32_t n_ladders) { return 2 * (size_t)(R - 1) + 2 * (size_t)R + n_ladders; }

int bisbm_tempering_set(bisbm_handle* h, uint32_t n_rungs, const double* temps, const uint32_t* rung_of_chain) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (n_rungs == 0) { free_ladder(h); return BISBM_OK; }
    if (!temps) return fail(BISBM_ERR_ARG, "null temperatures");
    const uint32_t n_chains = h->n_chains, R = n_rungs;
    if (n_chains % R) return fail(BISBM_ERR_ARG, "%u rungs do not divide %u chains", R, n_chains);
    for (uint32_t i = 0; i < R; ++i) {
        if (!(temps[i] > 0.0) || !std::isfinite(temps[i])) return fail(BISBM_ERR_ARG, "temperature %u (%g) must be finite and > 0", i, temps[i]);
        if (i && temps[i] < temps[i - 1]) return fail(BISBM_ERR_ARG, "temperatures must be non-decreasing (T%u = %g < T%u = %g)", i, temps[i], i - 1, temps[i - 1]);
    }
    const uint32_t n_ladders = n_chains / R, C = h->C;
    std::vector<uint32_t> rung(C, 0), at(n_chains);
    std::vector<double> rbeta(R), beta(C, 1.0);
    std::vector<uint8_t> trip(n_chains);
    for (uint32_t i = 0; i < R; ++i) rbeta[i] = 1.0 / temps[i];
    for (uint32_t l = 0; l < n_ladders; ++l) {
        std::vector<bool> seen(R, false);
        for (uint32_t i = 0; i < R; ++i) {
            const uint32_t c = l * R + i, r = rung_of_chain ? rung_of_chain[c] : i;
            if (r >= R || seen[r]) return fail(BISBM_ERR_ARG, "rung_of_chain of ladder %u is not a permutation of 0..%u", l, R - 1);
            seen[r] = true;
            rung[c] = r; at[l * R + r] = c; beta[c] = rbeta[r]; trip[c] = r == 0 ? 1 : 0;
        }
    }
    free_ladder(h);
    const size_t ns = ladder_stats_len(R, n_ladders);
    CU(cudaMalloc(&h->d_tp_rung_beta, R * sizeof(double)));
    CU(cudaMalloc(&h->d_tp_beta, C * sizeof(double)));
    CU(cudaMalloc(&h->d_tp_rung_of, C * sizeof(uint32_t)));
    CU(cudaMalloc(&h->d_tp_chain_at, n_chains * sizeof(uint32_t)));
    CU(cudaMalloc(&h->d_tp_trip, n_chains));
    CU(cudaMalloc(&h->d_tp_acc_prev, C * sizeof(unsigned long long)));
    CU(cudaMalloc(&h->d_tp_stats, ns * sizeof(unsigned long long)));
    CU(cudaMemcpyAsync(h->d_tp_rung_beta, rbeta.data(), R * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_tp_beta, beta.data(), C * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_tp_rung_of, rung.data(), C * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_tp_chain_at, at.data(), n_chains * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_tp_trip, trip.data(), n_chains, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(h->d_tp_stats, 0, ns * sizeof(unsigned long long), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->tp_rungs = R;
    h->tp_round = 0;
    return BISBM_OK;
}

int bisbm_tempering_run(bisbm_handle* h, uint64_t sweeps, uint64_t swap_every, uint64_t sample_every, const uint64_t* seeds,
                        uint64_t swap_seed, uint32_t max_inflight, double* accept_ratio) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!h->tp_rungs) return fail(BISBM_ERR_STATE, "no ladder: call bisbm_tempering_set first");
    if (swap_every == 0) return fail(BISBM_ERR_ARG, "swap interval must be >= 1");
    if (sample_every && !h->d_hist) { rc = bisbm_marginals_clear(h); if (rc) return rc; }
    rc = upload_seeds(h, seeds);
    if (rc) return rc;
    rc = sync_labels8(h);
    if (rc) return rc;
    const uint32_t C = h->C;
    const LadderView L = ladder_view(h);
    const unsigned lgrid = (L.n_ladders + 127) / 128;
    {
        std::vector<uint8_t> act(C, 0);
        std::fill(act.begin(), act.begin() + h->n_chains, 1);
        CU(cudaMemcpyAsync(h->d_active, act.data(), C, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemsetAsync(h->d_accepted, 0, C * sizeof(unsigned long long), h->stream));
        CU(cudaMemsetAsync(h->d_tp_acc_prev, 0, C * sizeof(unsigned long long), h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    h->last_launches = 0; h->last_sweep_launches = 0; h->last_moves = 0; h->last_ms = 0.0;
    h->last_marginal_launches = 0;
    CU(cudaEventRecord(h->ev0, h->stream));
    uint64_t unattributed = 0;       // sweeps whose moves the swap kernel has not yet credited to a rung
    for (uint64_t sw = 0; sw < sweeps; ++sw) {
        rc = launch_full_sweep(h, BISBM_CONSTANT, 1.0f, 0.0f, sw, max_inflight, h->d_tp_beta);
        if (rc) return rc;
        ++unattributed;
        if ((sw + 1) % swap_every == 0) {
            entropy_kernel<<<h->n_chains, 256, 0, h->stream>>>(gview(h), sview(h), tview(h, false), h->ent_base, h->n_chains,
                                                               h->d_ent_out, h->opt_vary_k, nullptr);
            tempering_swap_kernel<<<lgrid, 128, 0, h->stream>>>(L, h->d_ent_out, h->d_accepted, unattributed * h->n, 1, h->tp_round++, swap_seed);
            CU(cudaGetLastError());
            h->last_launches += 2;
            unattributed = 0;
        }
        if (sample_every && (sw + 1) % sample_every == 0) {
            rc = launch_marginal(h, h->d_tp_rung_of);
            if (rc) return rc;
            h->last_marginal_launches += 1;
            h->last_launches += marginal_launches(h);
        }
    }
    if (unattributed) {      // the sweeps after the last round: credited to the rungs the chains hold now
        tempering_swap_kernel<<<lgrid, 128, 0, h->stream>>>(L, h->d_ent_out, h->d_accepted, unattributed * h->n, 0, 0, 0);
        CU(cudaGetLastError());
        h->last_launches += 1;
    }
    CU(cudaEventRecord(h->ev1, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->last_ms = ms;
    if (accept_ratio) {
        std::vector<unsigned long long> acc(C);
        CU(cudaMemcpy(acc.data(), h->d_accepted, C * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        for (uint32_t c = 0; c < h->n_chains; ++c) accept_ratio[c] = sweeps ? (double)acc[c] / ((double)sweeps * (double)h->n) : 0.0;
    }
    return BISBM_OK;
}

int bisbm_tempering_stats(bisbm_handle* h, uint32_t* rung_of_chain, uint64_t* swaps_tried, uint64_t* swaps_accepted,
                          uint64_t* moves_tried, uint64_t* moves_accepted, uint64_t* round_trips) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!h->tp_rungs) return fail(BISBM_ERR_STATE, "no ladder: call bisbm_tempering_set first");
    const uint32_t R = h->tp_rungs, n_ladders = h->n_chains / R;
    std::vector<unsigned long long> st(ladder_stats_len(R, n_ladders));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(st.data(), h->d_tp_stats, st.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (rung_of_chain) CU(cudaMemcpy(rung_of_chain, h->d_tp_rung_of, h->n_chains * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    const unsigned long long* p = st.data();
    if (swaps_tried) std::copy(p, p + (R - 1), swaps_tried);
    p += R - 1;
    if (swaps_accepted) std::copy(p, p + (R - 1), swaps_accepted);
    p += R - 1;
    if (moves_tried) std::copy(p, p + R, moves_tried);
    p += R;
    if (moves_accepted) std::copy(p, p + R, moves_accepted);
    p += R;
    if (round_trips) std::copy(p, p + n_ladders, round_trips);
    return BISBM_OK;
}

int bisbm_sweep_info(bisbm_handle* h, int* kernel, uint32_t* warps_per_cta, uint32_t* ctas_per_group, uint32_t* slice) {
    if (!h) return fail(BISBM_ERR_ARG, "null handle");
    if (h->last_kernel < 0) return fail(BISBM_ERR_STATE, "no parallel sweep has run yet");
    if (kernel) *kernel = h->last_kernel;
    if (warps_per_cta) *warps_per_cta = h->last_wpc;
    if (ctas_per_group) *ctas_per_group = h->last_cpg;
    if (slice) *slice = h->last_slice;
    return BISBM_OK;
}

int bisbm_set_precision(bisbm_handle* h, int mode) {
    if (!h) return fail(BISBM_ERR_ARG, "null handle");
    if (mode != BISBM_PRECISION_FP32 && mode != BISBM_PRECISION_FP64) return fail(BISBM_ERR_ARG, "unknown precision mode %d", mode);
    h->precision = mode;
    return BISBM_OK;
}

int bisbm_share_graph(bisbm_handle* src, bisbm_handle** out) {
    if (!src || !out) return fail(BISBM_ERR_ARG, "null argument");
    *out = nullptr;
    if (!src->gdev) return fail(BISBM_ERR_STATE, "source handle has no graph");
    CU(cudaSetDevice(src->device));
    std::unique_ptr<bisbm_handle> h(new bisbm_handle());
    h->device = src->device; h->gdev = src->gdev; h->sm_count = src->sm_count;
    h->n = src->n; h->na = src->na; h->nb = src->nb; h->W = src->W; h->max_degree = src->max_degree; h->n_edges = src->n_edges;
    h->h_row_ptr = src->h_row_ptr; h->h_degvals = src->h_degvals; h->ent_base = src->ent_base;
    h->d_row_ptr = src->d_row_ptr; h->d_col = src->d_col; h->d_degidx = src->d_degidx; h->d_qtab = src->d_qtab; h->d_gl = src->d_gl; h->gl_n = src->gl_n;
    h->qn = src->qn; h->qk = src->qk;
    h->precision = src->precision; h->opt_inflight_div = src->opt_inflight_div; h->opt_logq_every = src->opt_logq_every;
    CU(cudaStreamCreate(&h->stream));
    CU(cudaEventCreate(&h->ev0));
    CU(cudaEventCreate(&h->ev1));
    *out = h.release();
    return BISBM_OK;
}

// chains started from equal-size blocks in node order (the reference's `-n` with equal sizes), labels written on the device
static int set_chains_equal_blocks(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb, double eps) {
    bool same_model = false;
    int rc = alloc_chains(h, n_chains, ka, kb, eps, &same_model);
    if (rc) return rc;
    const uint64_t tot = (uint64_t)h->n * h->C;
    equal_blocks_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(h->d_labels, h->n, h->na, h->nb, h->C, h->n_chains, h->d_ka, h->d_kb);
    CU(cudaGetLastError());
    wrote_labels32(h);
    rc = rebuild_counts(h);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

// the grid search's initial partitions in one pass: equal-size blocks in node order, then --randomize with the chain's seed,
// written straight into the u8 shadow; counts built once.  Same labels as set_chains_equal_blocks + bisbm_randomize.
static int set_chains_equal_blocks_randomized(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb, double eps,
                                              const uint64_t* seeds) {
    bool same_model = false;
    int rc = alloc_chains(h, n_chains, ka, kb, eps, &same_model);
    if (rc) return rc;
    if (h->KA > 256 || h->KB > 256) {        // labels that do not fit the shadow: the two-step form over the 4-byte array
        rc = set_chains_equal_blocks(h, n_chains, ka, kb, eps);
        return rc ? rc : bisbm_randomize(h, seeds);
    }
    rc = upload_seeds(h, seeds);
    if (rc) return rc;
    const uint64_t tot = (uint64_t)h->n * h->C;
    equal_blocks_random8_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(gview(h), h->d_lab8, h->C, h->n_chains, h->d_ka, h->d_kb,
                                                                                      h->d_seeds, feistel_half_bits(h->na), feistel_half_bits(h->nb));
    CU(cudaGetLastError());
    wrote_labels8(h);
    rc = rebuild_counts(h);
    if (rc) return rc;
    CU(cudaMemsetAsync(h->d_dS, 0, h->C * sizeof(double), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

// K class of a chain = the (KA, KB) strides of the pool it runs in.  max(Ka, Kb) <= 32: both types padded to the same
// power of two (>= 8), so chains of similar K share strides and keep the staged kernel.  Larger: each side is padded on
// its own ({8, 16, 24, 32, 48, 64, ...}) and the pool stays STAGED whenever the asymmetric m_rs fits shared memory at 16
// warps (64 x 16, 48 x 24: a det_k_bisbm grid is mostly such points) -- the smaller side is then grown as far as it still
// fits, so few pools result; only shapes that do not fit take the counts-in-L2 class (both sides padded to the power of two).
static bool k_fits_staged(uint32_t KA, uint32_t KB, uint32_t rs) {
    return KA <= 256 && KB <= 256 && sweep2_layout(KA, KB, 0, 16, rs).total <= kSmemMax && sweep2_layout(KA, KB, 1, 16, rs).total <= kSmemMax;
}
static uint32_t k_ladder(uint32_t k, bool next = false) {
    static const uint32_t steps[] = {8, 16, 24, 32, 48, 64, 96, 128, 192, 256};
    for (uint32_t s : steps) if (next ? s > k : s >= k) return s;
    return next ? 0u : k;
}
static uint64_t k_class(uint32_t ka, uint32_t kb, uint32_t rs) {
    uint32_t k = std::max(ka, kb), c = 8;
    while (c < k) c <<= 1;
    if (c > 32) {
        uint32_t pa = k_ladder(ka), pb = k_ladder(kb);
        if (k_fits_staged(pa, pb, rs)) {
            uint32_t& small = pa < pb ? pa : pb;
            for (uint32_t nx = k_ladder(small, true); nx && nx <= 32; nx = k_ladder(small, true)) {
                const uint32_t keep = small;
                small = nx;
                if (!k_fits_staged(pa, pb, rs)) { small = keep; break; }
            }
            return ((uint64_t)pa << 32) | pb;
        }
    }
    return ((uint64_t)c << 32) | c;
}

int bisbm_grid_search(bisbm_handle* g, uint32_t n_points, const uint32_t* ka, const uint32_t* kb, uint32_t restarts, double eps,
                      int schedule, float p0, float p1, uint64_t duration, uint64_t steps_await, uint64_t seed,
                      uint32_t max_inflight, double* entropy, double* accept, uint32_t* best_chain, uint32_t* best_labels,
                      double* stats) {
    if (!g || !ka || !kb || !entropy) return fail(BISBM_ERR_ARG, "null argument");
    if (n_points == 0 || restarts == 0) return fail(BISBM_ERR_ARG, "need at least one (Ka, Kb) point and one restart");
    const uint32_t n = g->n, na = g->na, nb = g->nb;
    for (uint32_t p = 0; p < n_points; ++p)
        if (ka[p] == 0 || kb[p] == 0 || ka[p] > na || kb[p] > nb)
            return fail(BISBM_ERR_ARG, "point %u: (Ka, Kb) = (%u, %u) needs 1 <= Ka <= na, 1 <= Kb <= nb", p, ka[p], kb[p]);
    std::map<uint64_t, std::vector<uint32_t>> buckets;      // K class -> points
    const uint32_t rs = g->precision == BISBM_PRECISION_FP32 ? 4u : 8u;
    for (uint32_t p = 0; p < n_points; ++p) buckets[k_class(ka[p], kb[p], rs)].push_back(p);
    double best = INFINITY;
    uint64_t total_moves = 0;
    double total_ms = 0.0;
    if (best_chain) *best_chain = 0;
    std::vector<uint32_t> cka, ckb;
    std::vector<uint64_t> seeds;
    std::vector<double> ent, acc;
    std::vector<uint64_t> sw;
    g->grid_report.clear();
    auto now_ms = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    for (auto& kv : buckets) {
        const double t_begin = now_ms();
        const std::vector<uint32_t>& pts = kv.second;
        const uint32_t nc = (uint32_t)pts.size() * restarts;
        // the bucket's pool: kept on the graph handle between calls (same shapes -> alloc_chains reuses every buffer)
        bisbm_handle* sub = nullptr;
        int rc = BISBM_OK;
        auto cached = g->grid_pools.find(kv.first);
        if (cached != g->grid_pools.end()) {
            sub = cached->second; sub->sweep_epoch = 0;
            sub->precision = g->precision; sub->opt_inflight_div = g->opt_inflight_div; sub->opt_logq_every = g->opt_logq_every;   // as bisbm_share_graph hands them on
        }
        else {
            rc = bisbm_share_graph(g, &sub);
            if (rc) return rc;
        }
        // initial labels: equal-size blocks in node order (the reference's `-n` with equal sizes,
        // src/mcmc_main.cc:302-326), then --randomize
        cka.resize(nc); ckb.resize(nc); seeds.resize(nc);
        for (uint32_t i = 0; i < nc; ++i) {
            const uint32_t p = pts[i / restarts], q = i % restarts;
            cka[i] = ka[p]; ckb[i] = kb[p];
            seeds[i] = seed * 0x9E3779B97F4A7C15ull + ((uint64_t)p << 20) + q + 1;
        }
        rc = set_chains_equal_blocks_randomized(sub, nc, cka.data(), ckb.data(), eps, seeds.data());
        ent.resize(nc); acc.resize(nc); sw.resize(nc);
        if (!rc && cudaStreamSynchronize(sub->stream) != cudaSuccess) rc = fail(BISBM_ERR_CUDA, "stream synchronize failed after the pool set-up");
        const double t_setup = now_ms();
        if (!rc) rc = bisbm_anneal(sub, schedule, p0, p1, duration, steps_await, seeds.data(), max_inflight, acc.data(), sw.data());
        const double t_anneal = now_ms();
        if (!rc) rc = bisbm_entropy_all(sub, ent.data());
        if (!rc) {
            total_ms += sub->last_ms;
            for (uint32_t i = 0; i < nc; ++i) total_moves += sw[i] * (uint64_t)n;
            uint32_t arg = 0;
            for (uint32_t i = 0; i < nc; ++i) {
                const uint32_t chain = pts[i / restarts] * restarts + i % restarts;
                entropy[chain] = ent[i];
                if (accept) accept[chain] = acc[i];
                if (ent[i] < ent[arg]) arg = i;
            }
            if (ent[arg] < best) {
                best = ent[arg];
                if (best_chain) *best_chain = pts[arg / restarts] * restarts + arg % restarts;
                if (best_labels) rc = bisbm_get_labels(sub, arg, best_labels);
            }
        }
        const std::string err = g_err;
        const double row[8] = {(double)sub->KA, (double)sub->KB, (double)nc, (double)sub->last_kernel, t_setup - t_begin, sub->last_ms,
                               t_anneal - t_setup, 0.0};
        // keep the pool for the next call unless memory is short (less than a quarter of the device left free) or the call failed
        size_t mem_free = 0, mem_total = 1;
        if (rc || cudaMemGetInfo(&mem_free, &mem_total) != cudaSuccess || mem_free < mem_total / 4) {
            g->grid_pools.erase(kv.first);
            bisbm_destroy(sub);
        } else g->grid_pools[kv.first] = sub;
        g->grid_report.insert(g->grid_report.end(), row, row + 8);
        g->grid_report.back() = now_ms() - t_anneal;
        if (rc) { g_err = err; return rc; }
    }
    if (stats) { stats[0] = (double)total_moves; stats[1] = total_ms; stats[2] = (double)buckets.size(); stats[3] = best; }
    return BISBM_OK;
}

int bisbm_grid_release(bisbm_handle* g) {
    if (!g) return fail(BISBM_ERR_ARG, "null handle");
    for (auto& kv : g->grid_pools) bisbm_destroy(kv.second);
    g->grid_pools.clear();
    return BISBM_OK;
}

int bisbm_grid_k_class(const bisbm_handle* g, uint32_t ka, uint32_t kb, uint32_t* KA, uint32_t* KB, int* staged) {
    if (!g || !KA || !KB) return fail(BISBM_ERR_ARG, "null argument");
    const uint32_t rs = g->precision == BISBM_PRECISION_FP32 ? 4u : 8u;
    const uint64_t c = k_class(ka, kb, rs);
    *KA = (uint32_t)(c >> 32); *KB = (uint32_t)c;
    if (staged) *staged = (g->max_degree <= 255u && k_fits_staged(*KA, *KB, rs)) ? 1 : 0;
    return BISBM_OK;
}

int bisbm_grid_search_report(const bisbm_handle* g, uint32_t max_rows, double* rows, uint32_t* n_rows) {
    if (!g || !n_rows || (max_rows && !rows)) return fail(BISBM_ERR_ARG, "null argument");
    const uint32_t have = (uint32_t)(g->grid_report.size() / 8);
    *n_rows = have;
    std::copy(g->grid_report.begin(), g->grid_report.begin() + 8 * (size_t)std::min(have, max_rows), rows);
    return BISBM_OK;
}

int bisbm_set_option(bisbm_handle* h, const char* name, int64_t value) {
    if (!h || !name) return fail(BISBM_ERR_ARG, "null argument");
    const std::string k(name);
    if (k == "kernel") {
        if (value != -1 && value != KERN_L2 && value != KERN_S2L_F64)
            return fail(BISBM_ERR_ARG, "kernel: -1 (automatic), 0 (round-1 kernel, counts in L2) or 5 (sweep2, counts in L2)");
        h->opt_kernel = (int)value;
    } else if (k == "inflight_div") {
        if (value < 1 || value > (1 << 30)) return fail(BISBM_ERR_ARG, "inflight_div must be >= 1");
        h->opt_inflight_div = (uint32_t)value;
    } else if (k == "vary_k") {
        h->opt_vary_k = value != 0;
    } else if (k == "warps") {
        if (value != 16 && value != 20 && value != 24) return fail(BISBM_ERR_ARG, "warps: 16, 20 or 24");
        h->opt_warps = (uint32_t)value;
    } else if (k == "generic") {
        h->opt_generic = value != 0;
    } else if (k == "logq_every") {
        if (value < 1 || value > 0x7fffffff) return fail(BISBM_ERR_ARG, "logq_every must be >= 1");
        h->opt_logq_every = (uint32_t)value;
    } else if (k == "spare_sms") {
        h->opt_spare_sms = value != 0;
    } else if (k == "reserve_ka" || k == "reserve_kb") {
        if (value < 0 || value > (1 << 20)) return fail(BISBM_ERR_ARG, "%s out of range", name);
        (k == "reserve_ka" ? h->opt_reserve_ka : h->opt_reserve_kb) = (uint32_t)value;
    } else {
        return fail(BISBM_ERR_ARG, "unknown option '%s'", name);
    }
    return BISBM_OK;
}

#ifdef BISBM_ROUND_CLOCKS
// instrumented builds only (scripts/round_clocks.py): copy the 11 counters of sweep2.cuh's g_round_clocks to `out`, then zero them
int bisbm_round_clocks(unsigned long long* out) {
    if (!out) return fail(BISBM_ERR_ARG, "null argument");
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(out, g_round_clocks, sizeof(unsigned long long) * 11));
    const unsigned long long zero[11] = {};
    CU(cudaMemcpyToSymbol(g_round_clocks, zero, sizeof zero));
    return BISBM_OK;
}
#endif

int bisbm_parallel_transition(bisbm_handle* h, uint32_t chain, uint32_t v, uint32_t s, double* dS, double* log_accu) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    const uint32_t ka = h->h_ka[chain], kb = h->h_kb[chain];
    if (v >= h->n || s >= ka + kb) return fail(BISBM_ERR_ARG, "vertex or block out of range");
    const bool va = v < h->na;
    if ((s < ka) != va) {   // cross-type proposal: +inf before accu_r_ is touched (src/metropolis_hasting.cc:121-123)
        if (dS) *dS = INFINITY;
        if (log_accu) *log_accu = NAN;
        return BISBM_OK;
    }
    uint32_t wpc = 32;
    const int kernel = plan_kernel(h, &wpc);
    if (!kern_is_s2(kernel))
        return fail(BISBM_ERR_STATE, "bisbm_parallel_transition needs the sweep2 kernel (degrees > 255 or K > 256 per type take the round-1 kernel)");
    const uint32_t type = va ? 0 : 1;
    rc = sync_labels8(h);
    if (rc) return rc;
    const uint32_t kmax = type ? h->KB : h->KA;
    const uint32_t tot = h->n_chains * kmax;
    logq_refresh_kernel<<<(tot * 16 + 127) / 128, 128, 0, h->stream>>>(sview(h), tview(h, false), h->d_lq, h->n_chains, type);
    CU(cudaMemsetAsync(h->d_kat_out, 0xff, 2 * sizeof(double), h->stream));   // NaN: "not written"
    LaunchPlan lp;
    memset(&lp, 0, sizeof lp);
    lp.kernel = kernel; lp.smem = kern_is_s2_staged(kernel); lp.hist_bytes = 1; lp.wpc = wpc; lp.warps_used = 1; lp.ctas_per_group = 1; lp.slice = 1;
    lp.smem_bytes = sweep2_layout(h->KA, h->KB, type, wpc, kern_is_f32(kernel) ? 4u : 8u, lp.smem).total;
    SweepParams P = base_params(h, type);
    P.n_groups = 1; P.group_offset = chain / 32;
    P.ctas_per_group = 1; P.warps_used = 1; P.pos_begin = 0; P.pos_end = 1; P.exclusive = 1;
    P.schedule = BISBM_CONSTANT; P.p0 = 1.0f; P.p1 = 0.0f; P.beta0 = 1.0;
    P.kat_mode = 1; P.kat_chain = chain; P.kat_v = v; P.kat_s = va ? s : s - ka;
    const bool stale = h->lab32_stale;
    rc = kern_is_f32(kernel) ? launch_sweep2<float>(h, P, lp, 1) : launch_sweep2<double>(h, P, lp, 1);
    h->lab32_stale = stale;   // nothing was written
    if (rc) return rc;
    double out[2];
    CU(cudaMemcpyAsync(out, h->d_kat_out, sizeof out, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    if (std::isnan(out[0]) && std::isnan(out[1])) { out[0] = 0.0; out[1] = 0.0; }   // s == r: dS = 0, accu_r = 1 (:109-112)
    if (dS) *dS = out[0];
    if (log_accu) *log_accu = out[1];
    return BISBM_OK;
}

// ---------------------------------------------------------------- the one collective of the path
int bisbm_nccl_get_unique_id(uint8_t* id128) {
    if (!id128) return fail(BISBM_ERR_ARG, "null argument");
    NcclApi* A = nccl_api();
    if (!A) return fail(BISBM_ERR_STATE, "libnccl.so.2 not found");
    ncclUniqueId id;
    NC(A->GetUniqueId(&id));
    memcpy(id128, id.internal, NCCL_UNIQUE_ID_BYTES);
    return BISBM_OK;
}

int bisbm_nccl_init(bisbm_handle* h, int nranks, int rank, const uint8_t* id128) {
    if (!h || !id128) return fail(BISBM_ERR_ARG, "null argument");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(BISBM_ERR_ARG, "bad rank %d of %d", rank, nranks);
    NcclApi* A = nccl_api();
    if (!A) return fail(BISBM_ERR_STATE, "libnccl.so.2 not found");
    CU(cudaSetDevice(h->device));
    if (h->comm) { A->CommDestroy(h->comm); h->comm = nullptr; }
    ncclUniqueId id;
    memcpy(id.internal, id128, NCCL_UNIQUE_ID_BYTES);
    NC(A->CommInitRank(&h->comm, nranks, id, rank));
    return BISBM_OK;
}

int bisbm_marginals_allreduce(bisbm_handle* h) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!h->d_hist) return fail(BISBM_ERR_STATE, "no marginal histogram yet");
    if (!h->comm) return fail(BISBM_ERR_STATE, "call bisbm_nccl_init first");
    NcclApi* A = nccl_api();
    NC(A->AllReduce(h->d_hist, h->d_hist, (size_t)h->n * h->hist_width, ncclUint32, ncclSum, h->comm, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

int bisbm_marginals_allreduce_local(bisbm_handle** hs, int n) {
    if (!hs || n < 1) return fail(BISBM_ERR_ARG, "bad argument");
    NcclApi* A = nccl_api();
    if (!A) return fail(BISBM_ERR_STATE, "libnccl.so.2 not found");
    std::vector<int> devs(n);
    for (int i = 0; i < n; ++i) {
        if (!hs[i] || !hs[i]->d_hist) return fail(BISBM_ERR_STATE, "handle %d has no marginal histogram", i);
        if (hs[i]->n != hs[0]->n || hs[i]->hist_width != hs[0]->hist_width) return fail(BISBM_ERR_ARG, "handle %d: histogram shape differs", i);
        devs[i] = hs[i]->device;
    }
    if (n == 1) return BISBM_OK;
    std::vector<ncclComm_t> comms(n);
    NC(A->CommInitAll(comms.data(), n, devs.data()));
    const size_t count = (size_t)hs[0]->n * hs[0]->hist_width;
    ncclResult_t r = A->GroupStart();
    for (int i = 0; i < n && r == ncclSuccess; ++i)
        r = A->AllReduce(hs[i]->d_hist, hs[i]->d_hist, count, ncclUint32, ncclSum, comms[i], hs[i]->stream);
    if (r == ncclSuccess) r = A->GroupEnd(); else A->GroupEnd();
    cudaError_t ce = cudaSuccess;
    for (int i = 0; i < n; ++i) {
        cudaSetDevice(hs[i]->device);
        cudaError_t e = cudaStreamSynchronize(hs[i]->stream);
        if (e != cudaSuccess) ce = e;
    }
    for (int i = 0; i < n; ++i) A->CommDestroy(comms[i]);
    if (r != ncclSuccess) return fail(BISBM_ERR_CUDA, "NCCL all-reduce failed: %s", A->GetErrorString(r));
    if (ce != cudaSuccess) return fail(BISBM_ERR_CUDA, "all-reduce: %s", cudaGetErrorString(ce));
    return BISBM_OK;
}

int bisbm_marginals_device(bisbm_handle* h, void** dev_ptr, uint64_t* n_elems, uint32_t* width) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!h->d_hist) return fail(BISBM_ERR_STATE, "no marginal histogram yet");
    if (dev_ptr) *dev_ptr = h->d_hist;
    if (n_elems) *n_elems = (uint64_t)h->n * h->hist_width;
    if (width) *width = h->hist_width;
    return BISBM_OK;
}

int bisbm_get_marginals(bisbm_handle* h, uint32_t* hist) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!h->d_hist) return fail(BISBM_ERR_STATE, "no marginal histogram yet");
    CU(cudaMemcpy(hist, h->d_hist, (size_t)h->n * h->hist_width * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return BISBM_OK;
}

int bisbm_marginal_argmax(bisbm_handle* h, uint32_t* labels) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!h->d_hist) return fail(BISBM_ERR_STATE, "no marginal histogram yet");
    uint32_t* d_out = nullptr;
    CU(cudaMalloc(&d_out, (size_t)h->n * sizeof(uint32_t)));
    marginal_argmax_kernel<<<(h->n + 255) / 256, 256, 0, h->stream>>>(h->n, h->d_hist, h->hist_width, d_out);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaMemcpy(labels, d_out, (size_t)h->n * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaFree(d_out);
    if (e != cudaSuccess) return fail(BISBM_ERR_CUDA, "marginal_argmax: %s", cudaGetErrorString(e));
    return BISBM_OK;
}

int bisbm_last_timing(bisbm_handle* h, double* sweep_ms, uint64_t* launches, uint64_t* moves) {
    if (!h) return fail(BISBM_ERR_ARG, "null handle");
    if (sweep_ms) *sweep_ms = h->last_ms;
    if (launches) *launches = h->last_launches;
    if (moves) *moves = h->last_moves;
    return BISBM_OK;
}

int bisbm_sweep_launches(bisbm_handle* h, uint64_t* sweep_kernel_launches) {
    if (!h || !sweep_kernel_launches) return fail(BISBM_ERR_ARG, "null argument");
    *sweep_kernel_launches = h->last_sweep_launches;
    return BISBM_OK;
}

int bisbm_stream(bisbm_handle* h, void** stream) {
    if (!h || !stream) return fail(BISBM_ERR_ARG, "null argument");
    *stream = (void*)h->stream;
    return BISBM_OK;
}

// ---------------------------------------------------------------- read-back
int bisbm_info(bisbm_handle* h, uint32_t* n, uint64_t* n_edges, uint32_t* max_degree, uint32_t* n_chains) {
    if (!h) return fail(BISBM_ERR_ARG, "null handle");
    if (n) *n = h->n;
    if (n_edges) *n_edges = h->n_edges;
    if (max_degree) *max_degree = h->max_degree;
    if (n_chains) *n_chains = h->n_chains;
    return BISBM_OK;
}

}  // extern "C"

template <typename OutT>
static int get_all_labels_impl(bisbm_handle* h, OutT* labels) {
    int rc = need_chains(h);
    if (rc) return rc;
    const uint32_t n = h->n, C = h->C;
    if (!h->d_labels_tmp) CU(cudaMalloc(&h->d_labels_tmp, (size_t)n * C * sizeof(int32_t)));
    OutT* stage = reinterpret_cast<OutT*>(h->d_labels_tmp);
    if constexpr (sizeof(OutT) == 1) {      // 8-bit labels: straight from the u8 shadow
        rc = sync_labels8(h);
        if (rc) return rc;
        dim3 grid((n + L8_NODES - 1) / L8_NODES, C / 32);
        export_labels8_kernel<<<grid, 256, 0, h->stream>>>(h->d_lab8, reinterpret_cast<uint8_t*>(stage), n, h->na, h->n_chains, C, h->d_ka);
    } else {
        rc = sync_labels32(h);
        if (rc) return rc;
        dim3 grid((n + 31) / 32, C / 32), block(32, 8);
        export_labels_kernel<OutT><<<grid, block, 0, h->stream>>>(h->d_labels, stage, n, h->na, h->n_chains, C, h->d_ka);
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(labels, stage, (size_t)h->n_chains * n * sizeof(OutT), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BISBM_OK;
}

extern "C" {

int bisbm_get_all_labels(bisbm_handle* h, uint32_t* labels) { return get_all_labels_impl<uint32_t>(h, labels); }

int bisbm_get_all_labels_u8(bisbm_handle* h, uint8_t* labels) {
    if (!h) return fail(BISBM_ERR_ARG, "null handle");
    for (uint32_t c = 0; c < h->n_chains; ++c)
        if (h->h_ka[c] + h->h_kb[c] > 256) return fail(BISBM_ERR_ARG, "chain %u: ka + kb > 256 does not fit 8-bit labels", c);
    return get_all_labels_impl<uint8_t>(h, labels);
}

int bisbm_get_labels(bisbm_handle* h, uint32_t chain, uint32_t* labels) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    const uint32_t n = h->n;
    // the chain's column is gathered on the device from whichever label array is current (no refresh of the other one),
    // then copied as n contiguous words
    if (!h->d_labels_tmp) CU(cudaMalloc(&h->d_labels_tmp, (size_t)n * h->C * sizeof(int32_t)));
    uint32_t* const d_col = reinterpret_cast<uint32_t*>(h->d_labels_tmp);
    if (h->lab32_stale) extract_chain_kernel<uint8_t><<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_lab8, h->C, chain, n, d_col);
    else extract_chain_kernel<int32_t><<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_labels, h->C, chain, n, d_col);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(labels, d_col, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    const uint32_t ka = h->h_ka[chain];
    for (uint32_t v = h->na; v < n; ++v) labels[v] += ka;
    return BISBM_OK;
}

// copy entries [first, first+count) of chain `chain` out of a group-interleaved count array
static int fetch_counts(bisbm_handle* h, const int32_t* d_src, size_t per_chain, uint32_t chain, std::vector<int32_t>& out) {
    out.resize(per_chain);
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy2D(out.data(), sizeof(int32_t), d_src + cnt_base(chain, per_chain), GROUP * sizeof(int32_t),
                    sizeof(int32_t), per_chain, cudaMemcpyDeviceToHost));
    return BISBM_OK;
}

int bisbm_get_m(bisbm_handle* h, uint32_t chain, int32_t* m) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    std::vector<int32_t> M;
    rc = fetch_counts(h, h->d_m, (size_t)h->KA * h->KB, chain, M);
    if (rc) return rc;
    const uint32_t ka = h->h_ka[chain], kb = h->h_kb[chain], K = ka + kb;
    std::fill(m, m + (size_t)K * K, 0);
    for (uint32_t a = 0; a < ka; ++a)
        for (uint32_t b = 0; b < kb; ++b) {
            const int32_t x = M[(size_t)a * h->KB + b];
            m[(size_t)a * K + ka + b] = x;
            m[(size_t)(ka + b) * K + a] = x;
        }
    return BISBM_OK;
}

static int get_slots(bisbm_handle* h, uint32_t chain, const int32_t* d_src, int32_t* out) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    std::vector<int32_t> tmp;
    rc = fetch_counts(h, d_src, (size_t)h->KA + h->KB, chain, tmp);
    if (rc) return rc;
    const uint32_t ka = h->h_ka[chain], kb = h->h_kb[chain];
    for (uint32_t a = 0; a < ka; ++a) out[a] = tmp[a];
    for (uint32_t b = 0; b < kb; ++b) out[ka + b] = tmp[h->KA + b];
    return BISBM_OK;
}

int bisbm_get_m_r(bisbm_handle* h, uint32_t chain, int32_t* e_r) { return get_slots(h, chain, h ? h->d_e : nullptr, e_r); }
int bisbm_get_n_r(bisbm_handle* h, uint32_t chain, int32_t* n_r) { return get_slots(h, chain, h ? h->d_nr : nullptr, n_r); }

int bisbm_get_eta(bisbm_handle* h, uint32_t chain, uint32_t* eta) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    std::vector<int32_t> tmp;
    rc = fetch_counts(h, h->d_eta, ((size_t)h->KA + h->KB) * h->W, chain, tmp);
    if (rc) return rc;
    const uint32_t ka = h->h_ka[chain], kb = h->h_kb[chain];
    const size_t Wf = (size_t)h->max_degree + 1;
    std::fill(eta, eta + (size_t)(ka + kb) * Wf, 0u);
    for (uint32_t q = 0; q < ka + kb; ++q) {
        const size_t slot = q < ka ? q : h->KA + (q - ka);
        for (uint32_t w = 0; w < h->W; ++w) eta[q * Wf + h->h_degvals[w]] = (uint32_t)tmp[slot * h->W + w];
    }
    return BISBM_OK;
}

int bisbm_entropy_all(bisbm_handle* h, double* entropy) {
    int rc = need_chains(h);
    if (rc) return rc;
    entropy_kernel<<<h->n_chains, 256, 0, h->stream>>>(gview(h), sview(h), tview(h, false), h->ent_base, h->n_chains,
                                                       h->d_ent_out, h->opt_vary_k, nullptr);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(entropy, h->d_ent_out, h->n_chains * sizeof(double), cudaMemcpyDeviceToHost));
    return BISBM_OK;
}

int bisbm_occupied_blocks(bisbm_handle* h, uint32_t* ka_kb) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (!ka_kb) return fail(BISBM_ERR_ARG, "null argument");
    uint32_t* d_k = nullptr;
    CU(cudaMalloc(&d_k, (size_t)h->n_chains * 2 * sizeof(uint32_t)));
    entropy_kernel<<<h->n_chains, 256, 0, h->stream>>>(gview(h), sview(h), tview(h, false), h->ent_base, h->n_chains, h->d_ent_out, 1, d_k);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaMemcpy(ka_kb, d_k, (size_t)h->n_chains * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaFree(d_k);
    if (e != cudaSuccess) return fail(BISBM_ERR_CUDA, "occupied_blocks: %s", cudaGetErrorString(e));
    return BISBM_OK;
}

int bisbm_entropy(bisbm_handle* h, uint32_t chain, double* entropy) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    std::vector<double> all(h->n_chains);
    rc = bisbm_entropy_all(h, all.data());
    if (rc) return rc;
    *entropy = all[chain];
    return BISBM_OK;
}

int bisbm_entropy_accum(bisbm_handle* h, uint32_t chain, double* entropy_accum) {
    int rc = need_chains(h);
    if (rc) return rc;
    if (chain >= h->n_chains) return fail(BISBM_ERR_ARG, "chain %u out of range", chain);
    auto it = h->replay.find(chain);
    CU(cudaStreamSynchronize(h->stream));
    if (it != h->replay.end()) {
        ReplayState hs;
        CU(cudaMemcpy(&hs, it->second.d_rs, sizeof hs, cudaMemcpyDeviceToHost));
        *entropy_accum = hs.entropy_accum;
    } else {
        CU(cudaMemcpy(entropy_accum, h->d_dS + chain, sizeof(double), cudaMemcpyDeviceToHost));
    }
    return BISBM_OK;
}

}  // extern "C"
