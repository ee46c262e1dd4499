// sweep_aux.cuh -- the small kernels around the sweep: state construction (init_bisbm), label
// import / export / randomisation, per-sweep bookkeeping, marginal histograms, entropy().
// Count arrays are group-interleaved (see state.cuh): entry j of chain c is at
// [(c/32 * per_chain + j) * 32 + c%32].
#pragma once
#include "sweep.cuh"

namespace bisbm {

#ifdef __CUDACC__

// ---- state construction (init_bisbm: compute_n_r / compute_m / compute_m_r / compute_eta_rk,
//      reference src/blockmodel.cc:681-746).  lane = chain, one warp per vertex. ----
// LabT = int32_t (canonical labels) or uint8_t (the u8 shadow, when that is the array holding the current labels)
template <typename LabT>
__global__ void build_counts_kernel(GraphView G, StateView S, const LabT* __restrict__ labels, uint32_t n_chains) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t wpc = blockDim.x >> 5;
    const uint32_t n_groups = S.C / 32;
    const uint64_t gw = (uint64_t)blockIdx.x * wpc + (threadIdx.x >> 5);
    const uint32_t group = gw % n_groups;
    const uint64_t v64 = gw / n_groups;
    if (v64 >= G.n) return;
    const uint32_t v = (uint32_t)v64;
    const uint32_t c = group * 32 + lane;
    if (c >= n_chains) return;
    const uint32_t KA = S.KA, KB = S.KB, W = S.W, KK = KA + KB;
    const bool tb = v >= G.na;
    const uint32_t b = (uint32_t)labels[(size_t)v * S.C + c];
    const uint32_t slot = (tb ? KA : 0) + b;
    atomicAdd(&S.nr[((size_t)group * KK + slot) * GROUP + lane], 1);
    atomicAdd(&S.eta[(((size_t)group * KK + slot) * W + G.degidx[v]) * GROUP + lane], 1);
    if (!tb) {
        int32_t* M = S.m + (((size_t)group * KA + b) * KB) * GROUP + lane;
        for (uint32_t e = G.row_ptr[v]; e < G.row_ptr[v + 1]; ++e) {
            const uint32_t t = (uint32_t)labels[(size_t)G.col[e] * S.C + c];
            atomicAdd(&M[(size_t)t * GROUP], 1);
        }
    }
}

// The same with m_rs and n_r accumulated per CTA in shared memory (one chain group per CTA, [entry][lane] like the
// sweep kernels) and added to the global counts once at the end: 2E * C global atomics become shared-memory ones.
// Used when the group's m_rs fits; eta (K x W x 32 per group) still goes straight to global memory.
// grid = n_groups * ctas_per_group, dynamic shared memory = (KA*KB + KA+KB) * 128 bytes.
template <typename LabT>
__global__ void __launch_bounds__(1024, 1) build_counts_staged_kernel(GraphView G, StateView S, const LabT* __restrict__ labels,
                                                                      uint32_t n_chains, uint32_t ctas_per_group) {
    extern __shared__ __align__(16) int32_t sm_counts[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const uint32_t n_groups = S.C / 32;
    const uint32_t group = blockIdx.x % n_groups, cta = blockIdx.x / n_groups;
    const uint32_t KA = S.KA, KB = S.KB, W = S.W, KK = KA + KB;
    int32_t* const sM = sm_counts;
    int32_t* const sN = sM + KA * KB * 32;
    for (uint32_t i = threadIdx.x; i < (KA * KB + KK) * 32; i += blockDim.x) sm_counts[i] = 0;
    __syncthreads();
    const uint32_t c = group * 32 + lane;
    const bool live = c < n_chains;
    int32_t* const gETA = S.eta + (size_t)group * KK * W * GROUP + lane;
    for (uint32_t v = cta * wpc + warp; v < G.n; v += ctas_per_group * wpc) {
        if (!live) continue;
        const bool tb = v >= G.na;
        const uint32_t b = (uint32_t)labels[(size_t)v * S.C + c];
        const uint32_t slot = (tb ? KA : 0) + b;
        atomicAdd(&sN[slot * 32 + lane], 1);
        atomicAdd(&gETA[((size_t)slot * W + G.degidx[v]) * GROUP], 1);
        if (!tb) {
            int32_t* const row = sM + (b * KB) * 32 + lane;
            const uint32_t e1 = G.row_ptr[v + 1];
            for (uint32_t e = G.row_ptr[v]; e < e1; ++e)
                atomicAdd(&row[(uint32_t)labels[(size_t)G.col[e] * S.C + c] * 32], 1);
        }
    }
    __syncthreads();
    int32_t* const gM = S.m + (size_t)group * KA * KB * GROUP;
    int32_t* const gN = S.nr + (size_t)group * KK * GROUP;
    for (uint32_t i = threadIdx.x; i < KA * KB * 32; i += blockDim.x) if (sM[i]) atomicAdd(&gM[i], sM[i]);
    for (uint32_t i = threadIdx.x; i < KK * 32; i += blockDim.x) if (sN[i]) atomicAdd(&gN[i], sN[i]);
}

__global__ void build_e_kernel(StateView S, uint32_t n_chains) {  // compute_m_r
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t KA = S.KA, KB = S.KB;
    if (idx >= n_chains * (KA + KB)) return;
    const uint32_t slot = idx / n_chains, c = idx % n_chains;  // consecutive threads = consecutive chains
    const int32_t* M = S.m + cnt_base(c, (size_t)KA * KB);
    int64_t sum = 0;
    if (slot < KA) for (uint32_t b = 0; b < KB; ++b) sum += M[((size_t)slot * KB + b) * GROUP];
    else for (uint32_t a = 0; a < KA; ++a) sum += M[((size_t)a * KB + (slot - KA)) * GROUP];
    S.e[cnt_base(c, (size_t)KA + KB) + (size_t)slot * GROUP] = (int32_t)sum;
}

// equal-size blocks in node order: block of type-a node v = v * ka / na (likewise type b), chain-minor type-local labels
__global__ void equal_blocks_kernel(int32_t* __restrict__ out, uint32_t n, uint32_t na, uint32_t nb, uint32_t C, uint32_t n_chains,
                                    const uint32_t* __restrict__ ka, const uint32_t* __restrict__ kb) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint64_t)n * C) return;
    const uint32_t v = (uint32_t)(idx / C), c = (uint32_t)(idx % C);
    int32_t l = 0;
    if (c < n_chains) l = v < na ? (int32_t)((uint64_t)v * ka[c] / na) : (int32_t)((uint64_t)(v - na) * kb[c] / nb);
    out[idx] = l;
}

// parallel-mode --randomize: per chain, permute the labels of each type with a keyed
// Feistel permutation (keeps block sizes, like shuffle_bisbm)
__global__ void randomize_kernel(GraphView G, const int32_t* in, int32_t* out, uint32_t C, uint32_t n_chains,
                                 const uint64_t* seeds, uint32_t hb_a, uint32_t hb_b) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint64_t)G.n * C) return;
    const uint32_t v = (uint32_t)(idx / C), c = (uint32_t)(idx % C);
    if (c >= n_chains) { out[idx] = in[idx]; return; }
    const bool tb = v >= G.na;
    const uint32_t v0 = tb ? G.na : 0, nv = tb ? G.nb : G.na;
    const uint64_t key = seeds[c] * 0x9E3779B97F4A7C15ull + (tb ? 0x632BE59BD9B4E019ull : 0x2545F4914F6CDD1Dull);
    const uint32_t src = v0 + feistel_perm(v - v0, nv, tb ? hb_b : hb_a, key);
    out[idx] = in[(size_t)src * C + c];
}


// equal_blocks_kernel followed by randomize_kernel in one pass, straight into the u8 label shadow (the grid search's
// initial partitions: no 4-byte label array written, permuted and narrowed): out[v] = equal-block label of the node the
// keyed permutation maps v to -- the same labels, chain by chain, as the two kernels give
__global__ void equal_blocks_random8_kernel(GraphView G, uint8_t* __restrict__ out, uint32_t C, uint32_t n_chains,
                                            const uint32_t* __restrict__ ka, const uint32_t* __restrict__ kb,
                                            const uint64_t* __restrict__ seeds, uint32_t hb_a, uint32_t hb_b) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (uint64_t)G.n * C) return;
    const uint32_t v = (uint32_t)(idx / C), c = (uint32_t)(idx % C);
    if (c >= n_chains) { out[idx] = 0; return; }
    const bool tb = v >= G.na;
    const uint32_t nv = tb ? G.nb : G.na;
    const uint64_t key = seeds[c] * 0x9E3779B97F4A7C15ull + (tb ? 0x632BE59BD9B4E019ull : 0x2545F4914F6CDD1Dull);
    const uint32_t src = feistel_perm(v - (tb ? G.na : 0), nv, tb ? hb_b : hb_a, key);      // type-local index of the source node
    out[idx] = (uint8_t)((uint64_t)src * (tb ? kb[c] : ka[c]) / nv);
}

// one chain's column of a chain-minor label array -> contiguous u32 (bisbm_get_labels: one copy of n words instead of a
// strided copy of n rows)
template <typename LabT>
__global__ void extract_chain_kernel(const LabT* __restrict__ lab, uint32_t C, uint32_t chain, uint32_t n, uint32_t* __restrict__ out) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n) out[v] = (uint32_t)lab[(size_t)v * C + chain];
}

// ---- label import / export: host layout [chain][node] with GLOBAL block ids  <->  device
//      layout [node][C] chain-minor, type-local.  32x32 tiles through shared memory so both
//      sides are coalesced.  `bad` receives 1 + (chain * n + node) of the first invalid label. ----
// InT = uint32_t or uint8_t (host label element type).  `prev` (may be null): the labels the handle holds now; *changed is
// set when any imported label differs from them (the caller then skips the count rebuild).
template <typename InT>
__global__ void import_labels_kernel(const InT* __restrict__ in, int32_t* __restrict__ out, uint32_t n,
                                     uint32_t na, uint32_t n_chains, uint32_t C, const uint32_t* __restrict__ ka,
                                     const uint32_t* __restrict__ kb, unsigned long long* bad,
                                     const int32_t* __restrict__ prev, uint32_t* changed) {
    __shared__ uint32_t tile[32][33];
    const uint32_t v0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (uint32_t j = threadIdx.y; j < 32; j += blockDim.y) {
        const uint32_t c = c0 + j, v = v0 + threadIdx.x;
        tile[j][threadIdx.x] = (c < n_chains && v < n) ? (uint32_t)in[(size_t)c * n + v] : 0u;
    }
    __syncthreads();
    bool diff = false;
    for (uint32_t j = threadIdx.y; j < 32; j += blockDim.y) {
        const uint32_t v = v0 + j, c = c0 + threadIdx.x;
        if (v >= n) continue;
        int32_t l = 0;
        if (c < n_chains) {
            const uint32_t g = tile[threadIdx.x][j];
            const uint32_t kac = ka[c], kbc = kb[c];
            bool ok;
            if (v < na) { ok = g < kac; l = (int32_t)g; }
            else { ok = (g >= kac) && (g < kac + kbc); l = (int32_t)(g - kac); }
            if (!ok) { atomicMin(bad, 1ull + (unsigned long long)c * n + v); l = 0; }
        }
        if (prev && prev[(size_t)v * C + c] != l) diff = true;
        out[(size_t)v * C + c] = l;
    }
    if (changed && __any_sync(0xffffffffu, diff) && (threadIdx.x == 0)) atomicOr(changed, 1u);
}

template <typename OutT>
__global__ void export_labels_kernel(const int32_t* __restrict__ in, OutT* __restrict__ out, uint32_t n,
                                     uint32_t na, uint32_t n_chains, uint32_t C, const uint32_t* __restrict__ ka) {
    __shared__ uint32_t tile[32][33];
    const uint32_t v0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (uint32_t j = threadIdx.y; j < 32; j += blockDim.y) {
        const uint32_t v = v0 + j, c = c0 + threadIdx.x;
        uint32_t g = 0;
        if (v < n && c < n_chains) {
            const uint32_t l = (uint32_t)in[(size_t)v * C + c];
            g = v < na ? l : ka[c] + l;
        }
        tile[j][threadIdx.x] = g;
    }
    __syncthreads();
    for (uint32_t j = threadIdx.y; j < 32; j += blockDim.y) {
        const uint32_t c = c0 + j, v = v0 + threadIdx.x;
        if (c < n_chains && v < n) out[(size_t)c * n + v] = (OutT)tile[threadIdx.x][j];
    }
}

// ---- 8-bit label import / export straight to / from the u8 shadow (K per type <= 256): host layout u8 [chain][node] with
//      GLOBAL block ids  <->  u8 [node][C] chain-minor, type-local.  Tiles of 32 chains x 128 nodes through shared memory;
//      with n a multiple of 16 both sides move 16 bytes per thread.  grid = (ceil(n/128), C/32), 256 threads.
//      `prev` (may be null, may alias `out`): the labels held now; *changed is set when an imported label differs. ----
enum { L8_NODES = 128, L8_PITCH = 132 };
__global__ void __launch_bounds__(256) import_labels8_kernel(const uint8_t* __restrict__ in, uint8_t* out, uint32_t n, uint32_t na,
                                                             uint32_t n_chains, uint32_t C, const uint32_t* __restrict__ ka,
                                                             const uint32_t* __restrict__ kb, unsigned long long* bad,
                                                             const uint8_t* prev, uint32_t* changed) {
    __shared__ __align__(16) uint8_t tile[32][L8_PITCH];
    __shared__ uint32_t s_ka[32], s_kb[32];
    const uint32_t v0 = blockIdx.x * L8_NODES, c0 = blockIdx.y * 32, tid = threadIdx.x;
    if (tid < 32) { const uint32_t c = c0 + tid; s_ka[tid] = c < n_chains ? ka[c] : 1u; s_kb[tid] = c < n_chains ? kb[c] : 1u; }
    {   // rows of the host array: thread -> chain tid/8, 16 nodes at (tid%8)*16
        const uint32_t j = tid >> 3, q = (tid & 7u) * 16u, c = c0 + j;
        uint4 w = make_uint4(0, 0, 0, 0);
        if (c < n_chains) {
            const uint8_t* src = in + (size_t)c * n + v0 + q;
            if ((n & 15u) == 0u && v0 + q + 16u <= n) w = *reinterpret_cast<const uint4*>(src);
            else {
                uint8_t b[16];
                for (uint32_t k = 0; k < 16; ++k) b[k] = (v0 + q + k < n) ? src[k] : (uint8_t)0;
                memcpy(&w, b, 16);
            }
        }
        uint32_t* t = reinterpret_cast<uint32_t*>(&tile[j][q]);
        t[0] = w.x; t[1] = w.y; t[2] = w.z; t[3] = w.w;
    }
    __syncthreads();
    // device rows: thread -> node tid/2, 16 chains at (tid%2)*16
    const uint32_t i = tid >> 1, h = (tid & 1u) * 16u, v = v0 + i;
    bool diff = false;
    if (v < n) {
        uint8_t o[16];
#pragma unroll
        for (uint32_t k = 0; k < 16; ++k) {
            const uint32_t cl = h + k, c = c0 + cl, g = tile[cl][i];
            uint32_t l = 0;
            if (c < n_chains) {
                const uint32_t kac = s_ka[cl], kbc = s_kb[cl];
                bool ok;
                if (v < na) { ok = g < kac; l = g; }
                else { ok = (g >= kac) && (g < kac + kbc); l = g - kac; }
                if (!ok) { atomicMin(bad, 1ull + (unsigned long long)c * n + v); l = 0; }
            }
            o[k] = (uint8_t)l;
        }
        uint4 w; memcpy(&w, o, 16);
        uint4* dst = reinterpret_cast<uint4*>(out + (size_t)v * C + c0 + h);
        if (prev) {
            const uint4 p = *reinterpret_cast<const uint4*>(prev + (size_t)v * C + c0 + h);
            diff = (p.x != w.x) || (p.y != w.y) || (p.z != w.z) || (p.w != w.w);
        }
        *dst = w;
    }
    if (changed && __any_sync(0xffffffffu, diff) && ((tid & 31u) == 0)) atomicOr(changed, 1u);
}

__global__ void __launch_bounds__(256) export_labels8_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, uint32_t n,
                                                             uint32_t na, uint32_t n_chains, uint32_t C, const uint32_t* __restrict__ ka) {
    __shared__ __align__(16) uint8_t tile[32][L8_PITCH];
    __shared__ uint32_t s_ka[32];
    const uint32_t v0 = blockIdx.x * L8_NODES, c0 = blockIdx.y * 32, tid = threadIdx.x;
    if (tid < 32) { const uint32_t c = c0 + tid; s_ka[tid] = c < n_chains ? ka[c] : 0u; }
    __syncthreads();
    {
        const uint32_t i = tid >> 1, h = (tid & 1u) * 16u, v = v0 + i;
        uint8_t b[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        if (v < n) {
            const uint4 w = *reinterpret_cast<const uint4*>(in + (size_t)v * C + c0 + h);
            memcpy(b, &w, 16);
        }
#pragma unroll
        for (uint32_t k = 0; k < 16; ++k) tile[h + k][i] = (uint8_t)(b[k] + ((v >= na) ? s_ka[h + k] : 0u));
    }
    __syncthreads();
    const uint32_t j = tid >> 3, q = (tid & 7u) * 16u, c = c0 + j;
    if (c < n_chains && v0 + q < n) {
        const uint32_t* t = reinterpret_cast<const uint32_t*>(&tile[j][q]);
        uint8_t* dst = out + (size_t)c * n + v0 + q;
        if ((n & 15u) == 0u && v0 + q + 16u <= n) *reinterpret_cast<uint4*>(dst) = make_uint4(t[0], t[1], t[2], t[3]);
        else for (uint32_t k = 0; k < 16 && v0 + q + k < n; ++k) dst[k] = tile[j][q + k];
    }
}

// u8 shadow of the chain-minor labels for the shared-memory sweep (blocks per type <= 256)
__global__ void labels8_kernel(const int32_t* __restrict__ in, uint8_t* __restrict__ out, uint64_t total) {
    const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < total) {
        const int4 v = *reinterpret_cast<const int4*>(in + i);
        uchar4 o; o.x = (uint8_t)v.x; o.y = (uint8_t)v.y; o.z = (uint8_t)v.z; o.w = (uint8_t)v.w;
        *reinterpret_cast<uchar4*>(out + i) = o;
    } else {
        for (uint64_t j = i; j < total; ++j) out[j] = (uint8_t)in[j];
    }
}

// the reverse: canonical i32 labels from the u8 shadow (after calls that ran the fp32 sweep kernel)
__global__ void labels32_kernel(const uint8_t* __restrict__ in, int32_t* __restrict__ out, uint64_t total) {
    const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < total) {
        const uchar4 v = *reinterpret_cast<const uchar4*>(in + i);
        int4 o; o.x = v.x; o.y = v.y; o.z = v.z; o.w = v.w;
        *reinterpret_cast<int4*>(out + i) = o;
    } else {
        for (uint64_t j = i; j < total; ++j) out[j] = (int32_t)in[j];
    }
}

// per-sweep bookkeeping of anneal (src/metropolis_hasting.cc:86-98) at sweep granularity
__global__ void bookkeep_kernel(uint32_t n_chains, uint8_t* active, const double* dS_accum, double* ent_min,
                                unsigned long long* u, unsigned long long* sweeps_done, uint64_t sweep,
                                uint64_t cold_steps, uint64_t steps_await, uint32_t* n_active) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chains || !active[c]) return;
    const double ent = dS_accum[c];
    if (ent < ent_min[c]) { ent_min[c] = ent; u[c] = 0; }
    else u[c] += cold_steps;
    sweeps_done[c] = sweep + 1;
    if (u[c] >= steps_await) { active[c] = 0; atomicSub(n_active, 1u); }
}

// marginal accumulation: hist[v][g] += #chains with global label g at v.  One warp per (vertex, chain group): the 32
// chains' labels are ONE 128-byte line of the chain-minor i32 labels (or one 32-byte sector of the u8 shadow, LabT =
// uint8_t); lanes holding the same label elect one of them, which adds their count -- a handful of atomics per warp
// instead of 32.  rung (may be null = every chain): parallel tempering samples only the chains with rung[c] == 0.
// map (may be null): label alignment (align.cuh), chain c's block g is counted as map[c * width + g].
template <typename LabT>
__global__ void marginal_kernel(GraphView G, const LabT* __restrict__ labels, uint32_t C, const uint32_t* __restrict__ ka,
                                uint32_t n_chains, uint32_t* hist, uint32_t width, const uint32_t* __restrict__ rung,
                                const uint32_t* __restrict__ map) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_groups = C / 32;
    const uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= (uint64_t)G.n * n_groups) return;
    const uint32_t v = (uint32_t)(w / n_groups), c = (uint32_t)(w % n_groups) * 32 + lane;
    uint32_t g = 0xffffffffu;     // padding lanes and masked chains: a key of their own, never added
    if (c < n_chains && (!rung || rung[c] == 0)) {
        const uint32_t l = (uint32_t)labels[(size_t)v * C + c];
        g = v < G.na ? l : ka[c] + l;
        if (map) g = map[(size_t)c * width + g];
    }
    const uint32_t peers = __match_any_sync(0xffffffffu, g);
    if (g != 0xffffffffu && lane == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&hist[(size_t)v * width + g], (uint32_t)__popc(peers));
}

__global__ void marginal_argmax_kernel(uint32_t n, const uint32_t* hist, uint32_t width, uint32_t* out) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    uint32_t best = 0, bc = 0;
    for (uint32_t g = 0; g < width; ++g) {
        const uint32_t x = hist[(size_t)v * width + g];
        if (x > bc) { bc = x; best = g; }
    }
    out[v] = best;
}

// blockmodel_t::entropy (src/blockmodel.cc:753-787) for every chain: one CTA per chain,
// fixed-order block reduction.  `base` holds the label-independent terms
// -sum_v lgamma(d_v+1) + sum_{i>j, A_ij>1} lgamma(A_ij+1), computed once per graph.
// occupied != 0 (estimate mode): the K-dependent terms use the number of NON-EMPTY blocks per type, also written to
// k_out[2c], k_out[2c+1] when k_out is not null
__global__ void entropy_kernel(GraphView G, StateView S, Tables tb, double base, uint32_t n_chains, double* out, int occupied,
                               uint32_t* k_out) {
    const uint32_t c = blockIdx.x;
    if (c >= n_chains) return;
    const uint32_t KA = S.KA, KB = S.KB, W = S.W;
    uint32_t ka = S.ka[c], kb = S.kb[c];
    const int32_t* M = S.m + cnt_base(c, (size_t)KA * KB);           // entry j at [j * GROUP]
    const int32_t* E = S.e + cnt_base(c, (size_t)KA + KB);
    const int32_t* NR = S.nr + cnt_base(c, (size_t)KA + KB);
    const int32_t* ETA = S.eta + cnt_base(c, ((size_t)KA + KB) * W);
    double acc = 0.0;
    for (uint32_t i = threadIdx.x; i < ka * kb; i += blockDim.x) {
        const uint32_t a = i / kb, b = i % kb;
        acc -= lgamma((double)M[((size_t)a * KB + b) * GROUP] + 1.0);
    }
    for (uint32_t i = threadIdx.x; i < (ka + kb) * W; i += blockDim.x) {
        const uint32_t q = i / W, w = i % W;
        const uint32_t slot = q < ka ? q : KA + (q - ka);
        acc -= lgamma((double)ETA[((size_t)slot * W + w) * GROUP] + 1.0);
    }
    for (uint32_t q = threadIdx.x; q < ka + kb; q += blockDim.x) {
        const uint32_t slot = q < ka ? q : KA + (q - ka);
        acc += lgamma((double)E[(size_t)slot * GROUP] + 1.0);
        acc += log_q(tb, E[(size_t)slot * GROUP], NR[(size_t)slot * GROUP]);
    }
    __shared__ double red[256];
    red[threadIdx.x] = acc;
    __syncthreads();
    for (uint32_t s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (occupied) {
            uint32_t oa = 0, ob = 0;
            for (uint32_t q = 0; q < ka; ++q) oa += NR[(size_t)q * GROUP] > 0;
            for (uint32_t q = 0; q < kb; ++q) ob += NR[(size_t)(KA + q) * GROUP] > 0;
            ka = oa; kb = ob;
            if (k_out) { k_out[2 * c] = oa; k_out[2 * c + 1] = ob; }
        }
        double ent = base + red[0];
        const double Ed = (double)G.n_edges, na = (double)G.na, nb = (double)G.nb;
        const double kab = (double)ka * (double)kb;
        // lbinom_fast(N, k) = lgamma(N+1) - lgamma(k+1) - lgamma(N-k+1), 0 if N==0, k==0 or k>N
        {
            const double N = kab + Ed - 1.0, k = Ed;
            if (!(N == 0.0 || k == 0.0 || k > N)) ent += lgamma(N + 1.0) - lgamma(k + 1.0) - lgamma(N - k + 1.0);
        }
        {
            const double N = na - 1.0, k = (double)ka - 1.0;
            if (!(N == 0.0 || k == 0.0 || k > N)) ent += lgamma(N + 1.0) - lgamma(k + 1.0) - lgamma(N - k + 1.0);
        }
        {
            const double N = nb - 1.0, k = (double)kb - 1.0;
            if (!(N == 0.0 || k == 0.0 || k > N)) ent += lgamma(N + 1.0) - lgamma(k + 1.0) - lgamma(N - k + 1.0);
        }
        ent += (na * nb == 0.0) ? 0.0 : log(na * nb);
        ent += lgamma(na + 1.0);
        ent += lgamma(nb + 1.0);
        out[c] = ent;
    }
}

#endif  // __CUDACC__

}  // namespace bisbm
