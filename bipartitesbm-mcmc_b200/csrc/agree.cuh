// agree.cuh -- partition agreement between the chains of a pool (bisbm_chain_agreement).
//
// For a pair of chains (x, y) and a node type t, n_ij = #nodes of type t in block i of x and block j of y.  Every metric
// of the pair (VI, NMI, adjusted Rand, matched overlap) is a closed form of a few exact statistics of that table, which
// the host composes in double:
//   agree_table_kernel   the contingency tables n_ij of a chunk of row chains against every column chain, per type
//   agree_final_kernel   per (row, column, type): S_xy = sum n log n, S_x, S_y over the row / column sums, the pair
//                        counts P_xy = sum C(n, 2), P_x, P_y, and M = the maximal sum_i n_{i, pi(i)} over bijections pi
// The tables are exact integers, so the result does not depend on scheduling; the finalise sums in a fixed order, so two
// calls are bit-identical.  A block permutation of either chain permutes rows or columns and changes none of it.
#pragma once
#include <cstdint>

#include "align.cuh"

namespace bisbm {

enum {
    AGREE_THREADS = 1024,   // threads of a table CTA
    AGREE_CHUNK = 64,       // row chains per chunk of tables (fewer when a quarter of the free memory holds fewer)
};

// exact sufficient statistics of one (row, column, type) table
struct AgreeStats {
    double s_xy, s_x, s_y;                       // sum n log n over the non-zero cells, row sums, column sums
    unsigned long long p_xy, p_x, p_y;           // sum C(n, 2) over the same
    unsigned long long m;                        // maximal matched overlap (0 when not asked for)
};

#ifdef __CUDACC__

// grid = (rows of the chunk, C / 32 column groups, passes * splits), AGREE_THREADS threads, dynamic shared memory =
// rpp * K * 32 * 4 bytes.  The CTA counts, for its row (chain row0 + blockIdx.x, or the reference) against the 32 chains
// of its column group, the nodes of one type whose row label falls in the pass's rows [r0, r0 + rpp): lane l keeps chain
// 32 g + l's counts in a shared [rpp][K][32] table (bank = lane, so the lanes of a warp never conflict).  Each warp walks
// every (AGREE_THREADS / 32)-th node of the split's node range: it reads the group's label row and the row chain's label
// (one value for the whole warp) and does one shared atomic per lane.  The non-zero bins are added to the chunk's global
// tab[row][group][K][K][32] with integer atomics.
// labels: the array the sweep keeps current (u8 shadow or i32 labels), already offset to the type's first node;
// krow: the row chains' block counts of the type; ref (may be null): the reference's type-local labels of the type's
// nodes, the row of every CTA.  Without a reference, groups below the row chain's own are skipped: their tables are the
// transposes of pairs counted already.  Padding lanes (c >= n_chains) read and add nothing.
template <typename LabT>
__global__ void __launch_bounds__(AGREE_THREADS, 1) agree_table_kernel(const LabT* __restrict__ labels, uint32_t C, uint32_t n_chains,
                                                                    uint32_t nt, uint32_t K, const uint32_t* __restrict__ krow,
                                                                    const uint32_t* __restrict__ ref, uint32_t row0, uint32_t rpp,
                                                                    uint32_t splits, uint32_t* __restrict__ tab) {
    extern __shared__ uint32_t s_tab[];
    const uint32_t rl = blockIdx.x, g = blockIdx.y, pass = blockIdx.z / splits, split = blockIdx.z % splits;
    const uint32_t c = row0 + rl;
    if (!ref && g < c / 32) return;
    const uint32_t r0 = pass * rpp;
    if (r0 >= (ref ? K : krow[c])) return;           // the row chain has no block in this pass
    const uint32_t rows = min(rpp, K - r0), cells = rows * K * 32;
    for (uint32_t i = threadIdx.x; i < cells; i += blockDim.x) s_tab[i] = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const uint32_t cp = g * 32 + lane;
    const bool live = cp < n_chains;
    const uint32_t per = (nt + splits - 1) / splits, begin = min(nt, split * per), end = min(nt, begin + per);
    uint32_t v = begin + warp;
    for (; v + 3 * nw < end; v += 4 * nw) {           // four independent node rows in flight per warp
        uint32_t r[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const size_t row = (size_t)(v + k * nw) * C;
            r[k] = ref ? ref[v + k * nw] : (uint32_t)labels[row + c];
            l[k] = live ? (uint32_t)labels[row + cp] : 0u;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (live && r[k] - r0 < rows) atomicAdd(&s_tab[((r[k] - r0) * K + l[k]) * 32 + lane], 1u);
    }
    for (; v < end; v += nw) {
        const size_t row = (size_t)v * C;
        const uint32_t r = ref ? ref[v] : (uint32_t)labels[row + c];
        if (live && r - r0 < rows) atomicAdd(&s_tab[((r - r0) * K + (uint32_t)labels[row + cp]) * 32 + lane], 1u);
    }
    __syncthreads();
    uint32_t* out = tab + (((size_t)rl * (C / 32) + g) * K + r0) * K * 32;
    for (uint32_t i = threadIdx.x; i < cells; i += blockDim.x) {
        const uint32_t x = s_tab[i];
        if (x) atomicAdd(&out[i], x);
    }
}

__device__ __forceinline__ double agree_warp_sum(double x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

__device__ __forceinline__ unsigned long long agree_warp_sum(unsigned long long x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

__device__ __forceinline__ double agree_nlogn(unsigned long long x) { return x ? (double)x * log((double)x) : 0.0; }

// grid = (n_chains columns, rows of the chunk, 2 types), one warp per CTA, dynamic shared memory =
// align_assign_smem(max(KA, KB)) with the overlap, else 0.  Reads the K x K table of (row row0 + blockIdx.y, column
// blockIdx.x, type) and writes its AgreeStats to stats[(row * n_chains + column) * 2 + type].  Lane-strided partials over
// rows (S_xy, P_xy, S_x, P_x) and over columns (S_y, P_y), then a fixed xor-shuffle tree: the order never depends on
// scheduling.  M: warp_min_assign (align.cuh) on w = n_ij (K + 1) + [i == j] -- the bonus (< K + 1) only breaks ties
// between assignments of equal overlap, so sum_j n_{pi(j), j} over the result is the maximal overlap.
// paired: rows are chains and only columns >= the row are computed (the host mirrors the rest).
__global__ void __launch_bounds__(32) agree_final_kernel(const uint32_t* __restrict__ tab_a, const uint32_t* __restrict__ tab_b,
                                                         uint32_t KA, uint32_t KB, uint32_t C, uint32_t n_chains, uint32_t row0,
                                                         int paired, int with_overlap, AgreeStats* __restrict__ stats) {
    extern __shared__ __align__(8) unsigned char s_as[];
    const uint32_t cp = blockIdx.x, rl = blockIdx.y, t = blockIdx.z, lane = threadIdx.x;
    const uint32_t row = row0 + rl;
    if (cp >= n_chains || (paired && cp < row)) return;
    const uint32_t K = t ? KB : KA;
    const uint32_t* T = (t ? tab_b : tab_a) + ((size_t)rl * (C / 32) + cp / 32) * K * K * 32 + cp % 32;
    auto at = [&](uint32_t i, uint32_t j) -> unsigned long long { return T[((size_t)i * K + j) * 32]; };
    double s_xy = 0.0, s_x = 0.0, s_y = 0.0;
    unsigned long long p_xy = 0, p_x = 0, p_y = 0, m = 0;
    for (uint32_t i = lane; i < K; i += 32) {
        unsigned long long a = 0;
        for (uint32_t j = 0; j < K; ++j) {
            const unsigned long long x = at(i, j);
            a += x;
            s_xy += agree_nlogn(x);
            p_xy += x * (x - (x > 0)) / 2;
        }
        s_x += agree_nlogn(a);
        p_x += a * (a - (a > 0)) / 2;
    }
    for (uint32_t j = lane; j < K; j += 32) {
        unsigned long long b = 0;
        for (uint32_t i = 0; i < K; ++i) b += at(i, j);
        s_y += agree_nlogn(b);
        p_y += b * (b - (b > 0)) / 2;
    }
    s_xy = agree_warp_sum(s_xy); s_x = agree_warp_sum(s_x); s_y = agree_warp_sum(s_y);
    p_xy = agree_warp_sum(p_xy); p_x = agree_warp_sum(p_x); p_y = agree_warp_sum(p_y);
    if (with_overlap) {
        const int64_t W1 = (int64_t)K + 1;
        auto cost = [&](uint32_t i, uint32_t j) -> int64_t { return -((int64_t)at(i - 1, j - 1) * W1 + (i == j ? 1 : 0)); };
        const int32_t* p = warp_min_assign(K, cost, s_as, lane);
        for (uint32_t j = 1 + lane; j <= K; j += 32) m += at((uint32_t)p[j] - 1, j - 1);
        m = agree_warp_sum(m);
    }
    if (lane == 0) {
        AgreeStats s;
        s.s_xy = s_xy; s.s_x = s_x; s.s_y = s_y;
        s.p_xy = p_xy; s.p_x = p_x; s.p_y = p_y; s.m = m;
        stats[((size_t)row * n_chains + cp) * 2 + t] = s;
    }
}

#endif  // __CUDACC__

}  // namespace bisbm
