// align.cuh -- maximum-overlap label alignment of the marginal samples (bisbm_marginals_align).
//
// Before a sample is counted, each chain's blocks are permuted, within each type, so that as many nodes as possible
// agree with a reference partition.  Two kernels per aligned sample, then marginal_kernel with the map:
//   align_overlap_kernel   O_c[r][r'] = #nodes in chain c's block r and the reference's block r', per type
//   align_assign_kernel    the permutation maximising sum_r w(r, pi(r)), w = O (K+1) + [r == r'], per (chain, type)
// The node order is sorted by reference block once, on the host (bisbm_marginals_align), and cut into segments that
// never cross a reference block: a CTA fills a single column r' of its chain group's tables.
#pragma once
#include <cstdint>

namespace bisbm {

enum { ALIGN_SEG = 2048 };   // nodes per segment of the reference-sorted order (one CTA each per chain group)

#ifdef __CUDACC__

// grid = (segments, C/32), 256 threads, dynamic shared memory = K_type * 32 * 4 bytes.  One warp walks every eighth node
// of the segment with lane = chain and counts the chain's label in a shared [K_type][32] table (bank = lane, so the
// lanes of a warp never conflict; warps of the CTA meet only in the atomics).  The non-zero bins go to the group-
// interleaved overlap[group][ka^2 + kb^2][32]: type a at r * ka + r', type b at ka^2 + r * kb + r'.
// LabT: the array the sweep keeps current (u8 shadow or i32 labels, as launch_marginal reads).  Padding lanes
// (c >= n_chains) read nothing and add nothing.
template <typename LabT>
__global__ void __launch_bounds__(256) align_overlap_kernel(const LabT* __restrict__ labels, uint32_t C, uint32_t n_chains,
                                                            uint32_t ka, uint32_t kb, const uint32_t* __restrict__ order,
                                                            const uint32_t* __restrict__ seg_begin,
                                                            const uint32_t* __restrict__ seg_ref, uint32_t* __restrict__ overlap) {
    extern __shared__ uint32_t s_ov[];
    const uint32_t seg = blockIdx.x, group = blockIdx.y;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const uint32_t gref = seg_ref[seg];
    const bool tb = gref >= ka;
    const uint32_t K = tb ? kb : ka, rp = tb ? gref - ka : gref;
    for (uint32_t i = threadIdx.x; i < K * 32; i += blockDim.x) s_ov[i] = 0;
    __syncthreads();
    const uint32_t c = group * 32 + lane;
    if (c < n_chains) {
        const uint32_t end = seg_begin[seg + 1];
        uint32_t i = seg_begin[seg] + warp;
        for (; i + 3 * wpc < end; i += 4 * wpc) {     // four independent loads in flight per lane
            uint32_t l[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) l[k] = (uint32_t)labels[(size_t)order[i + k * wpc] * C + c];
#pragma unroll
            for (int k = 0; k < 4; ++k) atomicAdd(&s_ov[l[k] * 32 + lane], 1u);
        }
        for (; i < end; i += wpc) atomicAdd(&s_ov[(uint32_t)labels[(size_t)order[i] * C + c] * 32 + lane], 1u);
    }
    __syncthreads();
    uint32_t* out = overlap + ((size_t)group * ((size_t)ka * ka + (size_t)kb * kb) + (tb ? (size_t)ka * ka : 0) + rp) * 32;
    for (uint32_t i = threadIdx.x; i < K * 32; i += blockDim.x) {
        const uint32_t x = s_ov[i];
        if (x) atomicAdd(&out[(size_t)(i >> 5) * K * 32 + (i & 31)], x);
    }
}

// shared memory of one align_assign_kernel warp for K blocks: u, v, minv (int64), p, way (int32), used (u8), each K + 1
__host__ __device__ inline size_t align_assign_smem(uint32_t K) { return (size_t)(K + 1) * (3 * 8 + 2 * 4 + 1); }

// grid = (n_chains, 2 types), one warp per CTA, dynamic shared memory = align_assign_smem(max(ka, kb)).
// Maximises sum_r w(r, pi(r)) with w(r, r') = O[r][r'] (K+1) + [r == r']: the overlap decides and the fixed-point bonus
// (at most K < K+1) only breaks ties, so among the permutations of maximal overlap the one with the most fixed points
// wins -- a chain equal to the reference keeps its labels, and empty blocks (zero rows and columns) stay in place.
// Shortest augmenting paths with potentials (Hungarian / Jonker-Volgenant, minimising -w) in exact int64 arithmetic:
// rows i = chain blocks, columns j = reference blocks, both 1-based (0 is the virtual start column).  The column loops
// are lane-parallel; the argmin takes the lowest column among equals, so the result is deterministic.
// map[c * (ka + kb) + g] = the global id chain c's block g is counted as.
__global__ void __launch_bounds__(32) align_assign_kernel(const uint32_t* __restrict__ overlap, uint32_t C, uint32_t ka, uint32_t kb,
                                                          uint32_t* __restrict__ map) {
    extern __shared__ __align__(8) unsigned char s_hu[];
    const uint32_t c = blockIdx.x, tb = blockIdx.y, lane = threadIdx.x;
    const uint32_t K = tb ? kb : ka;
    int64_t* const u = reinterpret_cast<int64_t*>(s_hu);
    int64_t* const v = u + (K + 1);
    int64_t* const minv = v + (K + 1);
    int32_t* const p = reinterpret_cast<int32_t*>(minv + (K + 1));
    int32_t* const way = p + (K + 1);
    uint8_t* const used = reinterpret_cast<uint8_t*>(way + (K + 1));
    const uint32_t* O = overlap + ((size_t)(c / 32) * ((size_t)ka * ka + (size_t)kb * kb) + (tb ? (size_t)ka * ka : 0)) * 32 + (c % 32);
    const int64_t W1 = (int64_t)K + 1;
    auto cost = [&](uint32_t i, uint32_t j) -> int64_t {       // -w of chain block i-1 against reference block j-1
        return -((int64_t)O[((size_t)(i - 1) * K + (j - 1)) * 32] * W1 + (i == j ? 1 : 0));
    };
    const int64_t INF = INT64_MAX / 4;
    for (uint32_t j = lane; j <= K; j += 32) { u[j] = 0; v[j] = 0; p[j] = 0; way[j] = 0; }
    __syncwarp();
    for (uint32_t i = 1; i <= K; ++i) {
        for (uint32_t j = lane; j <= K; j += 32) { minv[j] = INF; used[j] = 0; }
        if (lane == 0) p[0] = (int32_t)i;
        __syncwarp();
        uint32_t j0 = 0;
        do {
            if (lane == 0) used[j0] = 1;
            __syncwarp();
            const uint32_t i0 = (uint32_t)p[j0];
            const int64_t ui0 = u[i0];
            int64_t best = INF;
            uint32_t bj = 0xffffffffu;
            for (uint32_t j = 1 + lane; j <= K; j += 32) {
                if (used[j]) continue;
                const int64_t cur = cost(i0, j) - ui0 - v[j];
                if (cur < minv[j]) { minv[j] = cur; way[j] = (int32_t)j0; }
                if (minv[j] < best) { best = minv[j]; bj = j; }        // a lane's columns ascend: the first minimum is kept
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const int64_t ob = __shfl_xor_sync(0xffffffffu, best, off);
                const uint32_t oj = __shfl_xor_sync(0xffffffffu, bj, off);
                if (ob < best || (ob == best && oj < bj)) { best = ob; bj = oj; }
            }
            __syncwarp();
            for (uint32_t j = lane; j <= K; j += 32) {
                if (used[j]) { u[p[j]] += best; v[j] -= best; }        // the rows p[j] of used columns are distinct
                else minv[j] -= best;
            }
            __syncwarp();
            j0 = bj;
        } while (p[j0] != 0);
        if (lane == 0) {
            do { const uint32_t j1 = (uint32_t)way[j0]; p[j0] = p[j1]; j0 = j1; } while (j0);
        }
        __syncwarp();
    }
    const uint32_t base = tb ? ka : 0;
    uint32_t* const m = map + (size_t)c * (ka + kb) + base;
    for (uint32_t j = 1 + lane; j <= K; j += 32) m[p[j] - 1] = base + j - 1;
}

#endif  // __CUDACC__

}  // namespace bisbm
