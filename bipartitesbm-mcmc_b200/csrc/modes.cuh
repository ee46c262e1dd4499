// modes.cuh -- marginals resolved by mode (bisbm_marginal_modes_set): every sample goes to the histogram of the nearest of
// M reference partitions.
//
// Per sample, for each mode m the alignment kernels (align.cuh, unchanged) fill that mode's slice of the overlap tables and
// maps: pi_{c,m}, the permutation bisbm_marginals_align(refs[m]) would use.  Then:
//   modes_select_kernel          ov_{c,m} = nodes that agree after pi_{c,m}; m* = arg-max (lowest m among equals); the
//                                threshold; chain_mode[c] and counted[m*]
//   modes_marginal_kernel        hist_modes[m*][v][pi_{c,m*}(label)] += 1, warp-aggregated as marginal_kernel
// The histograms are contiguous rows of one width, so marginal_argmax_kernel takes them as M * n rows.
#pragma once
#include <cstdint>

namespace bisbm {

#ifdef __CUDACC__

// one warp per chain, 256 threads.  overlap: M slices of the group-interleaved tables of align_overlap_kernel, each
// C/32 * (ka^2 + kb^2) * 32; map: M slices of [C][ka + kb] (align_assign_kernel).  ov is exact: an integer sum over both
// types, compared with > so the lowest m wins among equals.  Every real chain gets nearest[c] = m* (the map it is reported
// with); chain_mode[c] = m* if counted, M if its overlap is below min_ov (counted[M] += 1), 0xffffffff if rung[c] != 0.
// Padding lanes write nothing.
__global__ void __launch_bounds__(256) modes_select_kernel(const uint32_t* __restrict__ overlap, const uint32_t* __restrict__ map,
                                                           uint32_t C, uint32_t n_chains, uint32_t ka, uint32_t kb, uint32_t M,
                                                           uint64_t min_ov, const uint32_t* __restrict__ rung,
                                                           uint32_t* __restrict__ nearest, uint32_t* __restrict__ chain_mode,
                                                           unsigned long long* __restrict__ counted) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (c >= n_chains) return;
    const uint32_t width = ka + kb;
    const size_t tab = (size_t)ka * ka + (size_t)kb * kb;
    uint64_t best = 0;
    uint32_t bm = 0;
    for (uint32_t m = 0; m < M; ++m) {
        const uint32_t* O = overlap + ((size_t)m * (C / 32) + c / 32) * tab * 32 + (c % 32);
        const uint32_t* pi = map + ((size_t)m * C + c) * width;
        uint64_t ov = 0;
        for (uint32_t g = lane; g < width; g += 32) {
            const uint32_t t = pi[g];
            ov += g < ka ? O[((size_t)g * ka + t) * 32] : O[(tab - (size_t)kb * kb + (size_t)(g - ka) * kb + (t - ka)) * 32];
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) ov += __shfl_xor_sync(0xffffffffu, ov, off);
        if (m == 0 || ov > best) { best = ov; bm = m; }
    }
    if (lane == 0) {
        nearest[c] = bm;
        uint32_t cm = 0xffffffffu;
        if (!rung || rung[c] == 0) {
            cm = best < min_ov ? M : bm;
            atomicAdd(&counted[cm], 1ull);
        }
        chain_mode[c] = cm;
    }
}

// hist_modes[(m n + v) width + g] += #chains counted in mode m with block g (after pi_{c,m}) at v.  One warp per (vertex,
// chain group), lane = chain, the shape of marginal_kernel: the key m width + g, or 0xffffffff for a chain that is counted in
// no histogram (padding lanes, chain_mode >= M); lanes with the same key elect one atomic.  Every chain has (ka, kb).
template <typename LabT>
__global__ void modes_marginal_kernel(const LabT* __restrict__ labels, uint32_t n, uint32_t na, uint32_t C, uint32_t n_chains,
                                      uint32_t ka, uint32_t width, uint32_t M, const uint32_t* __restrict__ chain_mode,
                                      const uint32_t* __restrict__ map, uint32_t* hist) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_groups = C / 32;
    const uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= (uint64_t)n * n_groups) return;
    const uint32_t v = (uint32_t)(w / n_groups), c = (uint32_t)(w % n_groups) * 32 + lane;
    uint32_t key = 0xffffffffu;
    if (c < n_chains) {
        const uint32_t m = chain_mode[c];
        if (m < M) {
            const uint32_t l = (uint32_t)labels[(size_t)v * C + c];
            key = m * width + map[((size_t)m * C + c) * width + (v < na ? l : ka + l)];
        }
    }
    const uint32_t peers = __match_any_sync(0xffffffffu, key);
    if (key != 0xffffffffu && lane == (uint32_t)(__ffs(peers) - 1)) {
        const uint32_t m = key / width, g = key - m * width;
        atomicAdd(&hist[((size_t)m * n + v) * width + g], (uint32_t)__popc(peers));
    }
}

#endif  // __CUDACC__

}  // namespace bisbm
