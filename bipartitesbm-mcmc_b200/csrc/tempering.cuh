// tempering.cuh -- parallel tempering (replica exchange) over the chains of a pool.  Ladder l is chains l R .. l R + R - 1;
// a swap exchanges the RUNGS (temperatures) of two chains of one ladder, never their labels or counts, so a swap round
// costs O(R) per ladder on top of the entropy() of every chain.
#pragma once
#include "sweep.cuh"

namespace bisbm {

#ifdef __CUDACC__

struct LadderView {
    uint32_t R, n_ladders;
    const double* rung_beta;       // [R] 1 / T_i of rung i
    uint32_t* rung_of;             // [C] rung each chain holds
    uint32_t* chain_at;            // [n_ladders * R] chain holding rung i of ladder l, at l R + i
    double* beta;                  // [C] 1 / T of each chain's rung: what the sweep kernels read (SweepParams::beta_chain)
    uint8_t* trip;                 // [n_chains] end of its ladder the chain touched last: 0 neither yet, 1 rung 0, 2 rung R - 1
    unsigned long long* acc_prev;  // [C] the chain's accepted-move counter at the last attribution
    unsigned long long* stats;     // swaps tried [R-1], swaps accepted [R-1], moves tried [R], moves accepted [R], round trips [n_ladders]
};

// One thread per ladder, after a full sweep:
//  1. the moves each chain made since the last call (`moves` tried, accepted[c] - acc_prev[c] accepted) are added to the
//     counters of the rung it held while making them;
//  2. swap != 0: round `round` proposes the pairs (i, i+1) with i = round (mod 2), in rung order, each accepted with
//     probability min(1, exp((beta_i - beta_{i+1}) (S_i - S_{i+1}))) where S is entropy() of the chain holding the rung.
//     The uniform draw is Philox keyed by swap_seed with counter (pair, ladder, round): a pure function of the call's
//     arguments, so a tempering run is deterministic whenever its sweeps are;
//  3. round trips: a chain that reaches rung R - 1 after rung 0, then rung 0 again, completes one.
__global__ void tempering_swap_kernel(LadderView L, const double* __restrict__ S, const unsigned long long* __restrict__ accepted,
                                      uint64_t moves, int swap, uint64_t round, uint64_t swap_seed) {
    const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L.n_ladders) return;
    const uint32_t R = L.R;
    uint32_t* const at = L.chain_at + (size_t)l * R;
    unsigned long long* const sw_tried = L.stats;
    unsigned long long* const sw_acc = sw_tried + (R - 1);
    unsigned long long* const mv_tried = sw_acc + (R - 1);
    unsigned long long* const mv_acc = mv_tried + R;
    unsigned long long* const trips = mv_acc + R;
    for (uint32_t i = 0; i < R; ++i) {
        const uint32_t c = at[i];
        const unsigned long long a = accepted[c];
        if (moves) atomicAdd(&mv_tried[i], (unsigned long long)moves);
        if (a != L.acc_prev[c]) atomicAdd(&mv_acc[i], a - L.acc_prev[c]);
        L.acc_prev[c] = a;
    }
    if (!swap || R < 2) return;
    for (uint32_t i = (uint32_t)(round & 1u); i + 1 < R; i += 2) {
        const uint32_t ci = at[i], cj = at[i + 1];
        const double x = (L.rung_beta[i] - L.rung_beta[i + 1]) * (S[ci] - S[cj]);
        u32x4 ctr; ctr.x = i; ctr.y = l; ctr.z = (uint32_t)round; ctr.w = (uint32_t)(round >> 32);
        const u32x4 ra = philox4x32(ctr, (uint32_t)swap_seed ^ 0x7F4A7C15u, (uint32_t)(swap_seed >> 32) ^ 0x3C6EF372u);
        const bool go = (x >= 0.0) || (((double)ra.x + 0.5) * (1.0 / 4294967296.0) < exp(x));
        atomicAdd(&sw_tried[i], 1ull);
        if (go) {
            atomicAdd(&sw_acc[i], 1ull);
            at[i] = cj; at[i + 1] = ci;
            L.rung_of[cj] = i; L.rung_of[ci] = i + 1;
            L.beta[cj] = L.rung_beta[i]; L.beta[ci] = L.rung_beta[i + 1];
        }
    }
    const uint32_t cold = at[0], hot = at[R - 1];
    if (L.trip[cold] == 2) trips[l] += 1;
    L.trip[cold] = 1;
    if (L.trip[hot] == 1) L.trip[hot] = 2;
}

#endif  // __CUDACC__

}  // namespace bisbm
