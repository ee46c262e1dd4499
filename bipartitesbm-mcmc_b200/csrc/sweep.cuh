// sweep.cuh -- parallel mode: many independent chains per launch.
//
// Mapping: LANE = CHAIN.  A warp takes one vertex v and evaluates v's move for the 32 chains of
// one chain group at once; labels are chain-minor (labels[v][C]) so "neighbour j's label for 32
// chains" is ONE coalesced 128-byte load and the CSR row of v is read once for all of them.
// A half sweep moves only the vertices of one type: their neighbours (all of the other type) are
// frozen, so every neighbour-block count is exact and the committed m_rs / e_r / n_r / eta
// deltas keep the counts exactly consistent with the labels; concurrent moves of one chain
// couple only through slightly stale count READS.
//
// The round-1 kernel here keeps every count (m_rs, e_r, n_r, eta) in HBM/L2: L2 loads
// (ld.global.cg) and global atomics per move, so every CTA sees every committed move at once
// and the "would empty block r" veto of apply_mcmc_moves is an exact atomic
// decrement-and-check.  It serves the graphs and K the staged kernel of sweep2.cuh cannot
// take (hubs of degree > 255, K > 256 per type).  In estimate mode (SweepParams::vary_k) the veto
// is off and dS carries the change of the K-dependent prior terms, as in sweep2_kernel.
//
// Per move this is the arithmetic of the reference's step():
//   proposal   single_vertex_change      reference src/blockmodel.cc:613-637
//   dS, accu_r transition_ratio          reference src/metropolis_hasting.cc:103-192
//   accept     step                      reference src/metropolis_hasting.cc:42-62
//   commit     apply_mcmc_moves          reference src/blockmodel.cc:461-503
// evaluated in ONE pass over v's neighbours (no N x K matrix k_, no 2E-entry lgamma table):
// with c = number of earlier neighbours of v in the same block t,
//   lgamma(m_rt+1) - lgamma(m_rt-k_t+1) - lgamma(m_st+k_t+1) + lgamma(m_st+1)
//        = sum over v's edges into t of  log(m_rt - c) - log(m_st + 1 + c)
//   accu0 = sum_edges (m_st + eps) / (e_t + eps K),
//   accu1 = sum_edges (m_rt + eps - (2c+1)) / (e_t + eps K)      [sum_c (2c+1) = k_t^2]
// the e_r terms by an Euler-Maclaurin (midpoint) difference, log q(n,k) from the exact table
// (n < 10001), a per-block second-order expansion refreshed every half sweep (large blocks),
// or the full formula.
#pragma once
#include "state.cuh"

namespace bisbm {

// expansion of f(e,n) = log q(e,n) about (e0,n0) for one (chain, block slot): second order in (e, n) plus the third
// order in e.  First derivatives in double (they multiply the degree / one node: fe * d ~ 0.1, fn ~ 10), the rest float.
// 48 bytes.
struct LogqExp {
    int32_t e0, n0;
    double fe, fn;
    float fee, fen, fnn, feee;
    uint32_t valid, pad;
};

struct SweepParams {
    GraphView g;
    StateView s;                     // s.m / s.e = BASE counts of this launch
    Tables tb;
    uint8_t* lab8;                   // sweep2_kernel: u8 shadow of the labels (chain-minor), 4x less gather traffic
    int32_t* m_next;                 // staged sweep2_kernel, sliced launches: where the staged m_rs / e_r are added
    int32_t* e_next;
    const uint64_t* seeds;           // [C]
    const uint8_t* active;           // [C]
    unsigned long long* accepted;    // [C]
    double* dS_accum;                // [C]
    const LogqExp* lq;               // [C/32][KA+KB][32]
    uint32_t n_chains;               // real chains (<= C)
    uint32_t type;                   // 0: move type-a vertices, 1: type-b
    uint32_t n_groups;               // C / 32
    uint32_t ctas_per_group;
    uint32_t warps_used;             // warps per CTA that take vertices (<= blockDim/32)
    uint32_t pos_begin, pos_end;     // slice of the permuted visiting order handled by this launch
    uint32_t half_bits;              // Feistel domain of this half sweep
    uint32_t kopp_max;               // max blocks of the opposite type (histogram stride)
    uint32_t exclusive;              // 1: one CTA per group -> write staged counts back directly
    uint64_t sweep;                  // sweep index: RNG counter and permutation key
    uint64_t step_base;              // global step index of position 0 of this half sweep
    int schedule;
    float p0, p1;
    // sweep2_kernel (sweep2.cuh)
    int32_t* nr_next;                // sliced launches: where the n_r view is added
    int32_t* nr_live;                // sliced launches: decrements of n_r within the launch (zero at its start), the exact "would
                                     // empty" counters of blocks small enough to empty within a launch
    // sweep2: where eta is READ and where its commits go.  Sliced staged launches read eta as it was at their start (a buffer no
    // launch writes meanwhile) and commit into the next launch's buffer; otherwise both are s.eta
    const int32_t* eta_read;
    int32_t* eta_commit;
    // sliced staged launches: after griddepcontrol.wait the CTAs of a group share the buffer work for the launches around this one
    // (launch_full_sweep): eta_commit += eta_read (moving type; with the launch's commits it becomes the next launch's eta_read),
    // eta_zero := 0 (the moving type's eta_commit of the next launch), m_zero / e_zero / nr_zero := 0 (the base of the previous
    // launch, where the next launch publishes), nr_live_zero := 0 (the nr_live of the next launch)
    int32_t* eta_zero;
    int32_t *m_zero, *e_zero, *nr_zero, *nr_live_zero;
    uint32_t group_offset;           // first chain group of this launch (0 except for single-group launches)
    uint32_t kat_mode;               // 1: evaluate ONE forced proposal (kat_v -> own-type block kat_s of chain kat_chain) and write
    uint32_t kat_chain, kat_v, kat_s;   //    {dS, log accu_r} to kat_out instead of accepting / committing (bisbm_parallel_transition)
    double* kat_out;
    double beta0;                    // 1 / p0, computed once on the host (constant schedule: 1/T of every step)
    // spare SMs (sliced staged launches whose groups x CTAs do not fill the GPU): `extras` more CTAs per launch, handed to the
    // groups in turn (extra slot number s of the half sweep goes to group s mod n_groups; launch l hands out slots
    // [l extras, (l+1) extras)); a group's positions then advance by (ctas_per_group + its extra) x per_cta per launch
    uint32_t extras, launch_idx, per_cta;
    uint32_t vary_k;                 // estimate mode (README "estimation"): blocks may empty and be re-populated; the K-dependent
                                     // prior terms of the description length enter dS with the OCCUPIED block counts
    const double* beta_chain;        // [C] parallel tempering: 1/T of each chain's rung, loaded once per lane (the launch then runs
                                     // at constant temperature and schedule / p0 / beta0 are ignored); null: one schedule for all
};

// temperature of global step t (same five schedules as src/metropolis_hasting.cc:10-37,
// device libm for pow / log); out of line, the constant schedule never calls it
BISBM_NOINLINE_HD static double par_temperature(int schedule, float p0, float p1, uint64_t t) {
    switch (schedule) {
        case 0: return (double)p0 * pow((double)p1, (double)t);
        case 1: return (double)(p0 - p1 * (float)t);
        case 2: {
            uint64_t i = (uint64_t)((float)t + p1);
            double l = (i == 0) ? 0.0 : log((double)i);
            return (double)p0 / l;
        }
        case 3: return (double)p0;
        default: return ((float)t < p0) ? 1.0 : 0.0;
    }
}

// lgamma(x + d) - lgamma(x) for integers x >= 1, d >= 0: Stirling difference with log1p for
// large x, direct lgamma for small x.  Out of line (rare path; keeps the kernel small).
BISBM_NOINLINE_HD static double lgamma_diff(double x, double d) {
    if (d == 0.0) return 0.0;
    if (x < 32.0) return lgamma(x + d) - lgamma(x);
    double y = x + d;
    double ix = 1.0 / x, iy = 1.0 / y;
    double ser = (iy - ix) * (1.0 / 12.0) - (iy * iy * iy - ix * ix * ix) * (1.0 / 360.0) +
                 (iy * iy * iy * iy * iy - ix * ix * ix * ix * ix) * (1.0 / 1260.0);
    return (x - 0.5) * log1p(d * ix) + d * (log(y) - 1.0) + ser;
}

// [lgamma(e_s+d+1) - lgamma(e_s+1)] - [lgamma(e_r+1) - lgamma(e_r-d+1)]
//   = sum_{i<d} log(e_s+1+i) - sum_{i<d} log(e_r-d+1+i).
// Midpoint Euler-Maclaurin: sum_{i<d} log(x+i) = d log c - (d^3-d)/(24 c^2) - (3d^5-10d^3+7d)/(960 c^4) - ...
// with c = x + (d-1)/2; used when both c >= 32 d (next term < 1e-10), else the Stirling form.
BISBM_HD double block_degree_delta(int e_r, int e_s, int d) {
    if (d == 0) return 0.0;
    const double D = (double)d;
    const double cs = (double)e_s + 0.5 * (D + 1.0), cr = (double)e_r - 0.5 * (D - 1.0);
    if (cs >= 32.0 * D && cr >= 32.0 * D) {
        const double is2 = 1.0 / (cs * cs), ir2 = 1.0 / (cr * cr);
        const double D2 = D * D;
        const double k3 = D * (D2 - 1.0) * (1.0 / 24.0);
        const double k5 = D * ((3.0 * D2 - 10.0) * D2 + 7.0) * (1.0 / 960.0);
        return D * log(cs / cr) - k3 * (is2 - ir2) - k5 * (is2 * is2 - ir2 * ir2);
    }
    return lgamma_diff((double)(e_s + 1), D) - lgamma_diff((double)(e_r - d + 1), D);
}

// exact (table / full asymptotic formula) difference: the rare slow path, out of line
BISBM_NOINLINE_HD static double logq_delta_exact(const Tables& tb, int e, int n, int de, int dn) {
    return log_q(tb, e + de, n + dn) - log_q(tb, e, n);
}

// log q difference f(e+de, n+dn) - f(e, n) for one block
BISBM_HD double logq_delta(const Tables& tb, const LogqExp& q, int e, int n, int de, int dn) {
    int x = e - q.e0, y = n - q.n0;
    int ax = x < 0 ? -x : x, ay = y < 0 ? -y : y, ad = de < 0 ? -de : de;
    if (q.valid && ax <= (q.e0 >> 4) && ay <= (q.n0 >> 4) && ad <= (q.e0 >> 10)) {
        double dx = (double)x, dy = (double)y, De = (double)de, Dn = (double)dn;
        return q.fe * De + q.fn * Dn + 0.5 * (double)q.fee * (De * De + 2.0 * dx * De) +
               (double)q.fen * (dx * Dn + dy * De + De * Dn) + 0.5 * (double)q.fnn * (Dn * Dn + 2.0 * dy * Dn) +
               (double)q.feee * De * ((1.0 / 6.0) * De * De + 0.5 * dx * (De + dx));
    }
    return logq_delta_exact(tb, e, n, de, dn);
}

// running sums of the one-pass evaluation of transition_ratio
struct MoveAcc {
    double a0, a1, num, den, logacc;
};
BISBM_HD void acc_init(MoveAcc& A) { A.a0 = 0.0; A.a1 = 0.0; A.num = 1.0; A.den = 1.0; A.logacc = 0.0; }
// one edge of v into block t: c earlier edges of v into t, counts m_rt, m_st, inv = 1/(e_t + eps K)
BISBM_HD void acc_edge(MoveAcc& A, int m_r, int m_s, int c, double inv, double eps) {
    A.a0 += ((double)m_s + eps) * inv;
    A.a1 += ((double)(m_r - 2 * c - 1) + eps) * inv;
    A.num *= (double)(m_r - c);
    A.den *= (double)(m_s + 1 + c);
}
BISBM_HD void acc_guard(MoveAcc& A) {  // keep the running products inside double range
    if (A.num > 1e140 || A.den > 1e140) { A.logacc += log(A.num / A.den); A.num = 1.0; A.den = 1.0; }
}

#ifdef __CUDACC__

// counts in global memory are updated with L2 atomics by every SM; L1 is not coherent, so every
// count READ from global goes to L2 (ld.global.cg).
__device__ __forceinline__ int ldc(const int32_t* p) { return __ldcg(p); }

#endif  // __CUDACC__ (reopened below)

// Coefficients of the expansion about (e0, n0) by central differences of the reference's asymptotic formula
// (log_q_approx, src/support/int_part.cc:73-98): first derivatives with a small step (truncation: third derivative
// times h^2 / 6 times the degree, below 1e-10), second / third derivatives with a larger one (round-off).  Blocks too
// small for the asymptotic branch, or where the expansion would be poor, get valid = 0 and take the exact routine.
// The 15 points of the stencil: 0 centre; 1, 2 (e0 +- h1); 3, 4 (n0 +- k1); 5 .. 8 (e0 + he, - he, + 2 he, - 2 he);
// 9, 10 (n0 +- hn); 11 .. 14 the corners (+,+), (+,-), (-,+), (-,-) of (he, hn).
BISBM_HD bool logq_expandable(int e0, int n0) { return e0 >= 16384 && n0 >= 1024 && 2 * (int64_t)n0 <= (int64_t)e0; }
BISBM_HD void logq_stencil(int e0, int n0, int i, int* e, int* n) {
    const int h1 = (e0 >> 13) > 1 ? (e0 >> 13) : 1, k1 = (n0 >> 11) > 1 ? (n0 >> 11) : 1;
    const int he = e0 >> 10, hn = n0 >> 8;
    int de = 0, dn = 0;
    switch (i) {
        case 1: de = h1; break;       case 2: de = -h1; break;
        case 3: dn = k1; break;       case 4: dn = -k1; break;
        case 5: de = he; break;       case 6: de = -he; break;
        case 7: de = 2 * he; break;   case 8: de = -2 * he; break;
        case 9: dn = hn; break;       case 10: dn = -hn; break;
        case 11: de = he; dn = hn; break;    case 12: de = he; dn = -hn; break;
        case 13: de = -he; dn = hn; break;   case 14: de = -he; dn = -hn; break;
        default: break;
    }
    *e = e0 + de; *n = n0 + dn;
}
BISBM_HD LogqExp logq_from_stencil(int e0, int n0, const double* f) {
    LogqExp q;
    q.e0 = e0; q.n0 = n0; q.pad = 0;
    const int h1 = (e0 >> 13) > 1 ? (e0 >> 13) : 1, k1 = (n0 >> 11) > 1 ? (n0 >> 11) : 1;
    const double He = (double)(e0 >> 10), Hn = (double)(n0 >> 8);
    q.fe = (f[1] - f[2]) / (2.0 * (double)h1);
    q.fn = (f[3] - f[4]) / (2.0 * (double)k1);
    q.fee = (float)((f[5] - 2.0 * f[0] + f[6]) / (He * He));
    q.fnn = (float)((f[9] - 2.0 * f[0] + f[10]) / (Hn * Hn));
    q.fen = (float)((f[11] - f[12] - f[13] + f[14]) / (4.0 * He * Hn));
    q.feee = (float)((f[7] - 2.0 * f[5] + 2.0 * f[6] - f[8]) / (2.0 * He * He * He));
    q.valid = 1;
    return q;
}
BISBM_HD LogqExp logq_invalid(int e0, int n0) {
    LogqExp q;
    q.e0 = e0; q.n0 = n0; q.fe = 0.0; q.fn = 0.0; q.fee = q.fen = q.fnn = q.feee = 0.f; q.valid = 0; q.pad = 0;
    return q;
}
BISBM_HD LogqExp logq_expand(const Tables& tb, int e0, int n0) {
    if (!logq_expandable(e0, n0)) return logq_invalid(e0, n0);
    double f[15];
    for (int i = 0; i < 15; ++i) {
        int e, n;
        logq_stencil(e0, n0, i, &e, &n);
        f[i] = log_q_approx(tb, e, n);
    }
    return logq_from_stencil(e0, n0, f);
}

#ifdef __CUDACC__
// Refresh the log q expansions of the blocks of one type (they only change during that
// type's half sweep).
// lazy != 0 (between the slice launches of a half sweep): only the blocks that have drifted more than 1/64 of (e0, n0) from
// their expansion point -- a quarter of the validity range of logq_fast -- are expanded again; at stationarity that is none
// and the kernel is a few loads per block, while quenches and burn-in (blocks changing by more than the 6 % range within one
// half sweep) stop falling onto the out-of-line exact path.
__global__ void logq_refresh_kernel(StateView s, Tables tb, LogqExp* lq, uint32_t n_chains, uint32_t type, uint32_t lazy = 0) {
    // 16 lanes per (chain, block): the 15 evaluations of the asymptotic formula run side by side (one thread doing all of them
    // set the kernel's duration: 123 us whenever a single block needed its expansion)
    const uint32_t gt = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t idx = gt >> 4, sub = gt & 15u;
    const uint32_t seg = (threadIdx.x & 16u), segmask = 0xffffu << seg;
    uint32_t kmax = type ? s.KB : s.KA;
    if (idx >= n_chains * kmax) return;
    // consecutive segments = consecutive chains of one block slot
    uint32_t b = idx / n_chains, c = idx % n_chains;
    uint32_t kc = type ? s.kb[c] : s.ka[c];
    uint32_t slot = (type ? s.KA : 0) + b;
    const size_t off = cnt_base(c, (size_t)s.KA + s.KB) + (size_t)slot * GROUP;
    if (b >= kc) {
        if (!lazy && sub == 0) lq[off] = logq_invalid(0, 0);
        return;
    }
    const int e = s.e[off], n = s.nr[off];
    if (lazy) {
        const int e0 = lq[off].e0, n0 = lq[off].n0;
        const int ax = e > e0 ? e - e0 : e0 - e, ay = n > n0 ? n - n0 : n0 - n;
        if (lq[off].valid ? (ax <= (e0 >> 6) && ay <= (n0 >> 6)) : (e == e0 && n == n0)) return;
    }
    if (!logq_expandable(e, n)) {
        if (sub == 0) lq[off] = logq_invalid(e, n);
        return;
    }
    int es, ns;
    logq_stencil(e, n, (int)(sub < 14u ? sub : 14u), &es, &ns);
    const double fv = log_q_approx(tb, es, ns);
    double f[15];
#pragma unroll
    for (int i = 0; i < 15; ++i) f[i] = __shfl_sync(segmask, fv, (int)seg + i);
    if (sub == 0) lq[off] = logq_from_stencil(e, n, f);
}

// shared memory of sweep_kernel: the warps' neighbour-block histograms, HistT hist[warps][kopp_max*32]
__host__ __device__ inline size_t sweep_smem_bytes(uint32_t KA, uint32_t KB, uint32_t type, uint32_t warps, uint32_t hist_bytes) {
    const uint32_t kopp = type ? KA : KB;
    return (size_t)warps * ((kopp * hist_bytes + 3) / 4) * 128;   // lane-major 32-bit words
}

// 16-byte staged copy (all staged arrays are multiples of 128 bytes; sweep2.cuh)
__device__ __forceinline__ void copy_i4(int32_t* dst, const int32_t* src, uint32_t n_int) {
    const int4* s4 = reinterpret_cast<const int4*>(src);
    int4* d4 = reinterpret_cast<int4*>(dst);
    const uint32_t n4 = n_int / 4;
    for (uint32_t i0 = threadIdx.x; i0 < n4; i0 += 4 * blockDim.x) {   // four loads in flight per thread
        int4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { const uint32_t i = i0 + u * blockDim.x; if (i < n4) v[u] = s4[i]; }
#pragma unroll
        for (int u = 0; u < 4; ++u) { const uint32_t i = i0 + u * blockDim.x; if (i < n4) d4[i] = v[u]; }
    }
}

// ---- explicit shared-space accesses on 32-bit shared addresses (ld/st/red.shared): the
//      staged counts of sweep2.cuh are only ever touched through these, so no generic-address
//      LD/ATOM and no 64-bit index arithmetic is left in the move loop ----
// (count / inverse loads are plain asm so the compiler may schedule them early; a value that is a
//  few instructions stale is harmless -- other warps update the same entries concurrently anyway)
__device__ __forceinline__ int sh_ld(uint32_t a) { int v; asm("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sh_red_add(uint32_t a, int v) { asm volatile("red.shared.add.s32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
template <typename T> struct ShHist;
template <> struct ShHist<uint8_t> {
    static __device__ __forceinline__ uint32_t ld(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
    static __device__ __forceinline__ void st(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
};
template <> struct ShHist<uint16_t> {
    static __device__ __forceinline__ uint32_t ld(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
    static __device__ __forceinline__ void st(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
};
template <> struct ShHist<uint32_t> {
    static __device__ __forceinline__ uint32_t ld(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
    static __device__ __forceinline__ void st(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
};

// one lane's view of a count array in global memory: entry j of this chain is element [j*32]; L2 loads, global reductions
struct Cnt {
    int32_t* p;
    __device__ __forceinline__ int ld(uint32_t idx32) const { return __ldcg(p + idx32); }
    __device__ __forceinline__ void add(uint32_t idx32, int v) const { atomicAdd(p + idx32, v); }
};

// estimate mode: change of the K-dependent terms of entropy() (src/blockmodel.cc:780-782: lbinom(Ka Kb + E - 1, E) +
// lbinom(na - 1, Ka - 1) + lbinom(nb - 1, Kb - 1)) when the number of occupied blocks of the moving type goes k -> k + dk.
// Out of line: a move changes the occupied count rarely.  Used by sweep_kernel and sweep2_kernel.
__device__ __noinline__ static double prior_k_delta(double E, double n_own, double k_own, double k_opp, int dk) {
    auto lbin = [](double N, double k) -> double {
        if (N == 0.0 || k == 0.0 || k > N) return 0.0;
        return lgamma(N + 1.0) - lgamma(k + 1.0) - lgamma(N - k + 1.0);
    };
    const double k2 = k_own + (double)dk;
    return (lbin(k2 * k_opp + E - 1.0, E) + lbin(n_own - 1.0, k2 - 1.0)) - (lbin(k_own * k_opp + E - 1.0, E) + lbin(n_own - 1.0, k_own - 1.0));
}

template <typename HistT, int NT>
__global__ void __launch_bounds__(NT, 1) sweep_kernel(SweepParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // lane / warp ids through volatile asm: the compiler must keep them in registers instead of
    // re-deriving them from S2R + ALU at every use (it did so ~40 times per vertex under the 64-register cap)
    uint32_t lane, warp;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(warp));
    warp >>= 5;
    const uint32_t wpc = blockDim.x >> 5;
    const GraphView& G = P.g;
    const uint32_t type = P.type;
    const uint32_t C = P.s.C, KB = P.s.KB, KA = P.s.KA, W = P.s.W, KK = KA + KB;
    const uint32_t kown_max = type ? KB : KA, kopp_max = P.kopp_max;
    const uint32_t group = blockIdx.x % P.n_groups;
    const uint32_t cta_in_group = blockIdx.x / P.n_groups;
    const uint32_t own_off = type ? KA : 0, opp_off = type ? 0 : KA;

    // global (group-interleaved) count arrays of this group
    int32_t* const gM = P.s.m + (size_t)group * KA * KB * GROUP;
    int32_t* const gE = P.s.e + (size_t)group * KK * GROUP;
    // (warp-uniform bases; the lane is added in the 32-bit index so they can live in uniform registers)
    int32_t* const gNR = P.s.nr + (size_t)group * KK * GROUP + (size_t)own_off * 32;         // own-type slots
    int32_t* const gETA = P.s.eta + (size_t)group * KK * W * GROUP + (size_t)own_off * W * 32;
    const LogqExp* const gLQ = P.lq + (size_t)group * KK * GROUP + (size_t)own_off * 32;

    const uint32_t c = group * 32 + lane;
    const bool live = (c < P.n_chains) && P.active[c];
    const uint32_t cc = (c < P.s.C) ? c : 0;
    const uint32_t ka = P.s.ka[cc], kb = P.s.kb[cc], K = ka + kb;
    const uint32_t kown = type ? kb : ka;
    const double eps = P.s.eps, epsK = eps * (double)K;

    HistT* const hist_all = reinterpret_cast<HistT*>(smem_raw);
    {
        uint32_t* hw = reinterpret_cast<uint32_t*>(hist_all);
        const uint32_t words = wpc * (((kopp_max * (uint32_t)sizeof(HistT) + 3u) / 4u)) * 32u;
        for (uint32_t i = threadIdx.x; i < words; i += blockDim.x) hw[i] = 0u;
    }
    __syncthreads();

    // lane-private accessors (entry j of this chain at element j*32)
    Cnt M, Eo, Ep;
    M.p = gM + lane; Eo.p = gE + own_off * 32 + lane; Ep.p = gE + opp_off * 32 + lane;
    // histogram bins are packed BPW per 32-bit word and the words are LANE-MAJOR ([t / BPW][lane]), so
    // lane l only ever touches bank l: bin t of this lane is at hist_base + (t / BPW) * 128 + (t % BPW) * sizeof(HistT)
    constexpr uint32_t BPW = 4u / (uint32_t)sizeof(HistT);
    const uint32_t hist_words = (kopp_max + BPW - 1) / BPW;
    const uint32_t hist_base = (uint32_t)__cvta_generic_to_shared(hist_all) + warp * hist_words * 128u + lane * 4u;
    auto hist_addr = [&](uint32_t t) -> uint32_t {
        if constexpr (BPW == 1) return hist_base + t * 128u;
        else return hist_base + (t / BPW) * 128u + (t % BPW) * (uint32_t)sizeof(HistT);
    };
    // m(x_own, t_opp) = M[x*sx + t*st]   (element indices, already multiplied by the 32-chain interleave)
    const uint32_t sx = (type ? 1u : KB) * 32u, st = (type ? KB : 1u) * 32u;
    int32_t* const LAB = P.s.labels;
    auto label_of = [&](uint32_t vtx) -> uint32_t { return (uint32_t)LAB[(size_t)vtx * C + cc]; };
    const uint64_t seed = P.seeds[cc];
    const uint32_t key0 = (uint32_t)seed, key1 = (uint32_t)(seed >> 32);
    const uint32_t nv = type ? G.nb : G.na, v0 = type ? G.na : 0;
    const uint64_t pkey = (P.sweep * 2 + type) * 0x9E3779B97F4A7C15ull + (uint64_t)group * 0xD1B54A32D192ED03ull;
    constexpr int SAFE_NR = 8192;   // > any number of concurrently evaluated moves of one chain (<= 148 SMs * 32 warps)
    const bool const_T = (P.schedule == 3) || P.beta_chain;
    double T_const = (double)P.p0, beta_const = 1.0 / (double)P.p0;
    if (P.beta_chain) { beta_const = P.beta_chain[cc]; T_const = 1.0 / beta_const; }   // (a ladder never holds T = 0)

    // estimate mode: occupied blocks of this lane's chain, per type (own type tracked through this warp's own moves)
    int occ_own = 0, occ_opp = 0;
    if (P.vary_k) {
        const int32_t* const gNRopp = P.s.nr + (size_t)group * KK * GROUP + (size_t)opp_off * 32;
        for (uint32_t b = 0; b < kown_max; ++b) occ_own += (ldc(&gNR[b * 32 + lane]) > 0) ? 1 : 0;
        for (uint32_t b = 0; b < kopp_max; ++b) occ_opp += (ldc(&gNRopp[b * 32 + lane]) > 0) ? 1 : 0;
    }

    unsigned long long n_acc = 0;
    double ds_sum = 0.0;

    if (warp < P.warps_used) {
        const uint32_t stride = P.ctas_per_group * P.warps_used;
        const uint32_t i_first = P.pos_begin + cta_in_group * P.warps_used + warp;
        // Vertices are taken in batches of 32: lane l prepares the l-th vertex of the batch (its
        // place in the permuted order, CSR row offset and degree) -- the Feistel permutation and
        // the dependent row_ptr loads cost one lane-parallel step per 32 vertices instead of one
        // warp-uniform step per vertex.  The first 32 neighbour ids of the NEXT vertex are
        // prefetched with one coalesced load (lane e holds neighbour e; broadcast by shuffle).
        uint32_t bv = 0, brow = 0, bdeg = 0, bdidx = 0;      // this lane's vertex of the current batch
        // software pipeline, one vertex ahead: everything below with suffix _n belongs to the NEXT
        // vertex and is loaded while the current one is evaluated (own label, Philox draw, the
        // proposal's random neighbour id and -- one stage later -- that neighbour's label)
        uint32_t v_n = 0, row_n = 0, d_n = 0, nbr_n = 0, r_n = 0, j_n = 0, t_n = 0, didx_n = 0;
        u32x4 ra_n; ra_n.x = ra_n.y = ra_n.z = ra_n.w = 0;
        auto refill = [&](uint32_t pos0) {        // lane l prepares the vertex at position pos0 + l*stride
            const uint64_t il = (uint64_t)pos0 + (uint64_t)lane * stride;
            bv = 0; brow = 0; bdeg = 0; bdidx = 0;
            if (il < P.pos_end) {
                bv = v0 + feistel_perm((uint32_t)il, nv, P.half_bits, pkey);
                brow = G.row_ptr[bv];
                bdeg = G.row_ptr[bv + 1] - brow;
                bdidx = G.degidx[bv];
            }
        };
        auto prefetch = [&](uint32_t slot) {      // stage 1 of the pipeline for the vertex in batch slot `slot`
            v_n = __shfl_sync(0xffffffffu, bv, slot);
            row_n = __shfl_sync(0xffffffffu, brow, slot);
            d_n = __shfl_sync(0xffffffffu, bdeg, slot);
            didx_n = __shfl_sync(0xffffffffu, bdidx, slot);
            nbr_n = (lane < d_n) ? G.col[row_n + lane] : 0u;
            r_n = live ? label_of(v_n) : 0u;
            u32x4 ctr; ctr.x = v_n; ctr.y = (uint32_t)P.sweep; ctr.z = (uint32_t)(P.sweep >> 32); ctr.w = 0;
            ra_n = philox4x32(ctr, key0, key1);
            j_n = (live && d_n != 0) ? G.col[row_n + mulhi32(ra_n.x, d_n)] : 0u;   // differs per lane: plain gather
        };
        if (i_first < P.pos_end) {
            refill(i_first);
            prefetch(0);
            t_n = (live && d_n != 0) ? label_of(j_n) : 0u;
        }
        for (uint32_t ib = i_first, k = 0; ib < P.pos_end; ib += stride, ++k) {
            // warp-uniform trip count: all 32 lanes (= chains) reconverge at every vertex
            __syncwarp();
            const uint32_t v = v_n, row = row_n, d = d_n, nbr0 = nbr_n, r = r_n, t_prop = t_n, didx = didx_n;
            const u32x4 ra = ra_n;
            const bool has_next = (ib + stride < P.pos_end);
            if (has_next) {
                if (((k + 1) & 31u) == 0) refill(ib + stride);
                prefetch((k + 1) & 31u);
            }
            const uint32_t i = ib;
            const double T = const_T ? T_const : par_temperature(P.schedule, P.p0, P.p1, P.step_base + i);

            // ---- proposal (single_vertex_change), branch-free: every lane computes both the uniform
            //      and the categorical candidate and selects ----
            const uint32_t tq = min(t_prop, kopp_max - 1u);   // (an isolated vertex has no proposal neighbour: any valid slot)
            const int e_t = Ep.ld(tq * 32u);
            const bool uniform_pick = (d == 0) || (((double)ra.y * (1.0 / 4294967296.0)) < epsK / ((double)e_t + epsK));
            const uint32_t sg = mulhi32(ra.z, K);      // uniform over ALL K blocks (either type)
            const bool sg_a = sg < ka;
            const uint32_t s_uni = sg_a ? sg : sg - ka;
            // categorical over row m[t][.]: block x of the own type w.p. m(x,t)/e_t;
            // s = #{x : cum_x <= z} (cum is non-decreasing), no early exit
            const uint32_t z = mulhi32(ra.z, (uint32_t)e_t);
            uint32_t cum = 0, cnt_le = 0;
            {
                uint32_t idx = tq * st;
#pragma unroll 8
                for (uint32_t x = 0; x < kown_max; ++x, idx += sx) {   // uniform bound; blocks >= kown hold 0
                    cum += (uint32_t)M.ld(idx);
                    cnt_le += (cum <= z) ? 1u : 0u;
                }
            }
            const uint32_t s_cat = cnt_le < kown ? cnt_le : kown - 1;
            const bool movable = live && (kown != 1);
            const bool cross = movable && uniform_pick && (sg_a != (type == 0));  // fell on a block of the other type: s stays r
            const uint32_t s = (movable && !cross) ? (uniform_pick ? s_uni : s_cat) : r;   // own-type local index of the target
            // stage 2 of the pipeline: the label of the next vertex's proposal neighbour (its id has
            // arrived by now)
            if (has_next) t_n = (live && d_n != 0) ? label_of(j_n) : 0u;
            // dS = +inf for a cross-type target (rejected); dS = 0, accu_r = 1 for s == r: at T > 0
            // accepted unless the block would empty, at T == 0 the reference requires dS < 0
            // (src/metropolis_hasting.cc:47-52)
            const bool eval = live && !cross && (s != r);
            if (live && !cross && s == r) {
                if (T != 0.0 && ldc(&gNR[r * 32 + lane]) != 1) ++n_acc;
            }
            __syncwarp();
            if (!__any_sync(0xffffffffu, eval)) continue;

            // ---- one pass over v's neighbours: dS and the Hastings factor (transition_ratio) ----
            int n_r = 0, n_s = 0, eta_r = 1, eta_s = 0;
            MoveAcc A; acc_init(A);
            const uint32_t ir = r * sx, is = s * sx;
            // issue the global (L2) loads early; they are consumed after the pass
            n_r = ldc(&gNR[r * 32 + lane]); n_s = ldc(&gNR[s * 32 + lane]);
            eta_r = ldc(&gETA[(r * W + didx) * 32 + lane]);
            eta_s = ldc(&gETA[(s * W + didx) * 32 + lane]);
            // Every lane runs the pass, also lanes whose proposal needs no evaluation (s == r, cross-type,
            // padding chains): masked lanes cost the same issue slots anyway, and dropping the per-lane
            // predicates removes the divergence bookkeeping from the loop.  Their result is ignored.
            uint32_t nbr = nbr0;  // lane e holds neighbour (base & ~31) + e
            auto consume = [&](uint32_t t) {
                const uint32_t ha = hist_addr(t);
                const int cnt = (int)ShHist<HistT>::ld(ha);
                ShHist<HistT>::st(ha, (uint32_t)(cnt + 1));
                const uint32_t it = t * st;
                const int m_r = M.ld(ir + it), m_s = M.ld(is + it);
                const double inv = 1.0 / ((double)Ep.ld(t * 32u) + epsK);
                acc_edge(A, m_r, m_s, cnt, inv, eps);
            };
            uint32_t base = 0;
            for (; base + 8 <= d; base += 8) {
                // gather 8 neighbour labels (independent 128-byte loads in flight), then consume them
                if (base != 0 && (base & 31u) == 0) nbr = (base + lane < d) ? G.col[row + base + lane] : 0u;
                uint32_t tt[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) tt[q] = label_of(__shfl_sync(0xffffffffu, nbr, (base + q) & 31));
#pragma unroll
                for (int q = 0; q < 8; ++q) consume(tt[q]);
                acc_guard(A);
            }
            if (base < d) {   // tail of < 8 neighbours
                if (base != 0 && (base & 31u) == 0) nbr = (base + lane < d) ? G.col[row + base + lane] : 0u;
                uint32_t tt[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const uint32_t nb = __shfl_sync(0xffffffffu, nbr, (base + q) & 31);
                    tt[q] = (base + q < d) ? label_of(nb) : 0u;
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) if (base + q < d) consume(tt[q]);
                acc_guard(A);
            }
            __syncwarp();

            // dS and the accept test are evaluated by every lane (masked lanes cost the same issue
            // slots); only `eval` lanes may commit
            bool go;
            double dS;
            {
                const int e_r = Eo.ld(r * 32u), e_s = Eo.ld(s * 32u);
                // log( prod (m_rt-c)/(m_st+1+c) * eta_r/(eta_s+1) ) with a single division
                dS = A.logacc + log((A.num * (double)(eta_r > 0 ? eta_r : 1)) / (A.den * (double)(eta_s + 1)));
                dS += block_degree_delta(e_r, e_s, (int)d);
                dS += logq_delta(P.tb, gLQ[r * 32 + lane], e_r, n_r, -(int)d, -1);
                dS += logq_delta(P.tb, gLQ[s * 32 + lane], e_s, n_s, (int)d, 1);
                // estimate mode: the move empties r and / or opens s, the K-dependent prior terms change with the occupied count
                const int dk = ((n_s == 0) ? 1 : 0) - ((n_r == 1) ? 1 : 0);
                if (P.vary_k && eval && dk != 0)
                    dS += prior_k_delta((double)G.n_edges, (double)nv, (double)occ_own, (double)occ_opp, dk);
                // ---- accept (step) ----
                const double beta = const_T ? beta_const : 1.0 / T;
                const double a = ((d == 0) ? 0.0 : log(A.a1 / A.a0)) - dS * beta;
                const bool go_hot = (a > 0.0) || (((double)ra.w + 0.5) * (1.0 / 4294967296.0) < exp(a));
                go = eval && ((T == 0.0) ? (dS < 0.0) : go_hot);
                if (go && P.vary_k) {
                    atomicSub(&gNR[r * 32 + lane], 1);   // estimate mode: a block may empty
                    occ_own += dk;
                } else if (go) {
                    // the exact "would empty block r" veto of apply_mcmc_moves.  n_r was read from L2 a moment
                    // ago; fewer than SAFE_NR moves of this chain can be in flight, so a block that large
                    // cannot empty and a fire-and-forget reduction is enough (no round trip on the critical path)
                    if (n_r > SAFE_NR) {
                        atomicSub(&gNR[r * 32 + lane], 1);
                    } else {
                        const int old = atomicSub(&gNR[r * 32 + lane], 1);
                        if (old <= 1) { atomicAdd(&gNR[r * 32 + lane], 1); go = false; }
                    }
                }
            }
            __syncwarp();

            // ---- clear the histogram and commit (apply_mcmc_moves): k_t is the histogram ----
            {
                // one 32-bit word holds BPW bins: read and clear them together
                uint32_t ha = hist_base, it = 0;
#pragma unroll 2
                for (uint32_t w = 0; w < hist_words; ++w, ha += 128u) {   // uniform bound; bins >= kopp stay 0
                    const uint32_t word = ShHist<uint32_t>::ld(ha);
                    ShHist<uint32_t>::st(ha, 0u);
#pragma unroll
                    for (uint32_t b = 0; b < BPW; ++b, it += st) {
                        int kk;
                        if constexpr (BPW == 1) kk = (int)word;
                        else kk = (int)((word >> (b * 8u * (uint32_t)sizeof(HistT))) & ((1u << (8u * (uint32_t)sizeof(HistT))) - 1u));
                        if (go && kk != 0) {
                            M.add(ir + it, -kk);
                            M.add(is + it, kk);
                        }
                    }
                }
                if (go) {
                    Eo.add(r * 32u, -(int)d);
                    Eo.add(s * 32u, (int)d);
                    atomicAdd(&gNR[s * 32 + lane], 1);
                    atomicSub(&gETA[(r * W + didx) * 32 + lane], 1);
                    atomicAdd(&gETA[(s * W + didx) * 32 + lane], 1);
                    LAB[(size_t)v * C + cc] = (int32_t)s;
                    ++n_acc;
                    ds_sum += dS;
                }
            }
        }
        if (live) {
            if (n_acc) atomicAdd(&P.accepted[c], n_acc);
            if (ds_sum != 0.0) atomicAdd(&P.dS_accum[c], ds_sum);
        }
    }
}

#endif  // __CUDACC__

}  // namespace bisbm
