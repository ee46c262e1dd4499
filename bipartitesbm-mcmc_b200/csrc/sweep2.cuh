// sweep2.cuh -- the staged-count sweep kernel of parallel mode (round 2), one kernel text for both
// arithmetic types: sweep2_kernel<double, ..> evaluates a move in DOUBLE like the reference's
// transition_ratio (src/metropolis_hasting.cc:103-192) and is the default; sweep2_kernel<float, ..>
// is the optional fp32 / MUFU form (bisbm_set_precision).
//
// Mapping as in sweep.cuh: LANE = CHAIN, one warp per vertex, half sweeps alternate types, the chain
// group's counts live in shared memory laid out [entry][lane].  What is new here:
//   * double arithmetic without conversions on the XU pipe: counts become doubles by splicing the
//     integer under the exponent of 2^52 (one DADD each), products of up to 32 count ratios are folded
//     into ONE logarithm per vertex, 1/(e_t + eps K) comes from a per-launch table (e_t of the frozen
//     type cannot change during a half sweep), reciprocals are MUFU.RCP64H + two Newton steps;
//   * neighbour labels arrive as whole 32-byte rows (lane -> 8 bytes of one row, 8 rows per load
//     instruction), ONE VERTEX AHEAD, and are parked in a per-warp tile in shared memory as they are
//     ([edge][chain]: one 8-byte store per lane and block of 8 rows; a lane reads its chain's label of
//     edge e as one byte, 32 lanes = one 32-byte row, conflict-free) -- the five serial gather round
//     trips of the round-1 kernel are gone and the proposal's random neighbour label comes from the tile too;
//   * the warp's u8 neighbour-block histogram is updated with one shared atomic per edge (old value =
//     c), four edges of a chunk are independent instruction streams;
//   * the commit walks the edges again (2 shared reductions per edge) instead of all K bins;
//   * n_r has a per-CTA view in shared memory like m_rs / e_r; only blocks small enough to empty
//     within one slice (or every block, when one CTA owns the group: then the view is exact) use an
//     exact atomic decrement-and-check for the "would empty block r" veto of apply_mcmc_moves
//     (src/blockmodel.cc:467-471);
//   * the CTA's share of the slice is prepared once (Feistel position -> vertex, CSR row, degree) and
//     handed out to warps dynamically (no warp waits for the slowest one's static share);
//   * staging is one thread issuing bulk-async copies (cp.async.bulk + mbarrier); publishing is one
//     thread issuing bulk-async REDUCTIONS of the staged arrays themselves (cp.reduce.async.bulk
//     .add.s32): the CTAs of the group have added -(ctas_per_group - 1) * base into the next base at the start of the
//     launch, so the sum of all CTAs' staged copies is base + sum of their deltas -- no base re-read, no per-entry atomics.
//
// Per move this is still the arithmetic of the reference's step():
//   proposal   single_vertex_change      reference src/blockmodel.cc:613-637
//   dS, accu_r transition_ratio          reference src/metropolis_hasting.cc:103-192
//   accept     step                      reference src/metropolis_hasting.cc:42-62
//   commit     apply_mcmc_moves          reference src/blockmodel.cc:461-503
#pragma once
#include <string.h>
#include "sweep.cuh"

namespace bisbm {

// integer -> double by splicing the integer under the exponent of 2^52 and subtracting 2^52 (one DADD, no XU-pipe
// conversion): +1.5 % on the C3 bench (profiles/r02_experiments.txt); -DBISBM_NO_CVT_MAGIC restores I2F
#if !defined(BISBM_NO_CVT_MAGIC) && !defined(BISBM_CVT_MAGIC)
#define BISBM_CVT_MAGIC 1
#endif

#define BISBM_LN2F 0.69314718055994530942f
#define BISBM_LOG2EF 1.44269504088896340736f

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ float f_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float f_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float f_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
#else
inline float f_lg2(float x) { return log2f(x); }
inline float f_ex2(float x) { return exp2f(x); }
inline float f_rcp(float x) { return 1.0f / x; }
#endif

// ---- arithmetic of one move, by type ---------------------------------------------------------
// lg() is the type's native logarithm (natural log for double, log2 on the MUFU unit for float);
// unit() converts lg units to natural-log units, ex() inverts lg().
template <typename R> struct Ar;

// ---- branch-free double log / exp for the move arithmetic -------------------------------------------
// The arguments here are positive, finite and normal (ratios of products of counts; acceptance exponents), so the
// special-case branches of the library routines are not needed -- and without them the three logarithms of one
// move are straight-line code the compiler interleaves.  fdlibm's algorithms (e_log.c / e_exp.c) and constants.
BISBM_HD int32_t dbl_hi(double x) {
#ifdef __CUDA_ARCH__
    return __double2hiint(x);
#else
    uint64_t u; memcpy(&u, &x, 8); return (int32_t)(u >> 32);
#endif
}
BISBM_HD int32_t dbl_lo(double x) {
#ifdef __CUDA_ARCH__
    return __double2loint(x);
#else
    uint64_t u; memcpy(&u, &x, 8); return (int32_t)(uint32_t)u;
#endif
}
BISBM_HD double dbl_make(int32_t hi, int32_t lo) {
#ifdef __CUDA_ARCH__
    return __hiloint2double(hi, lo);
#else
    uint64_t u = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; double x; memcpy(&x, &u, 8); return x;
#endif
}
BISBM_HD double dbl_rcp(double x) {   // x > 0, normal: MUFU.RCP64H (2^-23) + two Newton steps
#ifdef __CUDA_ARCH__
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;
#else
    return 1.0 / x;
#endif
}
// natural logarithm of a positive normal double, < 1 ulp
BISBM_HD double dlog(double x) {
    const int32_t hx = dbl_hi(x);
    const int32_t mant = hx & 0x000fffff;
    const int32_t adj = (mant >= 0x6a09f) ? 1 : 0;                    // mantissa above sqrt(2): halve it
    const int32_t k = (hx >> 20) - 1023 + adj;
    const double m = dbl_make(mant | (0x3ff00000 - (adj << 20)), dbl_lo(x));   // in [sqrt(1/2), sqrt(2))
    const double f = m - 1.0;
    const double s = f * dbl_rcp(2.0 + f);
    const double z = s * s, w = z * z;
    const double t1 = w * fma(w, fma(w, 1.531383769920937332e-01, 2.222219843214978396e-01), 3.999999999940941908e-01);
    const double t2 = z * fma(w, fma(w, fma(w, 1.479819860511658591e-01, 1.818357216161805012e-01), 2.857142874366239149e-01),
                              6.666666666666735130e-01);
    const double R = t1 + t2;
    const double hfsq = 0.5 * f * f;
    const double dk = (double)k;
    // k ln2_hi - ((hfsq - (s (hfsq + R) + k ln2_lo)) - f)
    return fma(dk, 6.93147180369123816490e-01, f - (hfsq - fma(s, hfsq + R, dk * 1.90821492927058770002e-10)));
}
// e^x for |x| <= 700 (clamped), < 1 ulp
BISBM_HD double dexp(double x) {
    x = x < -700.0 ? -700.0 : (x > 700.0 ? 700.0 : x);
    const double magic = 6755399441055744.0;                          // 1.5 * 2^52: rounds to nearest integer
    const double kd = fma(x, 1.44269504088896338700e+00, magic);
    const int32_t k = dbl_lo(kd);
    const double dk = kd - magic;
    double r = fma(dk, -6.93147180369123816490e-01, x);
    r = fma(dk, -1.90821492927058770002e-10, r);
    // e^r on |r| <= ln2 / 2: Taylor to r^13 (next term 4e-18)
    double p = 1.6059043836821613e-10;
    p = fma(p, r, 2.08767569878681e-09);
    p = fma(p, r, 2.505210838544172e-08);
    p = fma(p, r, 2.755731922398589e-07);
    p = fma(p, r, 2.7557319223985893e-06);
    p = fma(p, r, 2.48015873015873e-05);
    p = fma(p, r, 1.984126984126984e-04);
    p = fma(p, r, 1.3888888888888889e-03);
    p = fma(p, r, 8.333333333333333e-03);
    p = fma(p, r, 4.1666666666666664e-02);
    p = fma(p, r, 1.6666666666666666e-01);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    return dbl_make(dbl_hi(p) + (k << 20), dbl_lo(p));                 // p * 2^k (result normal: |x| <= 700)
}

template <> struct Ar<double> {
    static constexpr int FOLD = 32;       // count ratios multiplied between logarithms (32 factors < 2^31 fit a double)
    static constexpr bool SPLIT = true;   // accumulate sum (m+1-c1) inv, sum (m_s+c1) inv, sum c1 inv separately
    BISBM_HD static double unit() { return 1.0; }
    BISBM_HD static double inv_unit() { return 1.0; }
    // exact conversion of a 32-bit unsigned integer: 2^52 + x has x as its low mantissa word
    BISBM_HD static double cvt(uint32_t x) {
#if defined(__CUDA_ARCH__) && defined(BISBM_CVT_MAGIC)
        return __hiloint2double(0x43300000, (int)x) - 4503599627370496.0;
#else
        return (double)x;
#endif
    }
    BISBM_HD static double cvt_small(uint32_t x) { return cvt(x); }
    BISBM_HD static double cvt_small_p1(uint32_t x) {   // x + 1 as a double: the + 1 rides on the constant of the splice
#if defined(__CUDA_ARCH__) && defined(BISBM_CVT_MAGIC)
        return __hiloint2double(0x43300000, (int)x) - 4503599627370495.0;
#else
        return (double)(x + 1u);
#endif
    }
    BISBM_HD static double cvt_s(int x) {
#if defined(__CUDA_ARCH__) && defined(BISBM_CVT_MAGIC)
        return __hiloint2double(0x43300000, (int)((uint32_t)x ^ 0x80000000u)) - 4503601774854144.0;   // 2^52 + 2^31
#else
        return (double)x;
#endif
    }
    BISBM_HD static double rcp(double x) { return dbl_rcp(x); }
    BISBM_HD static double lg(double x) { return dlog(x); }
    BISBM_HD static double ex(double x) { return dexp(x); }
    BISBM_HD static double u01(uint32_t w) { return (cvt(w) + 0.5) * (1.0 / 4294967296.0); }
    // U < x / 2^32 for the 32-bit draw w
    BISBM_HD static bool draw_below(uint32_t w, double x32) { return cvt(w) < x32; }
};

template <> struct Ar<float> {
    static constexpr int FOLD = 4;        // 4 factors < 2^31 stay inside fp32 range
    static constexpr bool SPLIT = false;  // (m - 2c - 1) and m_s are formed exactly before the multiply
    BISBM_HD static float unit() { return BISBM_LN2F; }
    BISBM_HD static float inv_unit() { return BISBM_LOG2EF; }
    BISBM_HD static float cvt(uint32_t x) { return (float)(int)x; }
    BISBM_HD static float cvt_small(uint32_t x) {   // x <= 255: splice under the exponent of 2^23 (no XU-pipe conversion)
#ifdef __CUDA_ARCH__
        return __uint_as_float(0x4B000000u | x) - 8388608.0f;
#else
        return (float)x;
#endif
    }
    BISBM_HD static float cvt_small_p1(uint32_t x) {   // x <= 254
#ifdef __CUDA_ARCH__
        return __uint_as_float(0x4B000000u | x) - 8388607.0f;
#else
        return (float)(x + 1u);
#endif
    }
    BISBM_HD static float cvt_s(int x) { return (float)x; }
    BISBM_HD static float rcp(float x) { return f_rcp(x); }
    BISBM_HD static float lg(float x) { return f_lg2(x); }
    BISBM_HD static float ex(float x) { return f_ex2(x); }
    BISBM_HD static float u01(uint32_t w) { return ((float)(w >> 8) + 0.5f) * (1.0f / 16777216.0f); }
    BISBM_HD static bool draw_below(uint32_t w, float x32) {
#ifdef __CUDA_ARCH__
        return w < __float2uint_rz(x32);     // saturates at 2^32 - 1
#else
        return (double)w < (double)x32;
#endif
    }
};

// running sums of the one-pass evaluation of transition_ratio (header of sweep.cuh): with c1 = c + 1,
//   A = m_rt + 1 - c1 = m_rt - c,  B = m_st + c1 = m_st + 1 + c,  inv = 1 / (e_t + eps K)
//   sA = sum A inv, sB = sum B inv, sC = sum c1 inv   (SPLIT; accu0 = sB - sC + eps w, accu1 = sA - sC + eps w)
//   sA = sum (A - c1) inv, sB = sum (B - c1) inv      (!SPLIT)
//   w = sum inv, num / den = running products of A / B, lg = lg() of the products folded so far
template <typename R> struct MAcc { R sA, sB, sC, w, num, den, lg; };
template <typename R> BISBM_HD void macc_init(MAcc<R>& A) {
    A.sA = (R)0; A.sB = (R)0; A.sC = (R)0; A.w = (R)0; A.num = (R)1; A.den = (R)1; A.lg = (R)0;
}
template <typename R> BISBM_HD void macc_edge(MAcc<R>& A, int m_r, int m_s, uint32_t c, R inv) {   // c = c1 - 1: earlier edges with this label
    const R dC = Ar<R>::cvt_small_p1(c);
    const R dA = Ar<R>::cvt((uint32_t)m_r - c);
    const R dB = Ar<R>::cvt((uint32_t)m_s + c + 1u);
    if (Ar<R>::SPLIT) {
        A.sA = fma(dA, inv, A.sA);
        A.sB = fma(dB, inv, A.sB);
        A.sC = fma(dC, inv, A.sC);
    } else {
        A.sA = fma(dA - dC, inv, A.sA);
        A.sB = fma(dB - dC, inv, A.sB);
    }
    A.w += inv;
    A.num *= dA;
    A.den *= dB;
}
template <typename R> BISBM_HD void macc_fold(MAcc<R>& A) {
    A.lg += Ar<R>::lg(A.num * Ar<R>::rcp(A.den));
    A.num = (R)1; A.den = (R)1;
}

// e_r terms: [lgamma(e_s+d+1) - lgamma(e_s+1)] - [lgamma(e_r+1) - lgamma(e_r-d+1)] by the midpoint
// Euler-Maclaurin difference of sweep.cuh (block_degree_delta); *ok = false (midpoints < 32 d) -> the caller
// takes the Stirling / lgamma form.
template <typename R> BISBM_HD R bdd_fast(int e_r, int e_s, int d, bool* ok) {
    const R D = Ar<R>::cvt_small((uint32_t)d);
    const R cs = Ar<R>::cvt((uint32_t)e_s) + (R)0.5 * (D + (R)1), cr = Ar<R>::cvt((uint32_t)e_r) - (R)0.5 * (D - (R)1);
    *ok = (cs >= (R)32 * D) && (cr >= (R)32 * D);
    const R is = Ar<R>::rcp(cs), ir = Ar<R>::rcp(cr);
    const R is2 = is * is, ir2 = ir * ir, D2 = D * D;
    const R k3 = D * (D2 - (R)1) * (R)(1.0 / 24.0);
    const R k5 = D * (((R)3 * D2 - (R)10) * D2 + (R)7) * (R)(1.0 / 960.0);
    return D * Ar<R>::unit() * Ar<R>::lg(cs * ir) - k3 * (is2 - ir2) - k5 * (is2 * is2 - ir2 * ir2);
}

// log q(e+de, n+dn) - log q(e, n) from the block's second-order expansion (logq_refresh_kernel);
// *ok = false when the block has none or has drifted out of its range
template <typename R> BISBM_HD R logq_fast(const LogqExp& q, int e, int n, int de, int dn, bool* ok) {
    const int x = e - q.e0, y = n - q.n0;
    const int ax = x < 0 ? -x : x, ay = y < 0 ? -y : y, ad = de < 0 ? -de : de;
    const int re = q.e0 >> 4, rn = q.n0 >> 4;
    *ok = (q.valid != 0u) && ax <= re && ay <= rn && ad <= (q.e0 >> 10);   // |de| <= e0/1024: the 4th-order remainder in de stays below 1e-10
    const R dx = Ar<R>::cvt_s(x), dy = Ar<R>::cvt_s(y), De = Ar<R>::cvt_s(de), Dn = Ar<R>::cvt_s(dn);
    return (R)q.fe * De + (R)q.fn * Dn + (R)0.5 * (R)q.fee * (De * De + (R)2 * dx * De) +
           (R)q.fen * (dx * Dn + dy * De + De * Dn) + (R)0.5 * (R)q.fnn * (Dn * Dn + (R)2 * dy * Dn) +
           (R)q.feee * De * ((R)(1.0 / 6.0) * De * De + (R)0.5 * dx * (De + dx));
}

// dS (natural-log units) and the logarithm of the Hastings factor accu1 / accu0 (lg units) of one move, in two steps so
// the kernel can order them around its global loads: move_local needs only the running sums, move_finish adds eta and
// the block terms.
template <typename R> BISBM_HD void move_local(const MAcc<R>& A, uint32_t d, R eps, R* ratio, R* lh) {
    *ratio = A.num * Ar<R>::rcp(A.den);          // prod (m_rt-c)/(m_st+1+c) not yet folded into A.lg
    const R ew = eps * A.w;
    const R a0 = Ar<R>::SPLIT ? A.sB - A.sC : A.sB, a1 = Ar<R>::SPLIT ? A.sA - A.sC : A.sA;
    *lh = (d == 0) ? (R)0 : Ar<R>::lg((a1 + ew) * Ar<R>::rcp(a0 + ew));
}
template <typename R> BISBM_HD R move_lgm(const MAcc<R>& A, R ratio, int eta_r, int eta_s) {
    const R er = Ar<R>::cvt((uint32_t)(eta_r > 0 ? eta_r : 1)), es = Ar<R>::cvt((uint32_t)eta_s + 1u);
    return A.lg + Ar<R>::lg(ratio * (er * Ar<R>::rcp(es)));      // lg( prod * eta_r / (eta_s + 1) )
}
template <typename R>
BISBM_HD void move_finish(const MAcc<R>& A, int eta_r, int eta_s, R bdd, R lqr, R lqs, uint32_t d, R eps, R* dS, R* lh) {
    R ratio;
    move_local<R>(A, d, eps, &ratio, lh);
    *dS = Ar<R>::unit() * move_lgm<R>(A, ratio, eta_r, eta_s) + ((d == 0) ? (R)0 : bdd) + lqr + lqs;
}

// ---- shared-memory layout (byte offsets; every array is a multiple of 16 bytes) ---------------------
//   int32 sM  [KA*KB][32]       m_rs of the group
//   int32 sEo [kown][32]        e_r of the moving type (read / write)
//   int32 sNo [kown][32]        n_r of the moving type (read / write view)
//   int32 sEp [kopp][32]        e_t of the frozen type (read only: constant during a half sweep)
//   R     sInv[kopp][32]        1 / (e_t + eps K)
//   u32   sSmall[ceil(kown/32)][32]   bit b: block b of this lane's chain needs the exact n_r veto
//   uint4 sVtx[S2_VB]           the CTA's prepared vertices {vertex, CSR row offset, degree, degree index}
//   u8x4  hist[warps][ceil(kopp/4)][32]
//   u8    tile[warps][32 edges][32]   neighbour labels of the warp's vertex as they arrive, [edge][chain]
//   ctl   mbarrier (8 bytes) + vertex counter
struct Sweep2Layout { uint32_t oM, oEo, oNo, oEp, oInv, oSmall, oVtx, oHist, oTile, oCtl, total; };
enum { S2_VB = 448, S2_TILE = 32 * 32 };

inline
#ifdef __CUDACC__
__host__ __device__
#endif
Sweep2Layout sweep2_layout(uint32_t KA, uint32_t KB, uint32_t type, uint32_t warps, uint32_t rsize, bool staged = true) {
    const uint32_t kown = type ? KB : KA, kopp = type ? KA : KB;
    Sweep2Layout L;
    uint32_t o = 0;
    L.oM = o; o += staged ? KA * KB * 128u : 0u;        // counts in L2 (staged = false): only the read-only tables,
    L.oEo = o; o += staged ? kown * 128u : 0u;          // the vertex batch, the histograms and the label tiles
    L.oNo = o; o += staged ? kown * 128u : 0u;
    L.oEp = o; o += kopp * 128u;
    L.oInv = o; o += kopp * 32u * rsize;
    L.oSmall = o; o += staged ? ((kown + 31u) / 32u) * 128u : 0u;
    L.oVtx = o; o += (uint32_t)S2_VB * 16u;
    L.oHist = o; o += warps * ((kopp + 3u) / 4u) * 128u;
    L.oTile = o; o += warps * (uint32_t)S2_TILE;
    L.oCtl = o; o += 64u;
    L.total = o;
    return L;
}

#ifdef __CUDACC__

// ---- PTX helpers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t sh_ld_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sh_st_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t sh_ld_u32v(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sh_st_u32v(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint4 sh_ld_v4(uint32_t a) {
    uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v;
}
__device__ __forceinline__ uint32_t sh_atom_add_u32(uint32_t a, uint32_t v) {
    uint32_t o; asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory"); return o;
}
__device__ __forceinline__ int sh_atom_add_s32(uint32_t a, int v) {
    int o; asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory"); return o;
}
template <typename R> __device__ __forceinline__ R sh_ld_real(uint32_t a);
template <> __device__ __forceinline__ double sh_ld_real<double>(uint32_t a) { double v; asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v; }
template <> __device__ __forceinline__ float sh_ld_real<float>(uint32_t a) { float v; asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }

// 0, but only the hardware knows: `x + opaque_zero(y)` makes x's consumers wait for y without changing any value.
// Used to order the arithmetic after the pass: everything that needs only shared memory first, the values loaded
// from global memory (eta, log q expansions) last, so their latency is covered by work instead of a stall.
__device__ __forceinline__ int opaque_zero(double y) { int z; asm("and.b32 %0, %1, 0;" : "=r"(z) : "r"(__double2loint(y))); return z; }
__device__ __forceinline__ int opaque_zero(float y) { int z; asm("and.b32 %0, %1, 0;" : "=r"(z) : "r"(__float_as_int(y))); return z; }

__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t phase) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(mbar), "r"(phase) : "memory");
    } while (!ok);
}
// bulk-async copy global -> shared (completion counted in bytes on the mbarrier); 16-byte aligned, size % 16 == 0
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(mbar) : "memory");
}
// bulk-async reduction shared -> global: dst[i] += src[i] (int32), performed by the L2
__device__ __forceinline__ void bulk_red_add_s32(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.s32 [%0], [%1], %2;"
                 :: "l"(__cvta_generic_to_global(dst)), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_all() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// counts kept in L2 (STAGED = false): every read goes to L2 (ld.global.cg: other SMs update them with reductions)
// `on` == 0 (a padding lane of the last chain group): no request, 0 -- the padding chains' labels are all 0, so their lanes
// of EVERY warp of the group would otherwise ask one L2 slice for the same few lines (measured: a pool of 80 chains ran 4x
// slower than one of 96)
__device__ __forceinline__ int gl_ld(uint64_t base, uint32_t off, uint32_t on) {
    int v;
    asm("{\n\t.reg .u64 a;\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\tcvt.u64.u32 a, %2;\n\tadd.u64 a, a, %1;\n\tmov.s32 %0, 0;\n\t@p ld.global.cg.s32 %0, [a];\n\t}"
        : "=r"(v) : "l"(base), "r"(off), "r"(on));
    return v;
}
__device__ __forceinline__ void gl_red(uint64_t base, uint32_t off, int v) {
    asm volatile("{\n\t.reg .u64 a;\n\tcvt.u64.u32 a, %1;\n\tadd.u64 a, a, %0;\n\tred.global.add.s32 [a], %2;\n\t}" :: "l"(base), "r"(off), "r"(v) : "memory");
}
__device__ __forceinline__ int gl_atom(uint64_t base, uint32_t off, int v) {
    int o; asm volatile("{\n\t.reg .u64 a;\n\tcvt.u64.u32 a, %2;\n\tadd.u64 a, a, %1;\n\tatom.global.add.s32 %0, [a], %3;\n\t}" : "=r"(o) : "l"(base), "r"(off), "r"(v) : "memory"); return o;
}

#ifdef BISBM_ROUND_CLOCKS
// instrumented builds (scripts/round_clocks.py): clock64 cycles of the staged sweep's warps, summed over all launches --
// [0] proposal + pass, [1] dS / accept, [2] commit, [3] waiting at the barrier after the round's reads, [4] waiting at the
// barrier after its commits, [5] vertices, [6] the longest proposal + pass of one vertex, [7] warp-rounds; and per CTA (its
// thread 0): [8] kernel start -> first round (the prologue), [9] last round -> publish done (the epilogue), [10] CTAs
__device__ unsigned long long g_round_clocks[11];
#define RC_DECL() long long rc[5] = {0, 0, 0, 0, 0}, rc_t = 0, rc_v0 = 0, rc_pass_max = 0; unsigned long long rc_n = 0, rc_rounds = 0
#define RC_START() (rc_t = clock64())
#define RC_MARK(ph) do { const long long t_ = clock64(); rc[ph] += t_ - rc_t; rc_t = t_; } while (0)
#define RC_VSTART() (rc_v0 = rc[0], ++rc_rounds)
#define RC_PASS() do { RC_MARK(0); rc_pass_max = max(rc_pass_max, rc[0] - rc_v0); ++rc_n; } while (0)
#define RC_ROUND() (++rc_rounds)
#define RC_PUBLISH(on) do { if (on) {                                                                                  \
        for (int k_ = 0; k_ < 5; ++k_) atomicAdd(&g_round_clocks[k_], (unsigned long long)rc[k_]);                    \
        atomicAdd(&g_round_clocks[5], rc_n); atomicMax(&g_round_clocks[6], (unsigned long long)rc_pass_max);          \
        atomicAdd(&g_round_clocks[7], rc_rounds); } } while (0)
#define RC_CTA_DECL() long long rck_ = clock64()
#define RC_CTA_MARK(slot) do { const long long t_ = clock64();                                                        \
        if (threadIdx.x == 0) atomicAdd(&g_round_clocks[slot], (unsigned long long)(t_ - rck_)); rck_ = t_; } while (0)
#define RC_CTA_RESET() (rck_ = clock64())
#define RC_CTA_END() do { RC_CTA_MARK(9); if (threadIdx.x == 0) atomicAdd(&g_round_clocks[10], 1ull); } while (0)
#else
#define RC_DECL() do {} while (0)
#define RC_START() ((void)0)
#define RC_MARK(ph) ((void)0)
#define RC_VSTART() ((void)0)
#define RC_PASS() ((void)0)
#define RC_ROUND() ((void)0)
#define RC_PUBLISH(on) ((void)0)
#define RC_CTA_DECL() do {} while (0)
#define RC_CTA_MARK(slot) ((void)0)
#define RC_CTA_RESET() ((void)0)
#define RC_CTA_END() ((void)0)
#endif

// the rare double-precision completions, out of line (arguments by value)
__device__ __noinline__ static double slow2_block_degree_delta(int e_r, int e_s, int d) { return block_degree_delta(e_r, e_s, d); }
// log q(e + de, n + dn) - log q(e, n) for a block without a valid expansion (small, or drifted out of its range): the exact
// table below 10001, else the asymptotic formula from its tabulated g(u), lf(u) -- no fixed-point iteration on the device
__device__ __noinline__ static double slow2_logq_delta(const Tables tb, int e, int n, int de, int dn) {
    return log_q_tab(tb, e + de, n + dn) - log_q_tab(tb, e, n);
}

// estimate mode: occupied blocks of the moving type in this lane's view of n_r (the shared view, or the counts in L2).  Out of
// line, like prior_k_delta: only a move that empties or opens a block needs it.
template <bool STAGED>
__device__ __noinline__ static int s2_occupied(uint32_t no_base, uint64_t gnol, uint32_t kown, uint32_t on) {
    int occ = 0;
    for (uint32_t b = 0; b < kown; ++b) occ += ((STAGED ? sh_ld(no_base + b * 128u) : gl_ld(gnol, b * 128u, on)) > 0) ? 1 : 0;
    return occ;
}

// 1/T of global step t; T == 0 is returned as a negative value
__device__ __noinline__ static double slow2_beta(int schedule, float p0, float p1, uint64_t t) {
    const double T = par_temperature(schedule, p0, p1, t);
    return (T == 0.0) ? -1.0 : 1.0 / T;
}

// end of a sliced half sweep: eta of the moving type := S, the buffer its last launch committed into.  S and `prev` (the buffer
// that launch read; null when it read eta itself) are zeroed, so all of the ring is zero between half sweeps (the third buffer
// was zeroed by the last launch).
__global__ void eta_publish_kernel(int32_t* __restrict__ eta, int32_t* __restrict__ S, int32_t* __restrict__ prev, uint32_t n_groups,
                                   uint32_t KK, uint32_t own_off, uint32_t kown, uint32_t W) {
    const uint32_t per = kown * W * 32u;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_groups * per) return;
    const uint32_t g = i / per;
    const size_t j = ((size_t)g * KK + own_off) * W * 32u + (i - g * per);
    eta[j] = S[j];
    S[j] = 0;
    if (prev) prev[j] = 0;
}

// sliced staged launches, after griddepcontrol.wait: this CTA's 1/cpg share (cpg = the group's publishers) of its group's buffer
// work for the launches around this one.  Every publisher adds its whole staged copy into the next base, so the next base gets
// -(cpg - 1) x base where they publish (m_rs, and e_r / n_r of the moving type) and base elsewhere; it was zeroed by the launch
// before.  Out of line: the rounds' register allocation does not see it.
__device__ __noinline__ static void sliced_buffer_work(const SweepParams& P, uint32_t group, uint32_t cta_in_group, uint32_t cpg,
                                                       uint32_t type, uint32_t KA, uint32_t KB, uint32_t kown, uint32_t W) {
    const uint32_t KK = KA + KB;
    const uint32_t t0 = cta_in_group * blockDim.x + threadIdx.x, stride = cpg * blockDim.x;
    const uint32_t nM = KA * KB * 32u, nE = KK * 32u;
    const size_t offM = (size_t)group * KA * KB * GROUP, offE = (size_t)group * KK * GROUP;
    for (uint32_t i = t0; i < nM + 2u * nE; i += stride) {
        const bool in_m = i < nM, in_e = !in_m && i < nM + nE;
        const uint32_t j = in_m ? i : (in_e ? i - nM : i - nM - nE);
        const size_t o = (in_m ? offM : offE) + j;
        const int32_t* const src = in_m ? P.s.m : (in_e ? P.s.e : P.s.nr);
        int32_t* const dst = in_m ? P.m_next : (in_e ? P.e_next : P.nr_next);
        int32_t* const zero = in_m ? P.m_zero : (in_e ? P.e_zero : P.nr_zero);
        const uint32_t slot = j >> 5;
        const bool own = in_m || (type ? slot >= KA : slot < KA);
        const uint32_t a = (uint32_t)__ldcg(src + o);
        const int32_t add = (int32_t)(own ? 0u - (cpg - 1u) * a : a);
        if (add != 0) atomicAdd(dst + o, add);
        zero[o] = 0;
    }
    for (uint32_t i = t0; i < nE; i += stride) P.nr_live_zero[offE + i] = 0;
    // eta of the moving type: the buffer this launch commits into (zeroed by the launch before) also gets what it reads, so it
    // ends as the next launch's eta; the launch after next commits into eta_zero
    const size_t eta_off = (size_t)group * KK * W * GROUP + (size_t)(type ? KA : 0u) * W * 32;
    for (uint32_t i = t0; i < kown * W * 32u; i += stride) {
        const int32_t x = __ldcg(P.eta_read + eta_off + i);
        if (x != 0) atomicAdd(P.eta_commit + eta_off + i, x);
        P.eta_zero[eta_off + i] = 0;
    }
}

// KF > 0: Ka == Kb == KF padded strides and the moving type TYPE fixed at compile time; KF == 0: from SweepParams.
// 512 threads (16 warps x 128 registers), one CTA per SM.  Preconditions (plan_sweep): max degree <= 255 (u8
// histogram bins), K per type <= 256 (u8 labels).
// STAGED = false: K too large for shared memory -- m_rs / e_r / n_r stay in L2 (loads .cg, commits by global reductions,
// every CTA sees every committed move at once: no slices, no staging, no publish, warps take vertices from a shared counter);
// the rest of the kernel is the same.
template <typename R, int KF, int TYPE, bool STAGED = true, int NT = 512>
__global__ void __launch_bounds__(NT, 1) sweep2_kernel(const __grid_constant__ SweepParams P) {
    typedef Ar<R> AR;
    // staged counts always run in fixed rounds: the warps of a CTA take the vertices of a batch in turn (warp w: w,
    // w + warps_used, ..), every warp of a round evaluates its move against the counts left by the rounds before, then all commit: the counts a move
    // sees do not depend on timing, so a call's result is a function of its inputs -- except where a block of a chain is
    // small enough to empty within the launch: the "would empty block r" veto below is an atomic decrement-and-check whose
    // order among the moves out of r (other warps' in the commit phase, other CTAs' on nr_live) is not fixed
    RC_CTA_DECL();
    extern __shared__ __align__(128) unsigned char s2_smem[];
    unsigned char* const smem_raw = s2_smem;
    constexpr uint32_t FULL = 0xffffffffu;
    uint32_t lane, warp;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(warp));
    warp >>= 5;
    const uint32_t wpc = blockDim.x >> 5;
    const GraphView& G = P.g;
    const uint32_t type = KF ? (uint32_t)TYPE : P.type;
    const uint32_t C = P.s.C, KB = KF ? (uint32_t)KF : P.s.KB, KA = KF ? (uint32_t)KF : P.s.KA, W = P.s.W, KK = KA + KB;
    const uint32_t kown_max = type ? KB : KA, kopp_max = type ? KA : KB;
    // consecutive CTAs -> consecutive groups; spare-SM CTAs come after the regular ones: extra CTA j of launch l takes slot
    // l extras + j, i.e. group (slot mod n_groups)
    const uint32_t cta = blockIdx.x;
    const bool extra_cta = P.extras != 0u && cta >= P.n_groups * P.ctas_per_group;
    const uint32_t slot0 = (uint32_t)(((uint64_t)P.launch_idx * P.extras) % P.n_groups);
    const uint32_t grp0 = extra_cta ? (slot0 + (cta - P.n_groups * P.ctas_per_group)) % P.n_groups : cta % P.n_groups;
    const uint32_t group = P.group_offset + grp0;
    const uint32_t cta_in_group = extra_cta ? P.ctas_per_group : cta / P.n_groups;
    const uint32_t own_off = type ? KA : 0, opp_off = type ? 0 : KA;

    int32_t* const gM = P.s.m + (size_t)group * KA * KB * GROUP;
    int32_t* const gE = P.s.e + (size_t)group * KK * GROUP;
    int32_t* const gNR = P.s.nr + (size_t)group * KK * GROUP;
    int32_t* const gLIVE = P.nr_live + (size_t)group * KK * GROUP + (size_t)own_off * 32;
    const size_t eta_off = (size_t)group * KK * W * GROUP + (size_t)own_off * W * 32;
    int32_t* const gETA = P.eta_commit + eta_off;
    const int32_t* const gETAr = P.eta_read + eta_off;
    const LogqExp* const gLQ = P.lq + ((size_t)group * KK + own_off) * GROUP;

    const uint32_t c = group * 32 + lane;
    const bool live = (c < P.n_chains) && P.active[c];
    const uint32_t cc = (c < P.s.C) ? c : 0;
    const uint32_t ka = P.s.ka[cc], kb = P.s.kb[cc], K = ka + kb;
    const uint32_t kown = type ? kb : ka;
    const R eps = (R)P.s.eps;
    const R epsK32 = (R)(P.s.eps * (double)K * 4294967296.0);   // threshold scale of the uniform-vs-categorical test

    const Sweep2Layout L = sweep2_layout(KA, KB, type, wpc, (uint32_t)sizeof(R), STAGED);
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem_raw);
    int32_t* const sM = reinterpret_cast<int32_t*>(smem_raw + L.oM);
    int32_t* const sEo = reinterpret_cast<int32_t*>(smem_raw + L.oEo);
    int32_t* const sNo = reinterpret_cast<int32_t*>(smem_raw + L.oNo);
    int32_t* const sEp = reinterpret_cast<int32_t*>(smem_raw + L.oEp);
    R* const sInv = reinterpret_cast<R*>(smem_raw + L.oInv);
    uint32_t* const sSmall = reinterpret_cast<uint32_t*>(smem_raw + L.oSmall);
    uint4* const sVtx = reinterpret_cast<uint4*>(smem_raw + L.oVtx);
    uint32_t* const sCtr = reinterpret_cast<uint32_t*>(smem_raw + L.oCtl + 16);
    const uint32_t mbar = sbase + L.oCtl;
    const uint32_t hist_words = (kopp_max + 3u) / 4u;

    // Sliced staged launches run under programmatic dependent launch: until griddepcontrol.wait (a no-op in any other launch)
    // the launch before may still be running, so only what depends on no earlier launch goes first -- the mbarrier, the
    // histograms and the first vertex batch (Feistel map and graph only).
    if (STAGED && threadIdx.x == 0) {
        mbar_init(mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {
        uint32_t* const hw = reinterpret_cast<uint32_t*>(smem_raw + L.oHist);
        for (uint32_t i = threadIdx.x; i < wpc * hist_words * 32u; i += blockDim.x) hw[i] = 0u;
    }

    // ---- the CTA's share of the slice: positions pos_begin + cta + j * ctas_per_group, j < cnt ----
    const uint32_t nv = type ? G.nb : G.na, v0 = type ? G.na : 0;
    uint32_t cpg = P.ctas_per_group;                                     // CTAs of the group that take vertices
    uint32_t pos_begin = P.pos_begin, pos_end = P.pos_end;
    if (P.extras != 0u) {
        // this group's slice: it has advanced by per_cta x (ctas_per_group per launch + one per extra slot it was handed so far)
        const uint64_t s0 = (uint64_t)P.launch_idx * P.extras;
        const uint32_t before = (uint32_t)((s0 + P.n_groups - 1u - grp0) / P.n_groups);
        const bool has_extra = (grp0 + P.n_groups - slot0) % P.n_groups < P.extras;
        cpg += has_extra ? 1u : 0u;
        const uint64_t pb = ((uint64_t)P.launch_idx * P.ctas_per_group + before) * P.per_cta;
        pos_begin = (uint32_t)min(pb, (uint64_t)nv);
        pos_end = (uint32_t)min(pb + (uint64_t)cpg * P.per_cta, (uint64_t)nv);
    }
    const uint32_t span = pos_end - pos_begin;
    const uint32_t cnt = P.kat_mode ? (cta_in_group == 0u ? 1u : 0u)
                                    : ((cta_in_group < cpg && span > cta_in_group) ? (span - cta_in_group + cpg - 1u) / cpg : 0u);
    const uint64_t pkey = (P.sweep * 2 + type) * 0x9E3779B97F4A7C15ull + (uint64_t)group * 0xD1B54A32D192ED03ull;
    auto prepare = [&](uint32_t j0) -> uint32_t {   // entries j0 .. j0 + nb - 1 into sVtx; all threads
        const uint32_t nb = (cnt > j0) ? min((uint32_t)S2_VB, cnt - j0) : 0u;
        for (uint32_t i = threadIdx.x; i < nb; i += blockDim.x) {
            uint4 b;
            if (P.kat_mode) b.x = P.kat_v;
            else b.x = v0 + feistel_perm(pos_begin + cta_in_group + (j0 + i) * cpg, nv, P.half_bits, pkey);
            b.y = __ldcg(G.row_ptr + b.x);          // (.cg: nothing of the graph is reused through L1, which holds the log q expansions)
            b.z = __ldcg(G.row_ptr + b.x + 1) - b.y;
            b.w = __ldcg(G.degidx + b.x);
            sVtx[i] = b;
        }
        if (threadIdx.x == 0) *sCtr = 0u;
        return nb;
    };
    uint32_t nb = prepare(0);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    __syncthreads();
    // ---- stage the group's counts: one thread, bulk-async copies ----
    if (STAGED) {
        if (threadIdx.x == 0) {
            const uint32_t bM = KA * KB * 128u, bO = kown_max * 128u, bP = kopp_max * 128u;
            mbar_expect_tx(mbar, bM + 2u * bO + bP);
            for (uint32_t off = 0; off < bM; off += 32768u)
                bulk_g2s(sbase + L.oM + off, reinterpret_cast<const char*>(gM) + off, min(32768u, bM - off), mbar);
            bulk_g2s(sbase + L.oEo, gE + own_off * 32, bO, mbar);
            bulk_g2s(sbase + L.oNo, gNR + own_off * 32, bO, mbar);
            bulk_g2s(sbase + L.oEp, gE + opp_off * 32, bP, mbar);
        }
    } else {
        for (uint32_t i = threadIdx.x; i < kopp_max * 32u; i += blockDim.x) sEp[i] = __ldcg(gE + opp_off * 32 + i);
    }
    if (STAGED && !P.exclusive && !P.kat_mode) sliced_buffer_work(P, group, cta_in_group, cpg, type, KA, KB, kown_max, W);
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (STAGED) mbar_wait(mbar, 0);
    __syncthreads();
    // tables derived from the staged counts
    for (uint32_t i = threadIdx.x; i < kopp_max * 32u; i += blockDim.x) {
        const uint32_t ci = min(group * 32u + (i & 31u), C - 1u);
        const double Kc = (double)(P.s.ka[ci] + P.s.kb[ci]);
        sInv[i] = (R)(1.0 / ((double)sEp[i] + P.s.eps * Kc));
    }
    if (STAGED) {
        // a block is "small" when it could empty within this launch without this CTA noticing: only then the veto
        // needs an exact counter.  One CTA per group: the shared view is exact, every block takes the exact path.
        const int thresh = P.exclusive ? 0x7fffffff : (int)min(span, 0x7ffffff0u) + 1;
        const uint32_t words = (kown_max + 31u) / 32u;
        for (uint32_t i = threadIdx.x; i < words * 32u; i += blockDim.x) {
            const uint32_t w = i >> 5, l = i & 31u;
            uint32_t bits = 0;
            for (uint32_t b = 0; b < 32u && w * 32u + b < kown_max; ++b)
                if (sNo[(w * 32u + b) * 32u + l] <= thresh) bits |= 1u << b;
            sSmall[i] = bits;
        }
    }
    __syncthreads();

    // estimate mode: occupied blocks of the frozen type of this lane's chain (the moving type's are counted where a move
    // needs them, from the same view as its n_r)
    int occ_opp = 0;
    if (P.vary_k)
        for (uint32_t b = 0; b < kopp_max; ++b) occ_opp += (__ldcg(gNR + (opp_off + b) * 32 + lane) > 0) ? 1 : 0;

    // lane-private shared byte addresses (entry j of this chain at +j*128)
    const uint32_t lane4 = lane * 4u;
    const uint32_t M_base = sbase + L.oM + lane4;
    const uint32_t Eo_base = sbase + L.oEo + lane4;
    const uint32_t No_base = sbase + L.oNo + lane4;
    const uint32_t Ep_base = sbase + L.oEp + lane4;
    const uint32_t Inv_base = sbase + L.oInv + lane * (uint32_t)sizeof(R);
    constexpr uint32_t IS = 32u * (uint32_t)sizeof(R);             // bytes between inv entries of one lane
    const uint32_t Small_base = sbase + L.oSmall + lane4;
    const uint32_t hist_base = sbase + L.oHist + warp * hist_words * 128u + lane4;
    const uint32_t tile_w = sbase + L.oTile + warp * (uint32_t)S2_TILE;
    // the tile keeps the rows as they arrive, [edge][chain]: one 8-byte store per lane and block of 8 rows, one byte load per edge
    const uint32_t tile_lane = tile_w + lane;                                      // this chain's labels, edge e at + 32 e
    const uint32_t tile_st = tile_w + (lane >> 2) * 32u + (lane & 3u) * 8u;        // store base: row lane/4 (+ 8 j), chains 8 (lane%4) ..
    constexpr uint32_t TE = 32u;                                                   // bytes between consecutive edges of one chain
    // m(x_own, t_opp) at byte offset x*SX + t*ST of this lane's view of m_rs
    const uint32_t SX = (type ? 1u : KB) * 128u, ST = (type ? KB : 1u) * 128u;
    // count accessors: shared-memory views (STAGED) or the arrays in L2
    const uint64_t gMl = (uint64_t)__cvta_generic_to_global(gM + lane);
    const uint64_t gEol = (uint64_t)__cvta_generic_to_global(gE + own_off * 32 + lane);
    const uint64_t gNol = (uint64_t)__cvta_generic_to_global(gNR + own_off * 32 + lane);
    const uint32_t live_u = live ? 1u : 0u;
    auto m_ld = [&](uint32_t off) -> int {
        if constexpr (STAGED) return sh_ld(M_base + off); else return gl_ld(gMl, off, live_u);
    };
    auto m_red = [&](uint32_t off, int v) {
        if constexpr (STAGED) sh_red_add(M_base + off, v); else gl_red(gMl, off, v);
    };
    auto eo_ld = [&](uint32_t blk) -> int { if constexpr (STAGED) return sh_ld(Eo_base + blk * 128u); else return gl_ld(gEol, blk * 128u, live_u); };
    auto eo_red = [&](uint32_t blk, int v) { if constexpr (STAGED) sh_red_add(Eo_base + blk * 128u, v); else gl_red(gEol, blk * 128u, v); };
    auto no_ld = [&](uint32_t blk) -> int { if constexpr (STAGED) return sh_ld(No_base + blk * 128u); else return gl_ld(gNol, blk * 128u, live_u); };
    auto no_red = [&](uint32_t blk, int v) { if constexpr (STAGED) sh_red_add(No_base + blk * 128u, v); else gl_red(gNol, blk * 128u, v); };
    // counts in L2: a warp evaluates one move of a chain at a time, so about as many moves of one chain are in flight as its
    // group has warps (round 2 used the constant 8192 = 3.5 x the warps of a whole B200); with a four-fold margin for short
    // vertices finishing inside a long one's window, a block with more nodes than that cannot empty between the read of n_r and
    // the commit, and smaller blocks take the exact atomic
    const int SAFE_NR = (int)(4u * (P.ctas_per_group + 1u) * wpc);
    // the group's label rows: chain-minor u8, 32 bytes per vertex and group
    uint64_t LAB8 = (uint64_t)__cvta_generic_to_global(P.lab8 + (size_t)(group * 32u < C ? group * 32u : 0u));
    asm volatile("" : "+l"(LAB8));
    const uint32_t key0 = (uint32_t)P.seeds[cc], key1 = (uint32_t)(P.seeds[cc] >> 32);
    const bool const_T = (P.schedule == 3) || P.beta_chain;
    const R beta_lane = P.beta_chain ? (R)P.beta_chain[cc] : (R)P.beta0;   // parallel tempering: this chain's rung
    const bool movable_chain = live && (kown != 1);
    const uint32_t kat_lane = P.kat_mode ? (P.kat_chain & 31u) : 32u;

    uint32_t n_acc = 0;
    double ds_sum = 0.0;

    // neighbour label rows of a vertex: lane l loads 8 bytes (chains 8 (l%4) ..) of row l/4 + 8 j, j = 0..3
    uint32_t ids[4];
    uint2 rows[4];
    auto load_ids = [&](uint32_t row0, uint32_t dcnt) {       // dcnt <= 32 neighbours starting at CSR offset row0
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t rho = (lane >> 2) + 8u * j;
            ids[j] = 0u;
            if (rho < dcnt) asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(ids[j]) : "l"(__cvta_generic_to_global(G.col + row0 + rho)));
        }
    };
    auto load_rows = [&](uint32_t dcnt) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t rho = (lane >> 2) + 8u * j;
            rows[j].x = 0u; rows[j].y = 0u;
            if (rho < dcnt)
                asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %2, %3, %4;\n\tld.global.cg.v2.u32 {%0, %1}, [a];\n\t}"
                             : "=r"(rows[j].x), "=r"(rows[j].y) : "r"(ids[j]), "r"(C), "l"(LAB8 + (uint64_t)((lane & 3u) * 8u)));
        }
    };
    auto store_tile = [&](uint32_t dcnt) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (8u * j < dcnt) {
                asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(tile_st + 256u * j), "r"(rows[j].x), "r"(rows[j].y) : "memory");
            }
        }
    };
    auto lab_ld = [&](uint32_t vtx) -> uint32_t {     // label of vertex vtx in this lane's chain
        uint32_t x;
        asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %1, %2, %3;\n\tld.global.cg.u8 %0, [a];\n\t}" : "=r"(x) : "r"(vtx), "r"(C), "l"(LAB8 + (uint64_t)lane));
        return x;
    };
    auto lab_st = [&](uint32_t vtx, uint32_t x) {
        asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %0, %1, %2;\n\tst.global.u8 [a], %3;\n\t}" :: "r"(vtx), "r"(C), "l"(LAB8 + (uint64_t)lane), "r"(x) : "memory");
    };
    RC_DECL();
    RC_CTA_MARK(8);
    uint32_t ticket = warp;                               // STAGED: this warp's next vertex of the batch
    auto pop = [&]() -> uint32_t {
        if constexpr (STAGED) { const uint32_t i = ticket; ticket += P.warps_used; return i; }
        uint32_t i = 0;
        if (lane == 0) i = atomicAdd(sCtr, 1u);
        return __shfl_sync(FULL, i, 0);
    };
    const uint32_t round_threads = P.warps_used * 32u;
    auto round_barrier = [&]() {                          // STAGED: the warps that take vertices
        if constexpr (STAGED) asm volatile("bar.sync 1, %0;" :: "r"(round_threads) : "memory");
    };

    for (uint32_t j0 = 0;;) {
        if (warp < P.warps_used) {
            ticket = warp;
            uint32_t rounds = 0;
            RC_START();
            // pipeline: while vertex k is evaluated, the rows and the own label of vertex k+1 are in flight
            uint32_t nxt = pop();
            uint4 ninfo = make_uint4(0, 0, 0, 0);
            uint32_t r_nxt = 0;
            if (nxt < nb) {
                ninfo = sVtx[nxt];
                load_ids(ninfo.y, min(ninfo.z, 32u));
                load_rows(min(ninfo.z, 32u));
                r_nxt = lab_ld(ninfo.x);
            }
            while (nxt < nb) {
                ++rounds;
                RC_VSTART();
                const uint4 cur = ninfo;
                uint32_t v = cur.x;
                const uint32_t d = cur.z, didx = cur.w, r = r_nxt;
                const uint32_t pos_index = j0 + nxt;      // this vertex's index within the CTA's share
                __syncwarp();
                store_tile(min(d, 32u));
                asm volatile("" : "+r"(v));               // the draw (pure ALU on v) goes AFTER the tile stores: it covers their drain
                __syncwarp();
                // next vertex: ids now, rows after the pass (when the ids have arrived)
                nxt = pop();
                if (nxt < nb) {
                    ninfo = sVtx[nxt];
                    load_ids(ninfo.y, min(ninfo.z, 32u));
                }
                const uint32_t d_n = (nxt < nb) ? min(ninfo.z, 32u) : 0u;
                auto issue_next = [&]() {
                    if (nxt < nb) { load_rows(d_n); r_nxt = lab_ld(ninfo.x); }
                };
                auto load_q = [&](uint32_t slot) -> LogqExp {   // 48 bytes of this (block, chain); constant during the launch
                    const uint4* p = reinterpret_cast<const uint4*>(gLQ + slot * 32u + lane);
                    const uint4 a = __ldg(p), b = __ldg(p + 1), c4 = __ldg(p + 2);
                    LogqExp q;
                    q.e0 = (int)a.x; q.n0 = (int)a.y; q.fe = __hiloint2double((int)a.w, (int)a.z);
                    q.fn = __hiloint2double((int)b.y, (int)b.x);
                    q.fee = __uint_as_float(b.z); q.fen = __uint_as_float(b.w);
                    q.fnn = __uint_as_float(c4.x); q.feee = __uint_as_float(c4.y); q.valid = c4.z; q.pad = 0;
                    return q;
                };

                // ---- the draw of this move: Philox4x32-10, counter = (vertex, sweep, chain seed), pool-wide key ----
                u32x4 ctr; ctr.x = v; ctr.y = (uint32_t)P.sweep; ctr.z = key0; ctr.w = key1;
                const u32x4 ra = philox4x32(ctr, (uint32_t)(P.sweep >> 32) ^ 0xA4093822u, 0x299F31D0u);
                const uint32_t ry = ra.y, rz = ra.z, rw = ra.w;
                // the proposal's random neighbour (differs per lane): its label is in the tile
                uint32_t tq = 0;
                if (d != 0u) {
                    const uint32_t e = mulhi32(ra.x, d);
                    if (d <= 32u) tq = sh_ld_u8(tile_lane + e * TE);
                    else tq = (e < 32u) ? sh_ld_u8(tile_lane + e * TE) : lab_ld(__ldcg(G.col + cur.y + e));
                }
                tq = min(tq, kopp_max - 1u);
                R beta = beta_lane;
                if (!const_T) {
                    const uint64_t step = P.step_base + pos_begin + cta_in_group + (uint64_t)pos_index * cpg;
                    // abrupt_cool in line (a launch that straddles the switch; whole launches on one side arrive as constant T)
                    if (P.schedule == 4) beta = ((float)step < P.p0) ? (R)1 : (R)-1;
                    else beta = (R)slow2_beta(P.schedule, P.p0, P.p1, step);
                }
                const bool T_zero = beta < (R)0;

                // ---- proposal (single_vertex_change), branch-free ----
                const int e_t = sh_ld(Ep_base + tq * 128u);
                const R inv_t = sh_ld_real<R>(Inv_base + tq * IS);
                // U < eps K / (e_t + eps K), both sides scaled by 2^32
                const bool uniform_pick = (d == 0u) || AR::draw_below(ry, epsK32 * inv_t);
                const uint32_t sg = mulhi32(rz, K);      // uniform over ALL K blocks (either type)
                const bool sg_a = sg < ka;
                const uint32_t s_uni = sg_a ? sg : sg - ka;
                // categorical over row m[t][.]: s = #{x : cum_x <= z}; wz tracks cum - z - 1 (negative while cum <= z)
                int wz = -(int)mulhi32(rz, (uint32_t)e_t) - 1;
                uint32_t cnt_le = 0;
                {
                    uint32_t a = tq * ST;
#pragma unroll 8
                    for (uint32_t x = 0; x < kown_max; ++x, a += SX) {   // uniform bound; blocks >= kown hold 0
                        wz += m_ld(a);
                        cnt_le += ((uint32_t)wz) >> 31;
                    }
                }
                const uint32_t s_cat = cnt_le < kown ? cnt_le : kown - 1;
                // a uniform draw that falls on a block of the other type is rejected (dS = +inf): s stays r for it
                bool cross = movable_chain && uniform_pick && (sg_a != (type == 0));
                uint32_t s = (movable_chain && !cross) ? (uniform_pick ? s_uni : s_cat) : r;   // own-type local index
                if (P.kat_mode) { cross = false; s = (lane == kat_lane) ? P.kat_s : r; }
                const bool eval = live && (s != r);
                const int n_r = no_ld(r);
                if (!__any_sync(FULL, eval)) {
                    // s == r (dS = 0, accu_r = 1): accepted at T > 0 unless the block would empty, rejected at T == 0
                    // (src/metropolis_hasting.cc:47-52)
                    if (live && !cross && !T_zero && n_r != 1 && !P.kat_mode) ++n_acc;
                    issue_next();
                    RC_PASS();
                    round_barrier();
                    RC_MARK(3);
                    round_barrier();
                    RC_MARK(4);
                    continue;
                }
                // eta of the move is requested before the pass: the pass's shared-memory round trips cover its L2 latency, which
                // dS would otherwise wait for (+5.6 % on the C3 bench, profiles/r05_eta_early_ab.txt).  The staged form commits
                // only between the round's barriers, so these are the values a read after the pass would see; the counts-in-L2
                // form reads eta live and keeps the read after the pass
                int eta_r = 0, eta_s = 0;
                if constexpr (STAGED) {
                    eta_r = ldc(&gETAr[(r * W + didx) * 32 + lane]);
                    eta_s = ldc(&gETAr[(s * W + didx) * 32 + lane]);
                }

                // ---- one pass over v's neighbours: dS and the Hastings factor (transition_ratio).  Every lane
                //      runs it (masked lanes cost the same issue slots); only `eval` lanes may commit. ----
                MAcc<R> A; macc_init(A);
                const uint32_t Mr = r * SX, Ms = s * SX;
                // histogram bin of label t: word t / 4, byte t % 4 -- or, with exactly 8 words (the Ka = Kb = 32 instantiation),
                // word t % 8, byte t / 8: the byte's shift is then t & 0x18, one instruction less per edge
                auto h_sh = [&](uint32_t t) -> uint32_t { if constexpr (KF == 32) return t & 0x18u; else return (t & 3u) << 3; };
                auto h_ad = [&](uint32_t t) -> uint32_t { if constexpr (KF == 32) return hist_base + ((t & 7u) << 7); else return hist_base + ((t >> 2) << 7); };
                auto edge1 = [&](uint32_t t) {
                    const uint32_t sh3 = h_sh(t);
                    const uint32_t old = sh_atom_add_u32(h_ad(t), 1u << sh3);
                    const uint32_t off = t * ST;
                    const int m_r = m_ld(Mr + off), m_s = m_ld(Ms + off);
                    const R inv = sh_ld_real<R>(Inv_base + t * IS);
                    macc_edge(A, m_r, m_s, (old >> sh3) & 0xffu, inv);
                };
                auto edge4t = [&](uint32_t t0, uint32_t t1, uint32_t t2, uint32_t t3) {
                    const uint32_t h0 = h_sh(t0), h1 = h_sh(t1), h2 = h_sh(t2), h3 = h_sh(t3);
                    // the four histogram updates in edge order (a repeated label must see the earlier increment)
                    const uint32_t o0 = sh_atom_add_u32(h_ad(t0), 1u << h0);
                    const uint32_t o1 = sh_atom_add_u32(h_ad(t1), 1u << h1);
                    const uint32_t o2 = sh_atom_add_u32(h_ad(t2), 1u << h2);
                    const uint32_t o3 = sh_atom_add_u32(h_ad(t3), 1u << h3);
                    const uint32_t f0 = t0 * ST, f1 = t1 * ST, f2 = t2 * ST, f3 = t3 * ST;
                    const int r0 = m_ld(Mr + f0), s0 = m_ld(Ms + f0), r1 = m_ld(Mr + f1), s1 = m_ld(Ms + f1);
                    const int r2 = m_ld(Mr + f2), s2 = m_ld(Ms + f2), r3 = m_ld(Mr + f3), s3 = m_ld(Ms + f3);
                    const R i0 = sh_ld_real<R>(Inv_base + t0 * IS), i1 = sh_ld_real<R>(Inv_base + t1 * IS);
                    const R i2 = sh_ld_real<R>(Inv_base + t2 * IS), i3 = sh_ld_real<R>(Inv_base + t3 * IS);
                    macc_edge(A, r0, s0, (o0 >> h0) & 0xffu, i0);
                    macc_edge(A, r1, s1, (o1 >> h1) & 0xffu, i1);
                    macc_edge(A, r2, s2, (o2 >> h2) & 0xffu, i2);
                    macc_edge(A, r3, s3, (o3 >> h3) & 0xffu, i3);
                };
                for (uint32_t e0 = 0; e0 < d; e0 += 32u) {
                    const uint32_t nrem = min(32u, d - e0);
                    if (e0) {   // hubs: later blocks of 32 neighbours are fetched in place
                        __syncwarp();
                        uint32_t keep_ids[4];    // ids[] holds the NEXT vertex's neighbours; rows[] is free (already in the tile)
#pragma unroll
                        for (int j = 0; j < 4; ++j) keep_ids[j] = ids[j];
                        load_ids(cur.y + e0, nrem);
                        load_rows(nrem);
                        store_tile(nrem);
#pragma unroll
                        for (int j = 0; j < 4; ++j) ids[j] = keep_ids[j];
                        __syncwarp();
                        if (AR::FOLD >= 32) macc_fold(A);
                    }
                    const uint32_t nfull = nrem >> 2, tail = nrem & 3u;
                    {
                        uint32_t ta = tile_lane;
                        for (uint32_t q = 0; q < nfull; ++q, ta += 128u) {
                            const uint32_t t0 = sh_ld_u8(ta), t1 = sh_ld_u8(ta + 32u), t2 = sh_ld_u8(ta + 64u), t3 = sh_ld_u8(ta + 96u);
                            edge4t(t0, t1, t2, t3);
                            if (AR::FOLD < 32) macc_fold(A);
                        }
                        if (tail) {
                            edge1(sh_ld_u8(ta));
                            if (tail > 1u) edge1(sh_ld_u8(ta + 32u));
                            if (tail > 2u) edge1(sh_ld_u8(ta + 64u));
                            if (AR::FOLD < 32) macc_fold(A);
                        }
                    }
                }
                issue_next();
                __syncwarp();
                RC_PASS();

                // ---- dS, accept (step) ----
                bool go;
                R dS;
                // what stays in global memory -- the two log q expansions (read only) and, where it was not requested before the
                // pass, eta (L2, updated by atomics) -- is requested first; the e_r terms below only need shared memory and cover
                // part of the latency
                if constexpr (!STAGED) {
                    eta_r = ldc(&gETAr[(r * W + didx) * 32 + lane]);
                    eta_s = ldc(&gETAr[(s * W + didx) * 32 + lane]);
                }
                const int n_s = no_ld(s);
                {
                    const int e_r = eo_ld(r), e_s = eo_ld(s);
                    bool ok_b, ok_r, ok_s;
                    LogqExp q_r = load_q(r), q_s = load_q(s);
                    // (1) shared memory only: the e_r terms, the Hastings factor, the count-ratio product
                    R bdd = bdd_fast<R>(e_r, e_s, (int)d, &ok_b);
                    R ratio, lh;
                    move_local<R>(A, d, eps, &ratio, &lh);
                    // (2) the log q expansions (L1 / L2), gated behind the two logarithms above
                    const int z1 = opaque_zero(bdd) | opaque_zero(lh);
                    q_r.e0 += z1; q_s.e0 += z1;
                    R lqr = logq_fast<R>(q_r, e_r, n_r, -(int)d, -1, &ok_r);
                    R lqs = logq_fast<R>(q_s, e_s, n_s, (int)d, 1, &ok_s);
                    // (3) eta (L2, the longest wait) last: log( prod * eta_r / (eta_s + 1) )
                    const int z2 = opaque_zero(lqr) | opaque_zero(lqs) | opaque_zero(ratio);
                    const R lgm = move_lgm<R>(A, ratio, eta_r + z2, eta_s + z2);
                    if (__any_sync(FULL, eval && !(ok_b && ok_r && ok_s))) {
                        if (eval && !ok_b) bdd = (R)slow2_block_degree_delta(e_r, e_s, (int)d);
                        if (eval && !ok_r) lqr = (R)slow2_logq_delta(P.tb, e_r, n_r, -(int)d, -1);
                        if (eval && !ok_s) lqs = (R)slow2_logq_delta(P.tb, e_s, n_s, (int)d, 1);
                        __syncwarp();
                    }
                    dS = AR::unit() * lgm + ((d == 0u) ? (R)0 : bdd) + lqr + lqs;
                    if (P.vary_k) {
                        // the move empties r and / or opens s: the K-dependent prior terms change with the occupied count, read
                        // from the view n_r came from (every round's commits of this CTA, not only this warp's)
                        const int dk = ((n_s == 0) ? 1 : 0) - ((n_r == 1) ? 1 : 0);
                        if (__any_sync(FULL, eval && dk != 0)) {
                            if (eval && dk != 0) {
                                const int occ_own = s2_occupied<STAGED>(No_base, gNol, kown, live_u);
                                dS += (R)prior_k_delta((double)G.n_edges, (double)nv, (double)occ_own, (double)occ_opp, dk);
                            }
                            __syncwarp();
                        }
                    }
                    const R a2 = lh - dS * (beta * AR::inv_unit());          // lg of the acceptance ratio
                    const bool go_hot = (a2 > (R)0) || (AR::u01(rw) < AR::ex(a2));
                    go = eval && (T_zero ? (dS < (R)0) : go_hot);
                    if (P.kat_mode) {
                        if (lane == kat_lane && eval) { P.kat_out[0] = (double)dS; P.kat_out[1] = (double)(lh * AR::unit()); }
                        go = false;
                    }
                    // s == r: see above
                    if (live && !cross && s == r && !T_zero && n_r != 1 && !P.kat_mode) ++n_acc;
                    RC_MARK(1);
                    round_barrier();                         // every warp of the round has read its counts
                    RC_MARK(3);
                    if (go && P.vary_k) {
                        no_red(r, -1);                       // estimate mode: a block may empty
                    } else if (go) {
                        // the "would empty block r" veto of apply_mcmc_moves: exact where it can matter
                        if constexpr (STAGED) {
                            const uint32_t small_r = (sh_ld_u32v(Small_base + (r >> 5) * 128u) >> (r & 31u)) & 1u;
                            if (small_r) {
                                if (P.exclusive) {
                                    const int old = sh_atom_add_s32(No_base + r * 128u, -1);
                                    if (old <= 1) { sh_red_add(No_base + r * 128u, 1); go = false; }
                                } else {
                                    // n_r at the start of the launch + the decrements before this one (the base is read-only
                                    // during the launch)
                                    const int old = atomicSub(&gLIVE[r * 32 + lane], 1) +
                                                    ldc(P.s.nr + ((size_t)group * KK + own_off + r) * GROUP + lane);
                                    if (old <= 1) { atomicAdd(&gLIVE[r * 32 + lane], 1); go = false; }
                                    else sh_red_add(No_base + r * 128u, -1);
                                }
                            } else {
                                sh_red_add(No_base + r * 128u, -1);
                            }
                        } else {
                            // n_r was read from L2 a moment ago; fewer than SAFE_NR moves of this chain can be in flight, so a
                            // block that large cannot empty and a fire-and-forget reduction is enough
                            if (n_r > SAFE_NR) no_red(r, -1);
                            else {
                                const int old = gl_atom(gNol, r * 128u, -1);
                                if (old <= 1) { no_red(r, 1); go = false; }
                            }
                        }
                    }
                }
                __syncwarp();

                // ---- commit (apply_mcmc_moves) and clear the histogram ----
                const bool any_go = __any_sync(FULL, go);
                if (d <= 32u) {
                    // walk the edges again: m(r,t) -= 1, m(s,t) += 1 for the lanes that move.  Shared-memory counts: every lane
                    // runs the walk (a reduction of 0 costs nothing extra); counts in L2: only the lanes that move issue reductions
                    if (any_go && (STAGED || go)) {
                        const int g1 = go ? 1 : 0;
                        const uint32_t dMs = Ms - Mr;          // m(s,t) sits at a fixed distance from m(r,t)
                        auto move1 = [&](uint32_t t) { const uint32_t f = Mr + t * ST; m_red(f, -g1); m_red(f + dMs, g1); };
                        const uint32_t nfull = d >> 2, tail = d & 3u;
                        uint32_t q4 = tile_lane;
                        for (uint32_t q = 0; q < nfull; ++q, q4 += 128u) {
                            const uint32_t t0 = sh_ld_u8(q4), t1 = sh_ld_u8(q4 + 32u), t2 = sh_ld_u8(q4 + 64u), t3 = sh_ld_u8(q4 + 96u);
                            move1(t0); move1(t1); move1(t2); move1(t3);
                        }
                        if (tail) {
                            move1(sh_ld_u8(q4));
                            if (tail > 1u) move1(sh_ld_u8(q4 + 32u));
                            if (tail > 2u) move1(sh_ld_u8(q4 + 64u));
                        }
                    }
                    for (uint32_t w = 0; w < hist_words; ++w) sh_st_u32v(hist_base + w * 128u, 0u);
                } else {              // hubs: the histogram is k_t
                    uint32_t ha = hist_base;
                    for (uint32_t w = 0; w < hist_words; ++w, ha += 128u) {
                        uint32_t word = sh_ld_u32v(ha);
                        sh_st_u32v(ha, 0u);
                        word = go ? word : 0u;
#pragma unroll
                        for (uint32_t b = 0; b < 4; ++b) {
                            const uint32_t t = (KF == 32) ? w + 8u * b : w * 4u + b;
                            if (t < kopp_max) {
                                const int kk = (int)((word >> (8u * b)) & 0xffu);
                                if (STAGED || kk != 0) { m_red(Mr + t * ST, -kk); m_red(Ms + t * ST, kk); }
                            }
                        }
                    }
                }
                if (go) {
                    eo_red(r, -(int)d);
                    eo_red(s, (int)d);
                    no_red(s, 1);
                    if constexpr (STAGED)
                        if (!P.exclusive && ((sh_ld_u32v(Small_base + (s >> 5) * 128u) >> (s & 31u)) & 1u)) atomicAdd(&gLIVE[s * 32 + lane], 1);
                    atomicSub(&gETA[(r * W + didx) * 32 + lane], 1);
                    atomicAdd(&gETA[(s * W + didx) * 32 + lane], 1);
                    lab_st(v, s);
                    ++n_acc;
                    ds_sum += (double)dS;
                }
                RC_MARK(2);
                round_barrier();                             // every warp of the round has committed
                RC_MARK(4);
            }
            if constexpr (STAGED)                            // rounds of the batch in which this warp has no vertex
                for (const uint32_t all = (nb + P.warps_used - 1u) / P.warps_used; rounds < all; ++rounds) {
                    RC_ROUND(); round_barrier(); RC_MARK(3); round_barrier(); RC_MARK(4);
                }
        }
        j0 += (uint32_t)S2_VB;
        if (j0 >= cnt) break;
        __syncthreads();
        nb = prepare(j0);
        __syncthreads();
    }
    RC_PUBLISH(STAGED && warp < P.warps_used && lane == 0);
    RC_CTA_RESET();
    if (warp < P.warps_used && live) {
        if (n_acc) atomicAdd(&P.accepted[c], (unsigned long long)n_acc);
        if (ds_sum != 0.0) atomicAdd(&P.dS_accum[c], ds_sum);
    }

    // ---- publish the staged counts ----
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // shared-memory writes of this thread -> visible to the bulk engine
    __syncthreads();
    if (P.kat_mode || !STAGED) return;
    if (P.exclusive) {
        copy_i4(gM, sM, KA * KB * 32);
        copy_i4(gE + own_off * 32, sEo, kown_max * 32);
        copy_i4(gNR + own_off * 32, sNo, kown_max * 32);
    } else if (threadIdx.x == 0) {
        char* const nM = reinterpret_cast<char*>(P.m_next + (size_t)group * KA * KB * GROUP);
        const uint32_t bM = KA * KB * 128u, bO = kown_max * 128u;
        for (uint32_t off = 0; off < bM; off += 32768u) bulk_red_add_s32(nM + off, sbase + L.oM + off, min(32768u, bM - off));
        bulk_red_add_s32(P.e_next + (size_t)group * KK * GROUP + own_off * 32, sbase + L.oEo, bO);
        bulk_red_add_s32(P.nr_next + (size_t)group * KK * GROUP + own_off * 32, sbase + L.oNo, bO);
        bulk_commit_wait_all();
    }
    RC_CTA_END();
}

#endif  // __CUDACC__

}  // namespace bisbm
