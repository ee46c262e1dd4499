// staged_model.cc -- an exact host model of what every move of the staged sweep kernel (sweep2_kernel, STAGED) reads.
//
// The staged kernel is deterministic by construction (fixed rounds, eta as it was at a sliced launch's start, a Philox draw
// keyed by (vertex, sweep, seed)), so one sweep can be replayed move by move on the host.  The model restates the contract
// of DESIGN.md 3.2 independently of the kernel's text:
//   * visiting order: launch l, group g, CTA j of the group take positions pos_begin + j + i cpg (per-group pos_begin / cpg
//     with spare-SM extras), position p is vertex v0 + feistel_perm(p, nv, half_bits, pkey(sweep, type, g)); the positions
//     of all launches of a half sweep must cover [0, nv) once per group (checked here);
//   * rounds: the CTA's share in batches of 448, round k = entries k wu .. k wu + wu - 1; a move sees m_rs and the moving
//     type's e_r / n_r at the launch's start plus this CTA's commits of earlier rounds; eta at the launch's start (sliced)
//     or after the earlier rounds (one CTA); the frozen type's e_r at the launch's start;
//   * the proposal, dS / the Hastings factor (long double, lgamma and the oracle's log q), the acceptance and the veto.
// Only philox4x32, feistel_perm, feistel_half_bits and mulhi32 come from the device headers: they define the stream.
//
// A chain is marked ambiguous for the sweep where the device's decision could legitimately differ from the model's (a
// floating-point near-tie in the accept or epsilon test, or a veto whose outcome depends on the order of atomics); an
// ambiguous chain is not simulated further in that sweep.  Test aid, not product code.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include "../bipartitesbm-mcmc_b200/csrc/devmath.cuh"

using bisbm::feistel_half_bits;
using bisbm::feistel_perm;
using bisbm::mulhi32;
using bisbm::philox4x32;
using bisbm::u32x4;

extern "C" {
double* ora_build_log_q_table(uint32_t n_max, uint32_t k_max);
double ora_log_q_approx(uint64_t n, uint64_t k);
double ora_schedule(int schedule, float p0, float p1, uint64_t t);
void ora_free(void* p);
}

namespace {

typedef long double LD;
constexpr uint32_t VB = 448;   // vertices per batch of a CTA's share

enum { FLAG_AMBIGUOUS = 1u, FLAG_VETO = 2u, FLAG_TIE = 4u, FLAG_EPS = 8u };

struct Graph {
    uint32_t na, nb, n, W;
    uint64_t E;
    const uint32_t* rp;
    const uint32_t* col;
    std::vector<uint32_t> deg, didx;
    std::vector<LD> lgt;        // lgammal(i)
    double* qtab = nullptr;     // exact log q, [10001][qk + 1]
    uint32_t qk = 0;
    LD lg(int64_t i) const { return lgt[(size_t)i]; }
    LD logq(int64_t e, int64_t k, bool* approx, bool* oot) const {   // ora_log_q(e, k): e edges, k = n_r
        if (e <= 0 || k < 1) return 0;
        if (k > e) k = e;
        if (e < 10001) {
            if ((uint32_t)k > qk) { *oot = true; return 0; }
            return qtab[(size_t)e * (qk + 1) + k];
        }
        *approx = true;              // the device tabulates the asymptotic branch: a looser tie tolerance
        return ora_log_q_approx((uint64_t)e, (uint64_t)k);
    }
};

struct Plan { uint32_t cpg, slice, warps_used, extras, sliced; };

// one launch of one group: per CTA of the group, the positions it visits in order and their vertices
struct Launch { uint32_t span; std::vector<std::vector<uint32_t>> pos, vtx; };

// the launches of one half sweep for one group, restated from launch_full_sweep and the kernel's position arithmetic;
// pkey / half_bits / v0 map a position to its vertex (pass v0 = ~0u for positions only)
static int visiting_order(uint32_t nv, uint32_t G, uint32_t g, const Plan& pl, uint32_t v0, uint64_t pkey,
                          std::vector<Launch>* out) {
    const uint32_t hb = feistel_half_bits(nv);
    const uint32_t per_cta = pl.slice / std::max<uint32_t>(1, pl.cpg);
    std::vector<uint8_t> seen(nv, 0);
    for (uint64_t l = 0;; ++l) {
        const uint64_t pos = pl.extras ? (l * pl.cpg + (l * pl.extras) / G) * per_cta : l * pl.slice;
        if (pos >= nv) break;
        uint64_t pb = pos, pe = std::min<uint64_t>(nv, pos + pl.slice);
        uint32_t cpg = pl.cpg;
        if (pl.extras) {   // group g's own slice: it has been handed one slot per `extras` turn so far
            const uint64_t s0 = l * pl.extras, slot0 = s0 % G;
            const uint64_t before = (s0 + G - 1 - g) / G;
            const bool has_extra = (g + G - slot0) % G < pl.extras;
            cpg += has_extra ? 1 : 0;
            const uint64_t b = (l * pl.cpg + before) * per_cta;
            pb = std::min<uint64_t>(b, nv);
            pe = std::min<uint64_t>(b + (uint64_t)cpg * per_cta, nv);
        }
        Launch L;
        L.span = (uint32_t)(pe - pb);
        L.pos.resize(cpg);
        L.vtx.resize(cpg);
        for (uint32_t j = 0; j < cpg; ++j)
            for (uint64_t p = pb + j; p < pe; p += cpg) {
                if (seen[p]) return -1;
                seen[p] = 1;
                L.pos[j].push_back((uint32_t)p);
                if (v0 != ~0u) L.vtx[j].push_back(v0 + feistel_perm((uint32_t)p, nv, hb, pkey));
            }
        out->push_back(std::move(L));
    }
    for (uint32_t p = 0; p < nv; ++p)
        if (!seen[p]) return -2;
    return 0;
}

// the counts of one chain seen from the moving type: m[x][t] (x own, t frozen), e / n of the own blocks, eta [own][didx]
struct View { std::vector<int> m, eo, no; };

struct Chain {
    uint32_t ka, kb, kown, kopp;
    View B;                               // base: counts at the launch's start (one CTA: live)
    std::vector<int> ep, eta;             // frozen type's e_r; own eta [kown][W]
    int occ_opp = 0;
};

struct Args {
    const Graph* g;
    uint32_t* labels;                     // [n] global ids of this chain
    uint32_t ka, kb;
    double eps;
    uint64_t seed, epoch, step_base[2];
    int schedule;
    float p0, p1;
    const Plan* plan;                     // [2]
    const std::vector<Launch>* order[2];  // this chain's group
    int vary_k, fp32;
    uint64_t accepted = 0;
    double ds = 0, tol = 0;
    uint32_t flags = 0;
    uint64_t moves = 0;
};

static LD prior_k_delta(LD E, LD n_own, LD k_own, LD k_opp, int dk) {
    auto lbin = [](LD N, LD k) -> LD {
        if (N == 0 || k == 0 || k > N) return 0;
        return lgammal(N + 1) - lgammal(k + 1) - lgammal(N - k + 1);
    };
    const LD k2 = k_own + dk;
    return (lbin(k2 * k_opp + E - 1, E) + lbin(n_own - 1, k2 - 1)) - (lbin(k_own * k_opp + E - 1, E) + lbin(n_own - 1, k_own - 1));
}

struct Move { uint32_t v, r, s; double dS, tol; bool pre, cand, self_acc; };   // pre: accepted before the veto

// transition_ratio (reference src/metropolis_hasting.cc:103-192) of moving v from own block r to s on the view: dS and the
// log of the Hastings factor.  *approx: a log q argument beyond the exact table; *oot: beyond the table this model built.
static void transition(const Args& a, const Chain& ch, const View& V, uint32_t type, uint32_t v, uint32_t r, uint32_t s,
                       std::vector<int>& kt, LD* dS_out, LD* lh_out, bool* approx, bool* oot) {
    const Graph& g = *a.g;
    const uint32_t off_opp = type ? 0 : a.ka, d = g.deg[v], K = a.ka + a.kb;
    for (uint64_t e = g.rp[v]; e < g.rp[v + 1]; ++e) kt[a.labels[g.col[e]] - off_opp]++;
    LD dS = 0, a0 = 0, a1 = 0;
    const LD epsl = a.eps;
    for (uint64_t e = g.rp[v]; e < g.rp[v + 1]; ++e) {
        const uint32_t t = a.labels[g.col[e]] - off_opp;
        const int kk = kt[t];
        if (kk == 0) continue;
        kt[t] = 0;
        const int mr = V.m[r * ch.kopp + t], ms = V.m[s * ch.kopp + t];
        const LD inv = 1.0L / ((LD)ch.ep[t] + epsl * K);
        a0 += kk * ((LD)ms + epsl) * inv;
        a1 += kk * ((LD)mr - kk + epsl) * inv;
        dS += g.lg(mr + 1) - g.lg(mr - kk + 1) + g.lg(ms + 1) - g.lg(ms + kk + 1);
    }
    const int e0r = V.eo[r], e0s = V.eo[s], e1r = e0r - (int)d, e1s = e0s + (int)d, n_r = V.no[r], n_s = V.no[s];
    dS += g.lg(e1r + 1) + g.lg(e1s + 1) - g.lg(e0r + 1) - g.lg(e0s + 1);
    const int eta_r = ch.eta[r * g.W + g.didx[v]], eta_s = ch.eta[s * g.W + g.didx[v]];
    dS += logl((LD)eta_r) - logl((LD)eta_s + 1);
    dS += g.logq(e1r, n_r - 1, approx, oot) + g.logq(e1s, n_s + 1, approx, oot) - g.logq(e0r, n_r, approx, oot) -
          g.logq(e0s, n_s, approx, oot);
    if (a.vary_k) {
        // estimate mode: the K-dependent prior terms, with the occupied count of the same view as n_r
        const int dk = ((n_s == 0) ? 1 : 0) - ((n_r == 1) ? 1 : 0);
        if (dk) {
            int occ = 0;
            for (uint32_t x = 0; x < ch.kown; ++x) occ += V.no[x] > 0 ? 1 : 0;
            dS += prior_k_delta((LD)g.E, (LD)(type ? g.nb : g.na), occ, ch.occ_opp, dk);
        }
    }
    *dS_out = dS;
    *lh_out = d ? logl(a1 / a0) : 0;
}

// one move evaluated against the view V (m, own e / n), the base's frozen e and eta.  Returns false when ambiguous.
static bool evaluate(Args& a, const Chain& ch, const View& V, uint32_t type, uint32_t v, uint64_t pos, Move* mv,
                     std::vector<int>& kt) {
    const Graph& g = *a.g;
    const uint32_t off_own = type ? a.ka : 0, off_opp = type ? 0 : a.ka;
    const uint32_t r = a.labels[v] - off_own;
    const uint32_t d = g.deg[v], K = a.ka + a.kb;
    mv->v = v; mv->r = r; mv->s = r; mv->pre = mv->cand = false; mv->self_acc = false; mv->dS = 0; mv->tol = 0;
    u32x4 ctr; ctr.x = v; ctr.y = (uint32_t)a.epoch; ctr.z = (uint32_t)a.seed; ctr.w = (uint32_t)(a.seed >> 32);
    const u32x4 ra = philox4x32(ctr, (uint32_t)(a.epoch >> 32) ^ 0xA4093822u, 0x299F31D0u);
    uint32_t tq = 0;
    if (d) tq = a.labels[g.col[g.rp[v] + mulhi32(ra.x, d)]] - off_opp;
    // beta of this position's step
    LD beta;
    const uint64_t step = a.step_base[type] + pos;
    if (a.schedule == 4) beta = ((float)step < a.p0) ? 1 : -1;
    else {
        const double T = ora_schedule(a.schedule, a.p0, a.p1, step);
        beta = (T == 0.0) ? -1 : (LD)(1.0 / T);
    }
    const bool T_zero = beta < 0;
    const int e_t = ch.ep[tq];
    bool uniform = d == 0;
    if (!uniform) {   // U < eps K / (e_t + eps K), U = y / 2^32
        const LD thr = (LD)a.eps * K * 4294967296.0L / ((LD)e_t + (LD)a.eps * K);
        if (fabsl((LD)ra.y - thr) < 1e-6L * thr) { a.flags |= FLAG_EPS; return false; }
        uniform = (LD)ra.y < thr;
    }
    const uint32_t sg = mulhi32(ra.z, K);          // uniform over all K blocks of the chain
    const bool sg_a = sg < a.ka;
    const uint32_t s_uni = sg_a ? sg : sg - a.ka;
    uint32_t s_cat = 0;                            // categorical over the view's m[.][t]
    {
        const int64_t z = mulhi32(ra.z, (uint32_t)e_t);
        int64_t cum = 0;
        uint32_t le = 0;
        for (uint32_t x = 0; x < ch.kown; ++x) { cum += V.m[x * ch.kopp + tq]; le += (cum <= z) ? 1 : 0; }
        s_cat = std::min(le, ch.kown - 1);
    }
    const bool movable = ch.kown != 1;
    const bool cross = movable && uniform && (sg_a != (type == 0));   // a draw of the other type: rejected
    const uint32_t s = (movable && !cross) ? (uniform ? s_uni : s_cat) : r;
    mv->s = s;
    if (s == r) {
        mv->self_acc = !cross && !T_zero && V.no[r] != 1;
        return true;
    }
    LD dS, lh;
    bool approx = false, oot = false;
    transition(a, ch, V, type, v, r, s, kt, &dS, &lh, &approx, &oot);
    if (oot) { a.flags |= FLAG_TIE; return false; }
    LD tol;
    if (a.fp32) tol = 1e-4L * std::max<LD>(1, fabsl(dS) / 8) * std::max<LD>(1, fabsl(beta)) + 2e-5L * std::max<LD>(1, fabsl(lh));
    else tol = ((approx ? 4e-6L : 1e-8L) + 1e-10L * fabsl(dS)) * std::max<LD>(1, fabsl(beta)) + 1e-12L * std::max<LD>(1, fabsl(lh));
    bool go;
    if (T_zero) {
        if (fabsl(dS) < tol) { a.flags |= FLAG_TIE; return false; }
        go = dS < 0;
    } else {
        const LD x = lh - dS * beta;
        const uint32_t w = ra.w;
        const LD lu = logl(a.fp32 ? ((LD)(w >> 8) + 0.5L) / 16777216.0L : ((LD)w + 0.5L) / 4294967296.0L);
        if (fabsl(x - lu) < tol) { a.flags |= FLAG_TIE; return false; }
        go = lu < x;
    }
    mv->dS = (double)dS;
    mv->tol = (double)tol;
    mv->pre = mv->cand = go;
    return true;
}

// commit of an accepted move into a view (m, own e / n)
static void commit_view(const Args& a, const Chain& ch, View& V, uint32_t type, const Move& mv) {
    const Graph& g = *a.g;
    const uint32_t off_opp = type ? 0 : a.ka;
    for (uint64_t e = g.rp[mv.v]; e < g.rp[mv.v + 1]; ++e) {
        const uint32_t t = a.labels[g.col[e]] - off_opp;
        V.m[mv.r * ch.kopp + t]--;
        V.m[mv.s * ch.kopp + t]++;
    }
    V.eo[mv.r] -= (int)g.deg[mv.v]; V.eo[mv.s] += (int)g.deg[mv.v];
    V.no[mv.r]--; V.no[mv.s]++;
}

static void commit_label(Args& a, Chain& ch, uint32_t type, const Move& mv) {
    const uint32_t W = a.g->W, di = a.g->didx[mv.v];
    ch.eta[mv.r * W + di]--; ch.eta[mv.s * W + di]++;
    a.labels[mv.v] = mv.s + (type ? a.ka : 0);
    ++a.accepted;
    a.ds += mv.dS;
    a.tol += mv.tol;
}

static void build_chain(const Args& a, uint32_t type, Chain* ch) {
    const Graph& g = *a.g;
    ch->ka = a.ka; ch->kb = a.kb;
    ch->kown = type ? a.kb : a.ka; ch->kopp = type ? a.ka : a.kb;
    const uint32_t off_own = type ? a.ka : 0, off_opp = type ? 0 : a.ka;
    ch->B.m.assign((size_t)ch->kown * ch->kopp, 0);
    ch->B.eo.assign(ch->kown, 0); ch->B.no.assign(ch->kown, 0);
    ch->ep.assign(ch->kopp, 0);
    ch->eta.assign((size_t)ch->kown * g.W, 0);
    std::vector<int> nopp(ch->kopp, 0);
    const uint32_t o0 = type ? g.na : 0, o1 = type ? g.n : g.na;
    for (uint32_t v = 0; v < g.n; ++v) {
        const bool own = v >= o0 && v < o1;
        const uint32_t b = a.labels[v] - (own ? off_own : off_opp);
        if (own) {
            ch->B.no[b]++; ch->B.eo[b] += (int)g.deg[v]; ch->eta[b * g.W + g.didx[v]]++;
            for (uint64_t e = g.rp[v]; e < g.rp[v + 1]; ++e) ch->B.m[b * ch->kopp + (a.labels[g.col[e]] - off_opp)]++;
        } else {
            nopp[b]++; ch->ep[b] += (int)g.deg[v];
        }
    }
    ch->occ_opp = 0;
    for (int x : nopp) ch->occ_opp += x > 0 ? 1 : 0;
}

// veto of a move out of r: "old" (the count the atomic returns) lies in [lo, hi]; returns 1 pass, 0 veto, -1 undecided
static int veto_pass(int lo, int hi) { return lo > 1 ? 1 : (hi <= 1 ? 0 : -1); }


// one half sweep of one chain under the plan; returns early (flags |= FLAG_AMBIGUOUS) at the first ambiguous decision
static void half_sweep(Args& a, uint32_t type) {
    const Plan& pl = a.plan[type];
    const uint32_t wu = std::max<uint32_t>(1, pl.warps_used);
    Chain ch;
    build_chain(a, type, &ch);
    std::vector<int> kt(ch.kopp, 0);
    std::vector<Move> round, done;
    // the rounds of one CTA's share: batches of VB entries, round k of a batch = entries k wu .. k wu + wu - 1
    auto rounds = [&](const std::vector<uint32_t>& P, const std::vector<uint32_t>& Vx, View& V, auto&& on_round) -> bool {
        for (size_t b0 = 0; b0 < P.size(); b0 += VB) {
            const size_t b1 = std::min(P.size(), b0 + VB);
            for (size_t k0 = b0; k0 < b1; k0 += wu) {
                round.clear();
                for (size_t i = k0; i < std::min(b1, k0 + wu); ++i) {
                    Move mv;
                    if (!evaluate(a, ch, V, type, Vx[i], P[i], &mv, kt)) return false;
                    round.push_back(mv);
                }
                if (!on_round()) return false;
            }
        }
        return true;
    };
    for (const Launch& L : *a.order[type]) {
        if (!pl.sliced) {
            // one CTA: the view is the chain's counts, eta included; the veto sees the exact shared n_r of the round
            const bool ok = rounds(L.pos[0], L.vtx[0], ch.B, [&]() -> bool {
                for (Move& m : round) {
                    a.moves++;
                    if (m.self_acc) a.accepted++;
                    if (!m.cand || a.vary_k) continue;
                    int out = 0, in = 0;
                    for (const Move& o : round)
                        if (&o != &m && o.pre) { out += o.r == m.r; in += o.s == m.r; }
                    const int p = veto_pass(ch.B.no[m.r] - out, ch.B.no[m.r] + in);
                    if (p < 0) { a.flags |= FLAG_VETO; return false; }
                    if (p == 0) m.cand = false;
                }
                for (const Move& m : round)
                    if (m.cand) { commit_view(a, ch, ch.B, type, m); commit_label(a, ch, type, m); }
                return true;
            });
            if (!ok) { a.flags |= FLAG_AMBIGUOUS; return; }
            continue;
        }
        // several CTAs: CTA j sees the base plus its own commits; the veto of a "small" block (n_r(base) <= span + 1)
        // counts the launch's decrements from every CTA in an order the model does not know.  Its outcome is taken
        // from bounds on that count, iterated to a fixed point over the candidates of the whole launch.
        std::vector<int> c_out(ch.kown, 0), c_in(ch.kown, 0), n_out, n_in;
        uint64_t self_acc = 0;
        bool stable = false, open = false;
        for (int it = 0; it < 8 && !stable; ++it) {
            open = false;
            n_out.assign(ch.kown, 0); n_in.assign(ch.kown, 0);
            done.clear();
            self_acc = 0;
            for (size_t j = 0; j < L.pos.size(); ++j) {
                View V = ch.B;
                const bool ok = rounds(L.pos[j], L.vtx[j], V, [&]() -> bool {
                    for (Move& m : round) {
                        if (m.self_acc) self_acc++;
                        if (!m.cand) continue;
                        n_out[m.r]++; n_in[m.s]++;
                        if (a.vary_k || ch.B.no[m.r] > (int)L.span + 1) continue;
                        const int p = veto_pass(ch.B.no[m.r] - std::max(0, c_out[m.r] - 1), ch.B.no[m.r] + c_in[m.r]);
                        open |= p < 0;
                        if (p == 0) m.cand = false;
                    }
                    for (const Move& m : round)
                        if (m.cand) { commit_view(a, ch, V, type, m); done.push_back(m); }
                    return true;
                });
                if (!ok) { a.flags |= FLAG_AMBIGUOUS; return; }
            }
            stable = n_out == c_out && n_in == c_in;
            c_out.swap(n_out); c_in.swap(n_in);
        }
        if (!stable || open) { a.flags |= FLAG_VETO | FLAG_AMBIGUOUS; return; }
        for (size_t j = 0; j < L.pos.size(); ++j) a.moves += L.pos[j].size();
        a.accepted += self_acc;
        for (const Move& m : done) { commit_view(a, ch, ch.B, type, m); commit_label(a, ch, type, m); }
    }
}

static std::vector<double*> g_qtabs;      // exact log q tables kept between calls, by column count
static std::vector<uint32_t> g_qks;

}  // namespace

extern "C" {

// positions of every group's launches of one half sweep cover [0, nv) exactly once: 0, else < 0.  *n_launches: launches
int sm_visit_cover(uint32_t nv, uint32_t n_groups, uint32_t cpg, uint32_t slice, uint32_t extras, uint32_t* n_launches,
                   uint32_t* cta_max) {
    const Plan pl = {cpg, slice, 1, extras, 1};
    *cta_max = 0;
    for (uint32_t g = 0; g < n_groups; ++g) {
        std::vector<Launch> o;
        const int rc = visiting_order(nv, n_groups, g, pl, ~0u, 0, &o);
        if (rc) return rc;
        *n_launches = (uint32_t)o.size();
        for (const Launch& L : o) *cta_max = std::max<uint32_t>(*cta_max, (uint32_t)L.pos.size());
    }
    return 0;
}

static void make_graph(Graph* g, uint32_t na, uint32_t nb, uint64_t E, const uint32_t* rp, const uint32_t* col, uint32_t qk) {
    g->na = na; g->nb = nb; g->n = na + nb; g->E = E; g->rp = rp; g->col = col;
    g->deg.resize(g->n);
    uint32_t dmax = 0;
    for (uint32_t v = 0; v < g->n; ++v) { g->deg[v] = rp[v + 1] - rp[v]; dmax = std::max(dmax, g->deg[v]); }
    std::vector<uint32_t> idx(dmax + 1, ~0u);
    g->W = 0;
    for (uint32_t v = 0; v < g->n; ++v) if (idx[g->deg[v]] == ~0u) idx[g->deg[v]] = g->W++;
    g->didx.resize(g->n);
    for (uint32_t v = 0; v < g->n; ++v) g->didx[v] = idx[g->deg[v]];
    g->lgt.resize(E + g->n + 3);
    g->lgt[0] = INFINITY;
    for (size_t i = 1; i < g->lgt.size(); ++i) g->lgt[i] = lgammal((LD)i);
    for (size_t i = 0; i < g_qks.size(); ++i)
        if (g_qks[i] >= qk) { g->qtab = g_qtabs[i]; g->qk = g_qks[i]; return; }
    g->qtab = ora_build_log_q_table(10000, qk);
    g->qk = qk;
    g_qtabs.push_back(g->qtab); g_qks.push_back(qk);
}

// dS and log accu_r of moving v to global block s, on the counts rebuilt from `labels` (one chain), by the model's code
int sm_transition(uint32_t na, uint32_t nb, uint64_t E, const uint32_t* rp, const uint32_t* col, uint32_t* labels, uint32_t ka,
                  uint32_t kb, double eps, uint32_t v, uint32_t s, double* dS, double* lh) {
    Graph g;
    make_graph(&g, na, nb, E, rp, col, std::max(na, nb) + 1);
    Args a;
    a.g = &g; a.labels = labels; a.ka = ka; a.kb = kb; a.eps = eps; a.vary_k = 0; a.fp32 = 0;
    const uint32_t type = v >= na ? 1 : 0, off = type ? ka : 0;
    Chain ch;
    build_chain(a, type, &ch);
    std::vector<int> kt(ch.kopp, 0);
    LD d, l;
    bool approx = false, oot = false;
    transition(a, ch, ch.B, type, v, labels[v] - off, s - off, kt, &d, &l, &approx, &oot);
    *dS = (double)d; *lh = (double)l;
    return oot ? -1 : 0;
}

// One full sweep (type a, then type b) of every chain, as the staged kernel runs it under plan[type] = {ctas per group,
// slice, warps used, extras, sliced}.  labels [n_chains][n] (global ids) in / out; per chain: accepted moves, sum of dS of the
// accepted moves, the sum of their tie tolerances, flags (FLAG_*), visited moves.
int sm_replay_sweep(uint32_t na, uint32_t nb, uint64_t E, const uint32_t* rp, const uint32_t* col, uint32_t n_chains,
                    uint32_t* labels, const uint32_t* ka, const uint32_t* kb, double eps, const uint64_t* seeds, uint64_t epoch,
                    uint64_t sweep_in_call, int schedule, float p0, float p1, const uint32_t* plan, int vary_k, int fp32,
                    uint64_t* accepted, double* ds, double* tol, uint32_t* flags, uint64_t* moves) {
    const uint32_t n = na + nb, G = (n_chains + 31) / 32;
    // exact log q columns: twice the largest block, plus room
    uint32_t nmax = 1;
    for (uint32_t c = 0; c < n_chains; ++c) {
        std::vector<uint32_t> cnt(ka[c] + kb[c], 0);
        for (uint32_t v = 0; v < n; ++v) nmax = std::max(nmax, ++cnt[labels[(size_t)c * n + v]]);
    }
    Graph g;
    make_graph(&g, na, nb, E, rp, col, std::min<uint32_t>(std::max(na, nb), 2 * nmax + 64));
    Plan pl[2];
    for (int t = 0; t < 2; ++t) pl[t] = {plan[5 * t], plan[5 * t + 1], plan[5 * t + 2], plan[5 * t + 3], plan[5 * t + 4]};
    std::vector<std::vector<Launch>> order[2];
    for (uint32_t t = 0; t < 2; ++t) {
        order[t].resize(G);
        const uint32_t nv = t ? nb : na;
        if (nv == 0) continue;
        for (uint32_t grp = 0; grp < G; ++grp) {
            const uint64_t pkey = (epoch * 2 + t) * 0x9E3779B97F4A7C15ull + (uint64_t)grp * 0xD1B54A32D192ED03ull;
            const int rc = visiting_order(nv, G, grp, pl[t], t ? na : 0, pkey, &order[t][grp]);
            if (rc) return rc;
        }
    }
    std::vector<std::thread> th;
    std::atomic<uint32_t> next(0);
    const unsigned nth = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    for (unsigned i = 0; i < nth; ++i)
        th.emplace_back([&]() {
            for (uint32_t c; (c = next.fetch_add(1)) < n_chains;) {
                Args a;
                a.g = &g; a.labels = labels + (size_t)c * n; a.ka = ka[c]; a.kb = kb[c]; a.eps = eps; a.seed = seeds[c];
                a.epoch = epoch; a.step_base[0] = sweep_in_call * n; a.step_base[1] = sweep_in_call * n + na;
                a.schedule = schedule; a.p0 = p0; a.p1 = p1; a.plan = pl;
                a.order[0] = &order[0][c / 32]; a.order[1] = &order[1][c / 32];
                a.vary_k = vary_k; a.fp32 = fp32;
                for (uint32_t t = 0; t < 2 && !(a.flags & FLAG_AMBIGUOUS); ++t)
                    if (t ? nb : na) half_sweep(a, t);
                accepted[c] = a.accepted; ds[c] = a.ds; tol[c] = a.tol; flags[c] = a.flags; moves[c] = a.moves;
            }
        });
    for (auto& t : th) t.join();
    return 0;
}

}  // extern "C"
