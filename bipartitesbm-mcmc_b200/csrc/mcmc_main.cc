// mcmc_main.cc -- bin/mcmc: the reference's command line over libbisbm.so (include/bisbm.h).
//
// Drop-in for the straight path of the reference driver (reference src/mcmc_main.cc:29-487):
// the same option table (src/mcmc_main.cc:54-93), the same validation messages and exit codes,
// the same stderr lines ("acceptance ratio", "(Ka, Kb) = ...", "entropy: ...") and the same
// stdout label line (src/output_functions.hh:20-28).  The chain itself runs on the GPU:
//   default / --maximize   one chain, sequential REPLAY mode: the reference's own draw order, so with
//                          the same --seed (and --gen_seed for the reference's random_device-seeded
//                          second engine) the label line is identical to the reference's
//   --chains N             N parallel chains (restarts with randomised starts); prints the best
//   --marginalize          README "marginalization": -b burn-in sweeps, -t sampling sweeps, one sample
//                          every -f sweeps over --chains chains; prints the arg-max label per node.  With
//                          --tempering T0 T1 .. the chains form ladders of those temperatures (parallel tempering,
//                          swaps every --swap_every sweeps) and only the chains at T0 are sampled.  With --align the
//                          burn-in runs first, the lowest-entropy (cold) chain becomes the reference partition and
//                          every sample is relabelled to agree with it before it is counted (bisbm_marginals_align).
//                          With --coassign FILE --coassign_out OUT every sample also counts, for each pair of the query
//                          nodes in FILE, the chains in which the two share a block (bisbm_coassign_set); OUT gets the
//                          matrix, summed over the GPUs of --gpus
//   --agreement_out FILE   (one GPU: --chains N >= 2, --marginalize, --estimate) compares the final states of the chains
//                          pairwise (bisbm_chain_agreement): FILE gets NMI / VI / ARI / matched overlap per pair, stderr
//                          a one-line summary with the modes at overlap >= 0.95
//   --modes_out FILE       (--marginalize, one GPU, --chains N >= 2) after the burn-in, the modes of the chains (of the
//                          chains at T0 under --tempering) at overlap >= 0.95 become reference partitions, each the labels
//                          of its lowest-entropy member, and every sample is counted in the histogram of the nearest one
//                          (bisbm_marginal_modes_set); FILE gets the per-mode counts and arg-max labels
//   --estimate             README "estimation" output format for fixed (Ka, Kb): CSV lines
//                          sweep,Ka,Kb,loglik,labels... of the last 1000 samples
//   -g / --merge, -u / --nature, or initial labels whose block counts differ from -z: the agglomerative
//                          merge / split initialiser (src/mcmc_main.cc:350-451) over bisbm_replay_agg_merge -- the
//                          geospace ladder, one greedy sweep between rungs, then the abrupt_cool anneal; one replay
//                          chain, the label line of the reference for the merge paths
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <fstream>
#include <iterator>
#include <iostream>
#include <limits>
#include <map>
#include <random>
#include <sstream>
#include <string>
#include <vector>

#include <thread>
#include <unistd.h>

#include "bisbm.h"

namespace {

struct Options {
    std::map<std::string, std::vector<std::string>> vals;  // long name -> tokens
    bool has(const std::string& k) const { return vals.count(k) > 0; }
    const std::vector<std::string>& get(const std::string& k) const {
        static const std::vector<std::string> empty;
        auto it = vals.find(k);
        return it == vals.end() ? empty : it->second;
    }
};

struct Spec { const char* lng; char sht; int kind; };  // kind: 0 flag, 1 single value, 2 multitoken
const Spec kSpecs[] = {
    {"edge_list_path", 'e', 1}, {"membership_path", 0, 1}, {"mb", 0, 2}, {"n", 'n', 2}, {"types", 'y', 2},
    {"burn_in", 'b', 1}, {"sampling_steps", 't', 1}, {"sampling_frequency", 'f', 1}, {"bisbm_partition", 'z', 2},
    {"uni", 0, 0}, {"cooling_schedule", 'c', 1}, {"cooling_schedule_kwargs", 'a', 2}, {"steps_await", 'x', 1},
    {"epsilon", 'E', 1}, {"randomize", 'r', 0}, {"merge", 'g', 0}, {"nature", 'u', 0}, {"seed", 'd', 1},
    {"help", 'h', 0},
    // README-only modes and the extensions of this build
    {"maximize", 0, 0}, {"estimate", 0, 0}, {"marginalize", 0, 0}, {"chains", 0, 1}, {"gen_seed", 0, 1},
    {"device", 0, 1}, {"max_inflight", 0, 1}, {"gpus", 0, 1}, {"tempering", 0, 2}, {"swap_every", 0, 1},
    {"align", 0, 0}, {"coassign", 0, 1}, {"coassign_out", 0, 1}, {"agreement_out", 0, 1},
    {"modes_out", 0, 1},
};

const Spec* find_spec(const std::string& tok) {
    if (tok.size() >= 3 && tok[0] == '-' && tok[1] == '-') {
        std::string name = tok.substr(2);
        size_t eq = name.find('=');
        if (eq != std::string::npos) name = name.substr(0, eq);
        for (const Spec& s : kSpecs) if (name == s.lng) return &s;
        return nullptr;
    }
    if (tok.size() == 2 && tok[0] == '-' && !isdigit((unsigned char)tok[1]))
        for (const Spec& s : kSpecs) if (s.sht && tok[1] == s.sht) return &s;
    return nullptr;
}

bool looks_like_option(const std::string& t) {
    return t.size() >= 2 && t[0] == '-' && !(isdigit((unsigned char)t[1]) || t[1] == '.');
}

bool parse(int argc, char const* argv[], Options& o, std::string& err) {
    for (int i = 1; i < argc; ++i) {
        std::string tok = argv[i];
        const Spec* s = find_spec(tok);
        if (!s) { err = "unrecognised option '" + tok + "'"; return false; }
        std::vector<std::string>& v = o.vals[s->lng];
        size_t eq = tok.find('=');
        if (tok.compare(0, 2, "--") == 0 && eq != std::string::npos) { v.push_back(tok.substr(eq + 1)); continue; }
        if (s->kind == 0) continue;
        if (s->kind == 1) {
            if (i + 1 >= argc) { err = std::string("the required argument for option '--") + s->lng + "' is missing"; return false; }
            v.push_back(argv[++i]);
        } else {
            while (i + 1 < argc && !looks_like_option(argv[i + 1])) v.push_back(argv[++i]);
            if (v.empty()) { err = std::string("the required argument for option '--") + s->lng + "' is missing"; return false; }
        }
    }
    return true;
}

template <class T>
bool to_num(const std::string& s, T& out) {
    std::istringstream is(s);
    is >> out;
    return !is.fail();
}

void usage(const char* argv0) {
    std::clog << "MCMC algorithms for the bipartiteSBM (final output only)\n";
    std::clog << "Usage:\n  " << argv0 << " [--option_1=value] [--option_s2=value] ...\n";
    std::clog << "Options:\n"
                 "  -e [ --edge_list_path ] arg           Path to edge list file.\n"
                 "  --membership_path arg                 Path to membership file.\n"
                 "  --mb arg                              Initial memberships.\n"
                 "  -n [ --n ] arg                        Block sizes vector.\n"
                 "  -y [ --types ] arg                    Block types vector (NA NB).\n"
                 "  -b [ --burn_in ] arg (=1000)          Burn-in time.\n"
                 "  -t [ --sampling_steps ] arg (=1000)   Length of the simulated annealing process (steps);\n"
                 "                                        sampling sweeps in --marginalize / --estimate.\n"
                 "  -f [ --sampling_frequency ] arg (=10) Sweeps between samples (--marginalize / --estimate).\n"
                 "  -z [ --bisbm_partition ] arg          bipartite number of blocks to be inferred.\n"
                 "  --uni                                 --estimate: print the 1D format (K = Ka + Kb)\n"
                 "  -c [ --cooling_schedule ] arg (=abrupt_cool)\n"
                 "                                        exponential, linear, logarithmic, constant, abrupt_cool.\n"
                 "  -a [ --cooling_schedule_kwargs ] arg  Schedule parameters.\n"
                 "  -x [ --steps_await ] arg (=1000)      Stop after x steps without a new entropy minimum.\n"
                 "  -E [ --epsilon ] arg (=1)             epsilon of the smart proposal.\n"
                 "  -r [ --randomize ]                    Randomize initial block state.\n"
                 "  -g [ --merge ]                        Agglomerative merge from singleton blocks down to -z.\n"
                 "  -u [ --nature ]                       with -g: merge until a type has fewer than sqrt(2E)/2 blocks.\n"
                 "  -d [ --seed ] arg                     Seed of the mt19937 engine.\n"
                 "  -h [ --help ]                         Produce this help message.\n"
                 "  --maximize | --marginalize | --estimate   mode (default: the reference's annealing path)\n"
                 "  --chains arg (=1)                     parallel chains on the GPU\n"
                 "  --gen_seed arg                        seed of the reference's second engine (std::random_device there)\n"
                 "  --device arg (=0), --max_inflight arg (=0)\n"
                 "  --gpus arg (=1)                       GPUs of this node: the chains are dealt round-robin to devices\n"
                 "                                        device .. device+gpus-1 (graph replicated); --marginalize sums the\n"
                 "                                        per-node histograms with one NCCL all-reduce\n"
                 "  --tempering T0 T1 ...                 --marginalize with parallel tempering: the chains form ladders of\n"
                 "                                        these temperatures (non-decreasing, T0 the cold one; --chains a\n"
                 "                                        multiple of their count); -b burn-in and -t sampling sweeps, the\n"
                 "                                        marginals sample only the chains at T0\n"
                 "  --swap_every arg (=1)                 sweeps between two swap rounds of --tempering\n"
                 "  --align                               --marginalize: after the burn-in, take the chain of lowest entropy\n"
                 "                                        (at T0 under --tempering; over all GPUs with --gpus) as the reference\n"
                 "                                        and relabel every sample's blocks, within each type, to agree with it\n"
                 "                                        on as many nodes as possible before counting it (label switching)\n"
                 "  --coassign arg                        --marginalize: file of query node ids, one per line; every sample\n"
                 "                                        counts, per pair of query nodes of one type, the chains in which the\n"
                 "                                        two share a block (posterior co-assignment, label-switching free)\n"
                 "  --coassign_out arg                    file the counts go to: a line \"Q n_counted\", then Q lines of Q\n"
                 "                                        counts in query order (summed over the GPUs of --gpus)\n"
                 "  --agreement_out arg                   one GPU, --chains >= 2 (plain, --marginalize, --estimate): compare\n"
                 "                                        the chains' final states pairwise; the file gets a line n_chains,\n"
                 "                                        then per pair c1 < c2: c1 c2 nmi vi ari overlap, then the same four\n"
                 "                                        for type a and for type b (label-switching free)\n"
                 "  --modes_out arg                       --marginalize, one GPU, --chains >= 2: after the burn-in, the modes of\n"
                 "                                        the chains (at T0 under --tempering) at overlap >= 0.95, each\n"
                 "                                        represented by its lowest-entropy chain, and every sample counted in\n"
                 "                                        the histogram of the nearest mode; the file gets a line \"M counted_0\n"
                 "                                        .. counted_M\" (the last: samples of no mode), then M lines of per-mode\n"
                 "                                        arg-max labels\n";
}

// the ladder of block counts between (start_a, start_b) and (end_a, end_b) (reference src/support/util.hh:99-146): the type
// with the longer way to go shrinks by the factor `ratio` per rung, the other one follows geometrically with the same number
// of rungs.  (The reference divides start_b / end_b as integers before taking the root; kept.)
void geospace(int start_a, int end_a, int start_b, int end_b, double ratio, std::vector<int>& ga, std::vector<int>& gb) {
    ga.clear(); gb.clear();
    if (ratio <= 1.) { ga.push_back(0); gb.push_back(0); return; }
    bool swapped = false;
    if (start_a - end_a < start_b - end_b) { std::swap(start_a, start_b); std::swap(end_a, end_b); swapped = true; }
    size_t i = 0;
    for (int d = start_a; d > end_a; d = (int)std::floor(start_a / std::pow(ratio, (double)i))) { ga.push_back(d); ++i; }
    ga.push_back(end_a);
    const size_t rungs = ga.size();
    const double rb = std::pow((double)(start_b / end_b), 1. / (double)(rungs - 1));
    for (size_t k = 0; k + 1 < rungs; ++k) gb.push_back((int)std::floor(start_b / std::pow(rb, (double)k)));
    gb.push_back(end_b);
    if (swapped) std::swap(ga, gb);
}

bool check(int rc) {
    if (rc != BISBM_OK) { std::cerr << "libbisbm: " << bisbm_last_error() << "\n"; return false; }
    return true;
}

void output_vec(const std::vector<uint32_t>& v, std::ostream& os) {  // reference src/output_functions.hh:20-28
    for (uint32_t x : v) os << x << " ";
    os << "\n";
}

// --coassign's node file: one id per line (blank lines skipped), each < n and none twice
bool read_query_nodes(const std::string& path, size_t n, std::vector<uint32_t>& nodes, std::string& err) {
    std::ifstream f(path.c_str());
    if (!f.is_open()) { err = "cannot read the --coassign file " + path; return false; }
    std::vector<uint8_t> seen(n, 0);
    std::string line;
    for (size_t ln = 1; std::getline(f, line); ++ln) {
        std::stringstream ls(line);
        std::string tok, extra;
        if (!(ls >> tok)) continue;
        size_t used = 0;
        unsigned long long v = 0;
        bool ok = tok.find_first_not_of("0123456789") == std::string::npos && !(ls >> extra);
        if (ok) { try { v = std::stoull(tok, &used); } catch (...) { ok = false; } }
        if (!ok || used != tok.size()) { err = "--coassign file line " + std::to_string(ln) + ": not a node id"; return false; }
        if (v >= n) { err = "--coassign file line " + std::to_string(ln) + ": node " + tok + " >= " + std::to_string(n); return false; }
        if (seen[v]) { err = "--coassign file line " + std::to_string(ln) + ": node " + tok + " appears twice"; return false; }
        seen[v] = 1;
        nodes.push_back((uint32_t)v);
    }
    if (nodes.empty()) { err = "the --coassign file " + path + " has no node ids"; return false; }
    return true;
}

// --coassign_out: "Q n_counted", then Q lines of Q counts
bool write_coassign(const std::string& path, size_t q, const std::vector<uint64_t>& counts, uint64_t n_counted) {
    std::ofstream f(path.c_str());
    if (!f.is_open()) { std::cerr << "cannot write the --coassign_out file " << path << "\n"; return false; }
    f << q << " " << n_counted << "\n";
    for (size_t i = 0; i < q; ++i) {
        for (size_t j = 0; j < q; ++j) f << (j ? " " : "") << counts[i * q + j];
        f << "\n";
    }
    f.close();
    if (f.fail()) { std::cerr << "cannot write the --coassign_out file " << path << "\n"; return false; }
    return true;
}

// --coassign: a handle's counts added to the running sum
int add_coassign(bisbm_handle* h, size_t q, std::vector<uint64_t>& sum, uint64_t& n_counted) {
    std::vector<uint32_t> c(q * q);
    uint64_t nc = 0;
    const int rc = bisbm_coassign_get(h, c.data(), &nc);
    if (rc != BISBM_OK) return rc;
    sum.resize(q * q, 0);
    for (size_t i = 0; i < q * q; ++i) sum[i] += c[i];
    n_counted += nc;
    return BISBM_OK;
}

// index of (metric, slot, chain i, chain j) in bisbm_chain_agreement's output for every pair of nc chains
size_t agree_at(int metric, int slot, size_t nc, size_t i, size_t j) { return (((size_t)metric * 3 + slot) * nc + i) * nc + j; }

// the modes among the chains cand: the connected components of "whole-partition overlap >= 0.95", numbered in order of each
// component's first chain in cand.  a: bisbm_chain_agreement over every pair of the pool's nc chains.  Returns the mode of
// each entry of cand; sizes gets the members per mode.
std::vector<size_t> overlap_modes(const std::vector<double>& a, size_t nc, const std::vector<size_t>& cand, std::vector<size_t>& sizes) {
    const size_t k = cand.size();
    std::vector<size_t> mode(k, k);
    sizes.clear();
    for (size_t c = 0; c < k; ++c) {
        if (mode[c] < k) continue;
        const size_t id = sizes.size();
        sizes.push_back(0);
        std::vector<size_t> stack{c};
        mode[c] = id;
        while (!stack.empty()) {
            const size_t x = stack.back();
            stack.pop_back();
            ++sizes[id];
            for (size_t y = 0; y < k; ++y)
                if (mode[y] == k && a[agree_at(BISBM_AGREE_OVERLAP, 2, nc, cand[x], cand[y])] >= 0.95) { mode[y] = id; stack.push_back(y); }
        }
    }
    return mode;
}

// --agreement_out: every pair of the pool's chains compared on their current labels (bisbm_chain_agreement).  The file gets
// "n_chains", then per pair c1 < c2 the whole partition's nmi vi ari overlap, then type a's, then type b's; stderr one
// summary line: the whole partition's NMI over the pairs and the modes, the connected components of overlap >= 0.95
bool write_agreement(bisbm_handle* h, size_t nc, const std::string& path) {
    std::vector<double> a(4 * 3 * nc * nc);
    if (!check(bisbm_chain_agreement(h, nullptr, 1, a.data()))) return false;
    auto at = [&](int metric, int slot, size_t i, size_t j) { return a[agree_at(metric, slot, nc, i, j)]; };
    std::ofstream f(path.c_str());
    if (!f.is_open()) { std::cerr << "cannot write the --agreement_out file " << path << "\n"; return false; }
    f.precision(17);
    f << nc << "\n";
    const int metrics[4] = {BISBM_AGREE_NMI, BISBM_AGREE_VI, BISBM_AGREE_ARI, BISBM_AGREE_OVERLAP};
    std::vector<double> nmi;
    for (size_t i = 0; i < nc; ++i)
        for (size_t j = i + 1; j < nc; ++j) {
            f << i << " " << j;
            for (int slot : {2, 0, 1})
                for (int metric : metrics) f << " " << at(metric, slot, i, j);
            f << "\n";
            nmi.push_back(at(BISBM_AGREE_NMI, 2, i, j));
        }
    f.close();
    if (f.fail()) { std::cerr << "cannot write the --agreement_out file " << path << "\n"; return false; }
    std::sort(nmi.begin(), nmi.end());
    const size_t np = nmi.size();
    const double median = np % 2 ? nmi[np / 2] : 0.5 * (nmi[np / 2 - 1] + nmi[np / 2]);
    std::vector<size_t> all(nc), sizes;
    for (size_t c = 0; c < nc; ++c) all[c] = c;
    overlap_modes(a, nc, all, sizes);
    std::clog << "chain agreement: NMI median " << median << " min " << nmi[0] << ", modes at overlap >= 0.95: " << sizes.size() << " (sizes";
    for (size_t z : sizes) std::clog << " " << z;
    std::clog << ")\n";
    return true;
}

// --align's reference: the chain of lowest entropy() in the pool (under a ladder, among the chains at rung 0)
int lowest_entropy_chain(bisbm_handle* h, size_t n_chains, bool cold_only, double* S, uint32_t* best) {
    std::vector<double> ent(n_chains);
    std::vector<uint32_t> rung(n_chains, 0);
    int rc = bisbm_entropy_all(h, ent.data());
    if (rc == BISBM_OK && cold_only) rc = bisbm_tempering_stats(h, rung.data(), nullptr, nullptr, nullptr, nullptr, nullptr);
    if (rc != BISBM_OK) return rc;
    bool found = false;
    for (size_t c = 0; c < n_chains; ++c)
        if (rung[c] == 0 && (!found || ent[c] < *S)) { *S = ent[c]; *best = (uint32_t)c; found = true; }
    return BISBM_OK;
}

// --modes_out: the modes of the chains' current labels (under a ladder, of the chains at rung 0) as --agreement_out finds
// them, each represented by its member of lowest entropy(), become the references of every later sample (min_overlap 0)
int set_modes(bisbm_handle* h, size_t nc, size_t n, bool cold_only, uint32_t* n_modes) {
    std::vector<double> a(4 * 3 * nc * nc), ent(nc);
    std::vector<uint32_t> rung(nc, 0);
    int rc = bisbm_chain_agreement(h, nullptr, 1, a.data());
    if (rc == BISBM_OK) rc = bisbm_entropy_all(h, ent.data());
    if (rc == BISBM_OK && cold_only) rc = bisbm_tempering_stats(h, rung.data(), nullptr, nullptr, nullptr, nullptr, nullptr);
    if (rc != BISBM_OK) return rc;
    std::vector<size_t> cand, sizes;
    for (size_t c = 0; c < nc; ++c) if (rung[c] == 0) cand.push_back(c);
    const std::vector<size_t> mode = overlap_modes(a, nc, cand, sizes);
    std::vector<size_t> best(sizes.size(), nc);
    for (size_t i = 0; i < cand.size(); ++i)
        if (best[mode[i]] == nc || ent[cand[i]] < ent[best[mode[i]]]) best[mode[i]] = cand[i];
    std::vector<uint32_t> refs(sizes.size() * n);
    for (size_t m = 0; m < sizes.size(); ++m)
        if ((rc = bisbm_get_labels(h, (uint32_t)best[m], refs.data() + m * n)) != BISBM_OK) return rc;
    *n_modes = (uint32_t)sizes.size();
    return bisbm_marginal_modes_set(h, *n_modes, refs.data(), 0.0);
}

// --modes_out: "M counted_0 .. counted_M", then the M arg-max label lines; stderr one line with the mode weights
bool write_modes(bisbm_handle* h, uint32_t M, size_t n, const std::string& path) {
    std::vector<uint64_t> counted(M + 1);
    std::vector<uint32_t> am((size_t)M * n);
    if (!check(bisbm_marginal_modes_get(h, nullptr, counted.data(), nullptr, nullptr)) || !check(bisbm_marginal_modes_argmax(h, am.data())))
        return false;
    std::ofstream f(path.c_str());
    if (!f.is_open()) { std::cerr << "cannot write the --modes_out file " << path << "\n"; return false; }
    f << M;
    for (uint64_t x : counted) f << " " << x;
    f << "\n";
    for (uint32_t m = 0; m < M; ++m) output_vec(std::vector<uint32_t>(am.begin() + (size_t)m * n, am.begin() + (size_t)(m + 1) * n), f);
    f.close();
    if (f.fail()) { std::cerr << "cannot write the --modes_out file " << path << "\n"; return false; }
    uint64_t total = 0;
    for (uint32_t m = 0; m < M; ++m) total += counted[m];
    std::clog << "marginal modes: " << M << ", weights";
    for (uint32_t m = 0; m < M; ++m) std::clog << " " << (total ? (double)counted[m] / (double)total : 0.0);
    std::clog << " (samples " << total << ", unassigned " << counted[M] << ")\n";
    return true;
}

}  // namespace

int main(int argc, char const* argv[]) {
    Options o;
    std::string perr;
    if (!parse(argc, argv, o, perr)) { std::cerr << perr << "\n"; return 1; }
    if (o.has("help") || argc == 1) { usage(argv[0]); return 0; }  // reference :99-105
    if (!o.has("edge_list_path")) { std::cerr << "edge_list_path is required (-e flag)\n"; return 1; }
    const std::string edge_list_path = o.vals["edge_list_path"][0];

    std::vector<unsigned> y;
    size_t NA = 0, NB = 0;
    if (!o.has("types")) { std::cerr << "types is required for bisbm mode (-y flag)\n"; return 1; }
    for (auto& s : o.vals["types"]) { unsigned v; if (!to_num(s, v)) { std::cerr << "bad value for --types\n"; return 1; } y.push_back(v); }
    if (y.size() != 2) { std::cerr << "Number of types must be equal to 2!\n"; return 1; }
    NA = y[0]; NB = y[1];

    size_t burn_in = 1000, sampling_steps = 1000, sampling_frequency = 10, steps_await = 1000, seed = 0;
    double epsilon = 1.0;
    std::string cooling_schedule = "abrupt_cool";
    if (o.has("burn_in") && !to_num(o.vals["burn_in"][0], burn_in)) { std::cerr << "bad value for --burn_in\n"; return 1; }
    if (o.has("sampling_steps") && !to_num(o.vals["sampling_steps"][0], sampling_steps)) { std::cerr << "bad value for --sampling_steps\n"; return 1; }
    if (o.has("sampling_frequency") && !to_num(o.vals["sampling_frequency"][0], sampling_frequency)) { std::cerr << "bad value for --sampling_frequency\n"; return 1; }
    if (o.has("steps_await") && !to_num(o.vals["steps_await"][0], steps_await)) { std::cerr << "bad value for --steps_await\n"; return 1; }
    if (o.has("epsilon") && !to_num(o.vals["epsilon"][0], epsilon)) { std::cerr << "bad value for --epsilon\n"; return 1; }
    if (o.has("cooling_schedule")) cooling_schedule = o.vals["cooling_schedule"][0];
    std::vector<float> kw(2, 0.f);  // reference: float_vec_t cooling_schedule_kwargs(2, 0)
    if (o.has("cooling_schedule_kwargs")) {
        kw.clear();
        for (auto& s : o.vals["cooling_schedule_kwargs"]) { float v; if (!to_num(s, v)) { std::cerr << "bad value for --cooling_schedule_kwargs\n"; return 1; } kw.push_back(v); }
        kw.resize(std::max<size_t>(kw.size(), 2), 0.f);
    }

    // schedule defaults / validation, reference src/mcmc_main.cc:134-218
    if (!o.has("cooling_schedule_kwargs")) {
        if (cooling_schedule == "exponential") { kw[0] = 1; kw[1] = 0.99f; }
        if (cooling_schedule == "linear") { kw[0] = (float)(sampling_steps + 1); kw[1] = 1; }
        if (cooling_schedule == "logarithmic") { kw[0] = 1; kw[1] = 1; }
        if (cooling_schedule == "constant") { kw[0] = 1; }
        if (cooling_schedule == "abrupt_cool") { kw[0] = (float)steps_await; }
    } else {
        if (cooling_schedule == "exponential") {
            if (kw[0] <= 0) { std::cerr << "Invalid cooling schedule argument for linear schedule: T_0 must be grater than 0.\nPassed value: T_0=" << kw[0] << "\n"; return 1; }
            if (kw[1] <= 0 || kw[1] >= 1) { std::cerr << "Invalid cooling schedule argument for exponential schedule: alpha must be in ]0,1[.\nPassed value: alpha=" << kw[1] << "\n"; return 1; }
        } else if (cooling_schedule == "linear") {
            if (kw[0] <= 0) { std::cerr << "Invalid cooling schedule argument for linear schedule: T_0 must be grater than 0.\nPassed value: T_0=" << kw[0] << "\n"; return 1; }
            if (kw[1] <= 0 || kw[1] > kw[0]) { std::cerr << "Invalid cooling schedule argument for linear schedule: eta must be in ]0, T_0].\nPassed value: T_0=" << kw[0] << ", eta=" << kw[1] << "\n"; return 1; }
            if (kw[1] * sampling_steps > kw[0]) { std::cerr << "Invalid cooling schedule argument for linear schedule: eta * sampling_steps must be smaller or equal to T_0.\nPassed value: eta*sampling_steps=" << kw[1] * sampling_steps << ", T_0=" << kw[0] << "\n"; return 1; }
        } else if (cooling_schedule == "logarithmic") {
            if (kw[0] <= 0) { std::cerr << "Invalid cooling schedule argument for logarithmic schedule: c must be greater than 0.\nPassed value: c=" << kw[0] << "\n"; return 1; }
            if (kw[1] <= 0) { std::cerr << "Invalid cooling schedule argument for logarithmic schedule: d must be greater than 0.\nPassed value: d=" << kw[1] << "\n"; return 1; }
        } else if (cooling_schedule == "constant") {
            if (kw[0] <= 0) { std::cerr << "Invalid cooling schedule argument for constant schedule: temperature must be greater than 0.\nPassed value: T=" << kw[0] << "\n"; return 1; }
        } else if (cooling_schedule == "abrupt_cool") {
            if (kw[0] <= 0) { std::cerr << "Invalid cooling schedule argument for abrupt_cool schedule: tau must be larger than 0. \nPassed value: tau=" << kw[0] << "\n"; return 1; }
        } else {
            std::cerr << "Invalid cooling schedule. Options are exponential, linear, logarithmic, abrupt_cool.\n";
            return 1;
        }
    }
    bool randomize = o.has("randomize");
    const bool merge = o.has("merge"), nature = o.has("nature");
    if (o.has("seed")) { if (!to_num(o.vals["seed"][0], seed)) { std::cerr << "bad value for --seed\n"; return 1; } }
    else seed = (size_t)std::chrono::high_resolution_clock::now().time_since_epoch().count();  // reference :236-239
    uint32_t gen_seed;
    if (o.has("gen_seed")) { size_t g; if (!to_num(o.vals["gen_seed"][0], g)) { std::cerr << "bad value for --gen_seed\n"; return 1; } gen_seed = (uint32_t)g; }
    else gen_seed = std::random_device()();  // reference src/blockmodel.hh:17-18
    size_t chains = 1, device = 0, max_inflight = 0;
    if (o.has("chains") && (!to_num(o.vals["chains"][0], chains) || chains == 0)) { std::cerr << "bad value for --chains\n"; return 1; }
    if (o.has("device") && !to_num(o.vals["device"][0], device)) { std::cerr << "bad value for --device\n"; return 1; }
    if (o.has("max_inflight") && !to_num(o.vals["max_inflight"][0], max_inflight)) { std::cerr << "bad value for --max_inflight\n"; return 1; }
    size_t gpus = 1;
    if (o.has("gpus") && (!to_num(o.vals["gpus"][0], gpus) || gpus == 0)) { std::cerr << "bad value for --gpus\n"; return 1; }
    std::vector<double> temps;
    size_t swap_every = 1;
    for (auto& s : o.get("tempering")) { double v; if (!to_num(s, v)) { std::cerr << "bad value for --tempering\n"; return 1; } temps.push_back(v); }
    if (o.has("swap_every") && (!to_num(o.vals["swap_every"][0], swap_every) || swap_every == 0)) { std::cerr << "bad value for --swap_every\n"; return 1; }
    if (!temps.empty()) {
        if (o.has("estimate")) { std::cerr << "--tempering does not combine with --estimate\n"; return 1; }
        if (merge || nature) { std::cerr << "--tempering does not combine with the agglomerative paths (-g / -u)\n"; return 1; }
        if (gpus > 1) { std::cerr << "--tempering runs on one GPU (no --gpus > 1)\n"; return 1; }
        if (!o.has("marginalize")) { std::cerr << "--tempering needs --marginalize\n"; return 1; }
        if (chains % temps.size()) { std::cerr << "--chains must be a multiple of the number of --tempering temperatures\n"; return 1; }
    }
    const bool align = o.has("align");
    if (align && !o.has("marginalize")) { std::cerr << "--align needs --marginalize\n"; return 1; }
    const bool coassign = o.has("coassign");
    if (coassign != o.has("coassign_out")) { std::cerr << "--coassign and --coassign_out go together\n"; return 1; }
    if (coassign && !o.has("marginalize")) { std::cerr << "--coassign needs --marginalize\n"; return 1; }
    std::vector<uint32_t> query;
    if (coassign) {
        std::string qerr;
        if (!read_query_nodes(o.vals["coassign"][0], NA + NB, query, qerr)) { std::cerr << qerr << "\n"; return 1; }
    }
    std::vector<uint64_t> co_sum;
    uint64_t co_counted = 0;
    const bool agreement = o.has("agreement_out");
    if (agreement) {
        if (gpus > 1) { std::cerr << "--agreement_out compares the chains of one GPU (no --gpus > 1)\n"; return 1; }
        if (chains < 2) { std::cerr << "--agreement_out needs --chains >= 2\n"; return 1; }
    }
    const bool modes = o.has("modes_out");
    if (modes) {
        if (!o.has("marginalize")) { std::cerr << "--modes_out needs --marginalize\n"; return 1; }
        if (gpus > 1) { std::cerr << "--modes_out finds the modes of one GPU's chains (no --gpus > 1)\n"; return 1; }
        if (chains < 2) { std::cerr << "--modes_out needs --chains >= 2\n"; return 1; }
    }
    uint32_t n_modes = 0;
    if (gpus > chains) gpus = chains;
    // stdout carries the label line and nothing else: whatever NCCL has to say (its version banner under NCCL_DEBUG)
    // goes to stderr unless the user chose a file
    if (gpus > 1) setenv("NCCL_DEBUG_FILE", "/dev/stderr", 0);

    // ---- initial memberships, reference src/mcmc_main.cc:243-326
    std::vector<unsigned> n, z, memberships_init;
    for (auto& s : o.get("n")) { unsigned v; if (!to_num(s, v)) { std::cerr << "bad value for -n\n"; return 1; } n.push_back(v); }
    for (auto& s : o.get("bisbm_partition")) { unsigned v; if (!to_num(s, v)) { std::cerr << "bad value for -z\n"; return 1; } z.push_back(v); }
    size_t KA = 0, KB = 0, N = 0;
    bool prepared = false;
    if (o.has("membership_path")) {
        std::clog << "Loading nodes' membership from membership_path.\n";
        std::ifstream f(o.vals["membership_path"][0].c_str());
        if (!f.is_open()) {
            std::clog << "WARNING: error in loading memberships, read memberships from block sizes\n";
        } else {
            std::string line;
            while (std::getline(f, line)) {  // reference src/graph_utilities.cc:5-18
                std::stringstream ls(line);
                size_t m = 0;
                ls >> m;
                memberships_init.push_back((unsigned)m);
            }
            randomize = false;
            unsigned max_ka = 0, max_kb = 0;
            for (size_t i = 0; i < memberships_init.size(); ++i) {
                if (i < y[0] && memberships_init[i] > max_ka) max_ka = memberships_init[i];
                if (memberships_init[i] > max_kb) max_kb = memberships_init[i];
            }
            z.assign(2, 0);
            z[0] = max_ka + 1; z[1] = max_kb - max_ka;
            prepared = true;
            N = memberships_init.size();
            KA = z[0]; KB = z[1];
            std::clog << " ---- read membership from file! ---- \n";
        }
    } else if (o.has("mb")) {
        std::vector<unsigned> mb;
        for (auto& s : o.vals["mb"]) { unsigned v; if (!to_num(s, v)) { std::cerr << "bad value for --mb\n"; return 1; } mb.push_back(v); }
        size_t accu = 0;
        for (unsigned v : n) accu += v;
        if (mb.size() != accu) {
            std::cerr << "[error] input vector size of memberships is different from the number of nodes \n";
            output_vec(mb, std::cerr);
            std::cerr << "#mb = " << mb.size() << "; while #nodes = " << accu << ". \n";
            return 1;
        }
        memberships_init = mb;
        if (z.size() < 2) { std::cerr << "number of partitions is required (-z flag)\n"; return 1; }
        KA = z[0]; KB = z[1];
        N = memberships_init.size();
        prepared = true;
    }
    if (!prepared) {
        if (!o.has("n")) { std::cerr << "n is required (-n flag) if one does not specify the membership of nodes\n"; return 1; }
        for (size_t r = 0; r < n.size(); ++r)
            for (unsigned i = 0; i < n[r]; ++i) memberships_init.push_back((unsigned)r);
        if (z.size() < 2) { std::cerr << "number of partitions is required (-z flag)\n"; return 1; }
        KA = z[0]; KB = z[1];
        N = memberships_init.size();
    }
    if (memberships_init.size() != NA + NB) {
        std::cerr << memberships_init.size() << ", " << NA + NB << '\n';
        std::cerr << "Types do not sum to the number of vertices!\n";
        return 1;
    }

    // ---- graph, reference src/graph_utilities.cc:20-49 (an unreadable file gives an empty graph there too): the file's bytes
    //      go to the library as they are -- parsed on the device (bisbm_create_from_text), no host-side edge vectors
    std::string edge_text;
    {
        std::ifstream f(edge_list_path.c_str(), std::ios::binary);
        if (f.is_open()) edge_text.assign(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
    }
    auto create_graph = [&](int dev, bisbm_handle** out) {
        return bisbm_create_from_text((uint32_t)NA, (uint32_t)NB, edge_text.data(), edge_text.size(), dev, out);
    };
    // ---- the agglomerative paths (reference src/mcmc_main.cc:350-451): -g starts from singleton blocks; initial labels
    //      whose block counts differ from -z are merged (or split) to (KA, KB).  One replay chain; every agg_merge and every
    //      anneal below is the reference's call with the reference's arguments.
    {
        size_t ka = 0, kb = 0;
        for (size_t t = 0; t < NA + NB; ++t) {
            if (t < NA && memberships_init[t] > ka) ka = memberships_init[t];
            else if (t >= NA && memberships_init[t] > kb) kb = memberships_init[t];
        }
        kb -= ka; ka += 1;
        if (merge) { for (size_t v = 0; v < N; ++v) memberships_init[v] = (unsigned)v; ka = NA; kb = NB; }
        int diff_a = (int)ka - (int)KA, diff_b = (int)kb - (int)KB;
        if (merge || diff_a != 0 || diff_b != 0) {
            if (chains != 1 || o.has("marginalize") || o.has("estimate") || agreement) {
                std::cerr << "the agglomerative paths run one chain (no --chains / --marginalize / --estimate / --agreement_out)\n";
                return 1;
            }
            if ((double)ka * (double)kb * 128.0 > 16e9) { std::cerr << "too many initial blocks for the K x K block matrix\n"; return 1; }
            bisbm_handle* h = nullptr;
            if (!check(create_graph((int)device, &h))) return 1;
            // room for the blocks a split adds
            if (!check(bisbm_set_option(h, "reserve_ka", (int64_t)std::max(ka, KA))) || !check(bisbm_set_option(h, "reserve_kb", (int64_t)std::max(kb, KB)))) return 1;
            const uint32_t ka1 = (uint32_t)ka, kb1 = (uint32_t)kb;
            std::vector<uint32_t> lab(memberships_init.begin(), memberships_init.end());
            if (!check(bisbm_set_chains(h, 1, &ka1, &kb1, lab.data(), epsilon))) return 1;
            if (!check(bisbm_replay_init(h, 0, (uint32_t)seed, gen_seed, 0))) return 1;
            const double sigma = 1.01;
            double rate = 0.0;
            uint64_t sweeps = 0;
            auto greedy_sweep = [&]() -> int {   // anneal(abrupt_cool, {0}, N, steps_await): one sweep at T = 0
                if (cooling_schedule != "abrupt_cool") { std::cerr << "Only abrupt cooling annealing is supported."; return 1; }
                return check(bisbm_replay_anneal(h, 0, BISBM_ABRUPT_COOL, 0.f, 0.f, N, steps_await, &rate, &sweeps)) ? 0 : 1;
            };
            uint32_t cka = ka1, ckb = kb1;
            if (merge && nature) {
                uint64_t n_edges = 0;
                if (!check(bisbm_info(h, nullptr, &n_edges, nullptr, nullptr))) return 1;
                const size_t ceiling = (size_t)std::ceil(std::sqrt(2.0 * (double)n_edges) / 2);
                size_t tKA = NA, tKB = NB, tGroups = NA + NB;
                while (tKA >= ceiling && tKB >= ceiling) {
                    if (!check(bisbm_replay_agg_merge_total(h, 0, (int)std::ceil((double)tGroups * (sigma - 1) / sigma), 10))) return 1;
                    if (!check(bisbm_chain_k(h, 0, &cka, &ckb))) return 1;
                    tKA = cka; tKB = ckb; tGroups = tKA + tKB;
                    if (greedy_sweep()) return 1;
                }
            } else if (merge || (diff_a >= 0 && diff_b >= 0)) {
                std::vector<int> ka_s, kb_s;
                geospace((int)ka, (int)KA, (int)kb, (int)KB, sigma, ka_s, kb_s);
                if (!merge && ka_s.size() == 1 && !check(bisbm_replay_agg_merge(h, 0, diff_a, diff_b, 10))) return 1;
                for (size_t i = 0; i + 1 < ka_s.size(); ++i) {
                    if (!check(bisbm_replay_agg_merge(h, 0, -(ka_s[i + 1] - ka_s[i]), -(kb_s[i + 1] - kb_s[i]), 10))) return 1;
                    if (i != ka_s.size() - 2 && greedy_sweep()) return 1;
                }
            } else {
                if (!check(bisbm_replay_agg_merge(h, 0, diff_a, diff_b, 100))) return 1;
            }
            // the final anneal is always abrupt_cool with the user's schedule arguments (src/mcmc_main.cc:397-398, 446-447)
            if (!check(bisbm_replay_anneal(h, 0, BISBM_ABRUPT_COOL, kw[0], kw[1], sampling_steps, steps_await, &rate, &sweeps))) return 1;
            double S = 0.0;
            std::vector<uint32_t> out(N);
            if (!check(bisbm_chain_k(h, 0, &cka, &ckb)) || !check(bisbm_entropy(h, 0, &S)) || !check(bisbm_get_labels(h, 0, out.data()))) return 1;
            std::clog << "(Ka, Kb) = (" << cka << ", " << ckb << ") \n";
            std::clog << "entropy: " << S << "\n";
            if (merge && nature) std::cout << cka << " " << ckb << " ";
            output_vec(out, std::cout);
            bisbm_destroy(h);
            return 0;
        }
    }

    int sched = -1;
    if (cooling_schedule == "exponential") sched = BISBM_EXPONENTIAL;
    if (cooling_schedule == "linear") sched = BISBM_LINEAR;
    if (cooling_schedule == "logarithmic") sched = BISBM_LOGARITHMIC;
    if (cooling_schedule == "constant") sched = BISBM_CONSTANT;
    if (cooling_schedule == "abrupt_cool") sched = BISBM_ABRUPT_COOL;

    if (gpus > 1 && !o.has("estimate")) {
        // ---- several GPUs of one node, one host thread per device: chain c runs on device (c mod gpus) with a seed that
        //      depends only on c; the graph is replicated.  --marginalize: one NCCL all-reduce of the histograms.
        const bool marg = o.has("marginalize");
        std::vector<bisbm_handle*> hs(gpus, nullptr);
        std::vector<std::string> errs(gpus);
        std::vector<std::vector<double>> ent(gpus), acc(gpus);
        std::vector<std::thread> th;
        for (size_t g = 0; g < gpus; ++g)
            th.emplace_back([&, g]() {
                auto ok = [&](int rc) { if (rc != BISBM_OK) { errs[g] = bisbm_last_error(); return false; } return true; };
                if (!ok(create_graph((int)(device + g), &hs[g]))) return;
                std::vector<size_t> ids;
                for (size_t c = g; c < chains; c += gpus) ids.push_back(c);
                const size_t nc = ids.size();
                std::vector<uint32_t> ka_v(nc, (uint32_t)KA), kb_v(nc, (uint32_t)KB), labels(nc * N);
                for (size_t i = 0; i < nc; ++i)
                    for (size_t v = 0; v < N; ++v) labels[i * N + v] = memberships_init[v];
                std::vector<uint64_t> seeds(nc);
                for (size_t i = 0; i < nc; ++i) seeds[i] = (uint64_t)seed * 0x9E3779B97F4A7C15ull + ids[i];
                if (!ok(bisbm_set_chains(hs[g], (uint32_t)nc, ka_v.data(), kb_v.data(), labels.data(), epsilon))) return;
                if (randomize && !ok(bisbm_randomize(hs[g], seeds.data()))) return;
                acc[g].assign(nc, 0.0); ent[g].assign(nc, 0.0);
                std::vector<uint64_t> sw(nc);
                if (marg) {
                    if (!ok(bisbm_marginals_clear(hs[g]))) return;
                    if (coassign && !ok(bisbm_coassign_set(hs[g], (uint32_t)query.size(), query.data()))) return;
                    // --align: the burn-in only; the reference is chosen over all devices before any sample
                    if (!ok(bisbm_marginalize(hs[g], burn_in, align ? 0 : sampling_steps, std::max<size_t>(sampling_frequency, 1), seeds.data(), (uint32_t)max_inflight))) return;
                    if (align && !ok(bisbm_entropy_all(hs[g], ent[g].data()))) return;
                } else {
                    if (sched >= 0 && !ok(bisbm_anneal(hs[g], sched, kw[0], kw[1], sampling_steps, steps_await, seeds.data(), (uint32_t)max_inflight, acc[g].data(), sw.data()))) return;
                    if (!ok(bisbm_entropy_all(hs[g], ent[g].data()))) return;
                }
            });
        for (auto& t : th) t.join();
        for (size_t g = 0; g < gpus; ++g)
            if (!errs[g].empty()) { std::cerr << "libbisbm (device " << device + g << "): " << errs[g] << "\n"; return 1; }
        std::vector<uint32_t> out(N);
        if (marg && align) {
            // one reference for every device -- the lowest-entropy chain after the burn-in -- so that the all-reduced
            // histogram is aligned to one partition; then the sampling sweeps
            size_t bg = 0, bi = 0;
            for (size_t g = 0; g < gpus; ++g)
                for (size_t i = 0; i < ent[g].size(); ++i)
                    if (ent[g][i] < ent[bg][bi]) { bg = g; bi = i; }
            if (!check(bisbm_get_labels(hs[bg], (uint32_t)bi, out.data()))) return 1;
            th.clear();
            for (size_t g = 0; g < gpus; ++g)
                th.emplace_back([&, g]() {
                    auto ok = [&](int rc) { if (rc != BISBM_OK) { errs[g] = bisbm_last_error(); return false; } return true; };
                    std::vector<uint64_t> seeds;
                    for (size_t c = g; c < chains; c += gpus) seeds.push_back((uint64_t)seed * 0x9E3779B97F4A7C15ull + c);
                    if (!ok(bisbm_marginals_align(hs[g], out.data()))) return;
                    ok(bisbm_marginalize(hs[g], 0, sampling_steps, std::max<size_t>(sampling_frequency, 1), seeds.data(), (uint32_t)max_inflight));
                });
            for (auto& t : th) t.join();
            for (size_t g = 0; g < gpus; ++g)
                if (!errs[g].empty()) { std::cerr << "libbisbm (device " << device + g << "): " << errs[g] << "\n"; return 1; }
        }
        if (marg) {
            // stdout carries the label line and nothing else: NCCL prints its version banner on stdout when the environment
            // sets NCCL_DEBUG (whatever NCCL_DEBUG_FILE says), so file descriptor 1 points at stderr while NCCL initialises
            std::cout.flush(); fflush(stdout);
            const int saved_stdout = dup(1);
            if (saved_stdout >= 0) dup2(2, 1);
            const bool ar_ok = check(bisbm_marginals_allreduce_local(hs.data(), (int)gpus));
            fflush(stdout);
            if (saved_stdout >= 0) { dup2(saved_stdout, 1); close(saved_stdout); }
            if (!ar_ok) return 1;
            if (!check(bisbm_marginal_argmax(hs[0], out.data()))) return 1;
            if (coassign) {
                for (size_t g = 0; g < gpus; ++g)
                    if (!check(add_coassign(hs[g], query.size(), co_sum, co_counted))) return 1;
                if (!write_coassign(o.vals["coassign_out"][0], query.size(), co_sum, co_counted)) return 1;
            }
            output_vec(out, std::cout);
        } else {
            size_t bg = 0, bi = 0;
            for (size_t g = 0; g < gpus; ++g)
                for (size_t i = 0; i < ent[g].size(); ++i)
                    if (ent[g][i] < ent[bg][bi]) { bg = g; bi = i; }
            if (!check(bisbm_get_labels(hs[bg], (uint32_t)bi, out.data()))) return 1;
            std::clog << "acceptance ratio " << acc[bg][bi] << "\n";
            std::clog << "(Ka, Kb) = (" << KA << ", " << KB << ") \n";
            std::clog << "entropy: " << ent[bg][bi] << "\n";
            output_vec(out, std::cout);
        }
        for (auto* h : hs) bisbm_destroy(h);
        return 0;
    }

    bisbm_handle* h = nullptr;
    if (!check(create_graph((int)device, &h))) return 1;
    std::vector<uint32_t> ka_v(chains, (uint32_t)KA), kb_v(chains, (uint32_t)KB), labels(chains * N);
    for (size_t c = 0; c < chains; ++c)
        for (size_t v = 0; v < N; ++v) labels[c * N + v] = memberships_init[v];
    if (!check(bisbm_set_chains(h, (uint32_t)chains, ka_v.data(), kb_v.data(), labels.data(), epsilon))) return 1;
    std::vector<uint64_t> seeds(chains);
    for (size_t c = 0; c < chains; ++c) seeds[c] = (uint64_t)seed * 0x9E3779B97F4A7C15ull + c;
    std::vector<uint32_t> out(N);

    if (o.has("marginalize") || o.has("estimate")) {
        // README modes: burn-in, then sampling at T = 1
        if (randomize && !check(bisbm_randomize(h, seeds.data()))) return 1;
        if (o.has("marginalize") && !temps.empty()) {
            // parallel tempering: burn-in without samples, then -t sweeps sampling the cold rung every -f sweeps
            const size_t f = std::max<size_t>(sampling_frequency, 1);
            if (!check(bisbm_marginals_clear(h)) || !check(bisbm_tempering_set(h, (uint32_t)temps.size(), temps.data(), nullptr))) return 1;
            if (coassign && !check(bisbm_coassign_set(h, (uint32_t)query.size(), query.data()))) return 1;
            if (burn_in && !check(bisbm_tempering_run(h, burn_in, swap_every, 0, seeds.data(), (uint64_t)seed, (uint32_t)max_inflight, nullptr))) return 1;
            if (align) {
                double S = 0.0;
                uint32_t best = 0;
                if (!check(lowest_entropy_chain(h, chains, true, &S, &best)) || !check(bisbm_get_labels(h, best, out.data())) ||
                    !check(bisbm_marginals_align(h, out.data()))) return 1;
            }
            if (modes && !check(set_modes(h, chains, N, true, &n_modes))) return 1;
            if (!check(bisbm_tempering_run(h, sampling_steps, swap_every, f, seeds.data(), (uint64_t)seed, (uint32_t)max_inflight, nullptr))) return 1;
            if (!check(bisbm_marginal_argmax(h, out.data()))) return 1;
            if (agreement && !write_agreement(h, chains, o.vals["agreement_out"][0])) return 1;
            if (modes && !write_modes(h, n_modes, N, o.vals["modes_out"][0])) return 1;
            if (coassign && (!check(add_coassign(h, query.size(), co_sum, co_counted)) ||
                             !write_coassign(o.vals["coassign_out"][0], query.size(), co_sum, co_counted))) return 1;
            output_vec(out, std::cout);
        } else if (o.has("marginalize")) {
            const size_t f = std::max<size_t>(sampling_frequency, 1);
            if (!check(bisbm_marginals_clear(h))) return 1;
            if (coassign && !check(bisbm_coassign_set(h, (uint32_t)query.size(), query.data()))) return 1;
            if (align || modes) {
                // burn-in, then the references chosen from the chains: the lowest-entropy chain every sample is aligned to
                // (--align), the modes every sample is sorted into (--modes_out); then the sampling sweeps
                if (!check(bisbm_marginalize(h, burn_in, 0, f, seeds.data(), (uint32_t)max_inflight))) return 1;
                if (align) {
                    double S = 0.0;
                    uint32_t best = 0;
                    if (!check(lowest_entropy_chain(h, chains, false, &S, &best)) || !check(bisbm_get_labels(h, best, out.data())) ||
                        !check(bisbm_marginals_align(h, out.data()))) return 1;
                }
                if (modes && !check(set_modes(h, chains, N, false, &n_modes))) return 1;
                if (!check(bisbm_marginalize(h, 0, sampling_steps, f, seeds.data(), (uint32_t)max_inflight))) return 1;
            } else if (!check(bisbm_marginalize(h, burn_in, sampling_steps, f, seeds.data(), (uint32_t)max_inflight))) return 1;
            if (!check(bisbm_marginal_argmax(h, out.data()))) return 1;
            if (agreement && !write_agreement(h, chains, o.vals["agreement_out"][0])) return 1;
            if (modes && !write_modes(h, n_modes, N, o.vals["modes_out"][0])) return 1;
            if (coassign && (!check(add_coassign(h, query.size(), co_sum, co_counted)) ||
                             !write_coassign(o.vals["coassign_out"][0], query.size(), co_sum, co_counted))) return 1;
            output_vec(out, std::cout);
        } else {
            // README "estimation": the number of groups is sampled too.  -z (or the membership file) gives the upper
            // bounds; blocks may empty and be re-populated ("vary_k"), and every printed sample carries the number of
            // OCCUPIED blocks and the log-likelihood (minus the description length).  --uni prints the 1D format
            // (K = Ka + Kb); the sampler itself keeps the bipartite constraint.
            if (!check(bisbm_set_option(h, "vary_k", 1))) return 1;
            std::vector<double> acc(chains);
            std::vector<uint64_t> sw(chains);
            std::vector<uint32_t> kk(2 * chains);
            if (burn_in && !check(bisbm_anneal(h, BISBM_CONSTANT, 1.f, 0.f, burn_in * N, std::numeric_limits<uint64_t>::max(), seeds.data(), (uint32_t)max_inflight, acc.data(), sw.data()))) return 1;
            const size_t f = std::max<size_t>(sampling_frequency, 1);
            const size_t n_samples = sampling_steps / f;
            const size_t first_printed = n_samples > 1000 ? n_samples - 1000 : 0;  // README: last 1000 samples
            for (size_t k = 0; k < n_samples; ++k) {
                if (!check(bisbm_anneal(h, BISBM_CONSTANT, 1.f, 0.f, f * N, std::numeric_limits<uint64_t>::max(), seeds.data(), (uint32_t)max_inflight, acc.data(), sw.data()))) return 1;
                if (k < first_printed) continue;
                double S = 0;
                if (!check(bisbm_entropy(h, 0, &S)) || !check(bisbm_get_labels(h, 0, out.data())) || !check(bisbm_occupied_blocks(h, kk.data()))) return 1;
                std::cout << (k + 1) * f << ",";
                if (o.has("uni")) std::cout << kk[0] + kk[1];
                else std::cout << kk[0] << "," << kk[1];
                std::cout << "," << -S;
                for (uint32_t x : out) std::cout << "," << x;
                std::cout << "\n";
            }
            if (agreement && !write_agreement(h, chains, o.vals["agreement_out"][0])) return 1;
        }
        bisbm_destroy(h);
        return 0;
    }

    double rate = 0.0, S = 0.0;
    if (chains == 1) {
        // the reference's straight path, bit for bit: shuffle_bisbm | init_bisbm, anneal, summary (:453-485)
        if (!check(bisbm_replay_init(h, 0, (uint32_t)seed, gen_seed, randomize ? 1 : 0))) return 1;
        if (sched >= 0) {
            uint64_t sweeps = 0;
            if (!check(bisbm_replay_anneal(h, 0, sched, kw[0], kw[1], sampling_steps, steps_await, &rate, &sweeps))) return 1;
        }
        if (!check(bisbm_entropy(h, 0, &S)) || !check(bisbm_get_labels(h, 0, out.data()))) return 1;
    } else {
        // many restarts in one launch; print the chain with the smallest description length
        if (randomize && !check(bisbm_randomize(h, seeds.data()))) return 1;
        std::vector<double> acc(chains), ent(chains);
        std::vector<uint64_t> sw(chains);
        if (sched >= 0 && !check(bisbm_anneal(h, sched, kw[0], kw[1], sampling_steps, steps_await, seeds.data(), (uint32_t)max_inflight, acc.data(), sw.data()))) return 1;
        if (!check(bisbm_entropy_all(h, ent.data()))) return 1;
        size_t best = 0;
        for (size_t c = 1; c < chains; ++c) if (ent[c] < ent[best]) best = c;
        rate = acc[best]; S = ent[best];
        if (!check(bisbm_get_labels(h, (uint32_t)best, out.data()))) return 1;
        if (agreement && !write_agreement(h, chains, o.vals["agreement_out"][0])) return 1;
    }
    std::clog << "acceptance ratio " << rate << "\n";
    std::clog << "(Ka, Kb) = (" << KA << ", " << KB << ") \n";  // blockmodel_t::summary, reference src/blockmodel.cc:748-751
    std::clog << "entropy: " << S << "\n";
    output_vec(out, std::cout);
    bisbm_destroy(h);
    return 0;
}
