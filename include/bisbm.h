/* include/bisbm.h -- C ABI of libbisbm.so: the B200-native Metropolis-Hastings sweep of the
 * degree-corrected bipartite SBM.
 *
 * This is the drop-in boundary for ONE path of junipertcy/bipartiteSBM-MCMC: the simulated
 * annealing / sampling loop  metropolis_hasting::anneal -> step -> {single_vertex_change,
 * transition_ratio, apply_mcmc_moves}.  The reference exposes no FFI; the entry points
 * below are what a binding for that path would bind, each citing the reference interface
 * it replaces (paths under the reference tree).  Plain C types only; the caller owns
 * every host buffer, the handle owns all device memory; every call returns 0 on success
 * and a non-zero code otherwise (bisbm_last_error() gives the message); nothing aborts.
 * There is no CPU fallback: without a CUDA device every compute call fails with
 * BISBM_ERR_CUDA.
 *
 * Two execution modes over the same device-resident state:
 *   replay   -- one chain, strictly sequential, consuming the reference's two mt19937
 *               streams (`engine`, `gen`) through libstdc++-exact distribution transforms;
 *               reproduces the reference's label trajectory, m_rs, e_r, n_r bit for bit.
 *   parallel -- many independent chains per launch (lane = chain, chain-minor labels),
 *               counter-based RNG, type-alternating half sweeps; statistically
 *               equivalent, not draw-for-draw identical.
 */
#ifndef BISBM_H
#define BISBM_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bisbm_handle bisbm_handle;

enum {
    BISBM_OK = 0,
    BISBM_ERR_ARG = 1,    /* invalid argument / inconsistent sizes */
    BISBM_ERR_CUDA = 2,   /* CUDA runtime error (incl. no device) */
    BISBM_ERR_STATE = 3,  /* call out of order (e.g. anneal before set_chains) */
    BISBM_ERR_ALLOC = 4
};

/* cooling schedules, reference src/metropolis_hasting.cc:10-37 and src/mcmc_main.cc:463-482 */
enum {
    BISBM_EXPONENTIAL = 0, /* p0 * pow(p1, t)                    */
    BISBM_LINEAR = 1,      /* p0 - p1 * t            (float)     */
    BISBM_LOGARITHMIC = 2, /* p0 / log(trunc(t + p1))            */
    BISBM_CONSTANT = 3,    /* p0                                 */
    BISBM_ABRUPT_COOL = 4  /* t < p0 ? 1 : 0                     */
};

const char* bisbm_last_error(void);
/* library version string; also proves the library loaded */
const char* bisbm_version(void);

/* ---- graph -------------------------------------------------------------------------
 * Replaces edge_to_adj + the adjacency part of the blockmodel_t constructor
 * (src/graph_utilities.cc:36-49, src/blockmodel.cc:15-75).  Node ids 0..na-1 are type a,
 * na..na+nb-1 type b (src/mcmc_main.cc:121-130).  Edges are (ea[i], eb[i]) in FILE ORDER;
 * the adjacency keeps that order and multi-edges, as the reference does. */
int bisbm_create(uint32_t na, uint32_t nb, uint64_t n_edges, const uint32_t* ea, const uint32_t* eb,
                 int device, bisbm_handle** out);
/* Same, from the TEXT of an edge-list file (load_edge_list, src/graph_utilities.cc:20-34: one edge per line, two unsigned
 * integers separated by blanks).  The text is copied to the device once and parsed there (line starts per 4 KB chunk ->
 * exclusive scan -> parse at the line start), and the edge arrays go straight into the device-side CSR build: no host-side
 * edge vectors.  Lines whose first token is not a number are skipped; a missing second number reads as 0. */
int bisbm_create_from_text(uint32_t na, uint32_t nb, const char* text, uint64_t n_bytes, int device, bisbm_handle** out);
/* the graph as the library holds it: row_ptr[n+1] and col_idx[2E] (either may be NULL), rows in the reference's adjacency order */
int bisbm_get_csr(bisbm_handle* h, uint32_t* row_ptr, uint32_t* col_idx);
/* Same, from a ready CSR (row_ptr[n+1], col_idx[2E]) whose rows are already in the
 * reference's adjacency order. */
int bisbm_create_csr(uint32_t na, uint32_t nb, const uint32_t* row_ptr, const uint32_t* col_idx,
                     int device, bisbm_handle** out);
int bisbm_destroy(bisbm_handle* h);
/* A second handle over the SAME device-resident graph (ref-counted, read only): its own chains, stream and options.
 * This is how several pools of chains -- e.g. one per K class of a (Ka, Kb) grid -- run over one copy of the graph. */
int bisbm_share_graph(bisbm_handle* src, bisbm_handle** out);

/* ---- chains ------------------------------------------------------------------------
 * Replaces the blockmodel_t state + init_bisbm (src/blockmodel.hh:92-143,
 * src/blockmodel.cc:681-746).  labels[c*n + v] is chain c's GLOBAL block id of node v
 * (type-a blocks 0..ka[c]-1, type-b blocks ka[c]..ka[c]+kb[c]-1).  Builds n_r, e_r, m_rs,
 * eta_rk on the device.  eps is the reference's epsilon (-E). */
int bisbm_set_chains(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb,
                     const uint32_t* labels, double eps);
/* The same with 8-bit labels (global block ids, needs ka[c] + kb[c] <= 256): a quarter of the host <-> device bytes. */
int bisbm_set_chains_u8(bisbm_handle* h, uint32_t n_chains, const uint32_t* ka, const uint32_t* kb,
                        const uint8_t* labels, double eps);
/* Both forms compare the incoming labels with the ones the handle already holds (same chain count, K and epsilon): when
 * nothing changed -- a caller handing back what it read, e.g. after a checkpoint -- the counts are kept, not rebuilt. */
/* Parallel-mode --randomize: permutes each chain's labels within type a and within
 * type b with a counter-based RNG keyed by seeds[c] (same block sizes as shuffle_bisbm,
 * src/blockmodel.cc:672-679, different stream), then rebuilds the counts. */
int bisbm_randomize(bisbm_handle* h, const uint64_t* seeds);

/* ---- replay mode (one chain, bit-exact) ----------------------------------------------
 * Seeds the two engines of the reference: `engine` (src/mcmc_main.cc:242) and `gen`
 * (src/blockmodel.hh:17-18), resets vlist to identity (src/blockmodel.cc:41) and, if
 * randomize != 0, runs shuffle_bisbm with `engine` (src/blockmodel.cc:672-679). */
int bisbm_replay_init(bisbm_handle* h, uint32_t chain, uint32_t engine_seed, uint32_t gen_seed, int randomize);
/* metropolis_hasting::anneal (src/metropolis_hasting.cc:64-101) with the reference's
 * float-typed schedule parameters; duration is in single-vertex steps. */
int bisbm_replay_anneal(bisbm_handle* h, uint32_t chain, int schedule, float p0, float p1, uint64_t duration,
                        uint64_t steps_await, double* accept_ratio, uint64_t* sweeps_done);
/* metropolis_hasting::step on one vertex at temperature T (src/metropolis_hasting.cc:42-62) */
int bisbm_replay_step(bisbm_handle* h, uint32_t chain, uint32_t v, double T, int* accepted);
/* metropolis_hasting::transition_ratio for moving v to global block s
 * (src/metropolis_hasting.cc:103-192); accu_r is the member left by the call. */
int bisbm_replay_transition(bisbm_handle* h, uint32_t chain, uint32_t v, uint32_t s, double* dS, double* accu_r);
int bisbm_replay_get_vlist(bisbm_handle* h, uint32_t chain, uint32_t* vlist);
int bisbm_replay_rng_words(bisbm_handle* h, uint32_t chain, uint64_t* engine_words, uint64_t* gen_words);

/* ---- agglomerative merge / split of a replay chain (the initialiser of the reference's -g / -u paths and of initial labels
 * whose block counts differ from -z, src/mcmc_main.cc:350-451) ------------------------------
 * blockmodel_t::agg_merge(engine, diff_a, diff_b, nm) (src/blockmodel.cc:109-204): diff_a (diff_b) type-a (type-b) blocks
 * fewer; nm block-move proposals per block (single_block_change, :639-669), consumed from the chain's two engines exactly as
 * the reference does; the proposals with the smallest description-length change (compute_dS, :335-370) are applied
 * (apply_block_moves, :505-553: blocks renumbered in order of first appearance, counts rebuilt).  A negative diff splits:
 * agg_split (:555-611), one new block of that type per unit.  Afterwards the chain has bisbm_chain_k blocks; the pool's
 * strides (the maxima given to bisbm_set_chains) stay, so a split needs a pool created with room for the new block.
 * Merge path: labels, counts and RNG word counts bit-identical to the reference (tests/test_merge_gpu.py).  Split path:
 * the reference's compute_dS(mb, split_move) indexes a vector out of bounds (undefined behaviour); this library implements
 * the evident intent and its parity is property-tested only. */
int bisbm_replay_agg_merge(bisbm_handle* h, uint32_t chain, int diff_a, int diff_b, uint32_t nm);
/* blockmodel_t::agg_merge(engine, diff, nm) (src/blockmodel.cc:206-256), the -u / --nature form: diff merges of any type; a
 * round that ends on an infinite candidate is redone with fresh proposals. */
int bisbm_replay_agg_merge_total(bisbm_handle* h, uint32_t chain, int diff, uint32_t nm);
/* blockmodel_t::get_KA / get_KB of one chain (they change under agg_merge) */
int bisbm_chain_k(bisbm_handle* h, uint32_t chain, uint32_t* ka, uint32_t* kb);

/* ---- parallel mode (all chains per launch) -------------------------------------------
 * anneal for every chain at once.  duration / steps_await as in the reference (steps);
 * seeds[c] keys chain c's counter-based RNG.  max_inflight bounds how many moves of ONE
 * chain may be evaluated concurrently against slightly stale block counts (0 = let the
 * library fill the GPU; 1 = strictly sequential chains).  Outputs per chain. */
int bisbm_anneal(bisbm_handle* h, int schedule, float p0, float p1, uint64_t duration, uint64_t steps_await,
                 const uint64_t* seeds, uint32_t max_inflight, double* accept_ratio, uint64_t* sweeps_done);
/* Marginalisation (README "marginalization" mode; no code in the reference snapshot):
 * burn_in sweeps at T=1, then `sweeps` sweeps sampling every `every` sweeps into the
 * device-resident per-node label histogram uint32[n][hist_width] (summed over chains). */
int bisbm_marginalize(bisbm_handle* h, uint64_t burn_in, uint64_t sweeps, uint64_t every, const uint64_t* seeds,
                      uint32_t max_inflight);
int bisbm_marginals_clear(bisbm_handle* h);
/* adds ONE sample of every chain's current labels to the histogram (asynchronous on the handle's stream) */
int bisbm_marginal_sample(bisbm_handle* h);
/* Label alignment of the marginals (SURVEY H9; no counterpart in the reference).  Block ids mean nothing across chains: a
 * chain started from a randomised partition, or one that exchanged two blocks on its way, calls a group "block 3" that
 * its neighbours call "block 1", and the summed histogram mixes unrelated groups.  ref_labels[n]: a partition in the
 * pool's global numbering (type-a ids < ka, type-b ids in [ka, ka + kb)), e.g. what bisbm_get_labels or
 * bisbm_marginal_argmax return.  While a reference is set, every marginal sample (bisbm_marginal_sample,
 * bisbm_marginalize, bisbm_tempering_run's rung-0 samples) first relabels each chain, within each type, by the
 * permutation of its blocks that maximises the number of nodes whose block agrees with the reference.  Among maximal
 * permutations it takes the one with the most fixed points, so a chain equal to the reference keeps its labels (and, in
 * estimate mode, "vary_k", empty blocks stay where they are); any remaining tie is broken deterministically (the same
 * overlaps always give the same permutation), so an aligned run is as reproducible as an unaligned one.  The chains themselves are not touched.  NULL clears the reference.
 * The reference's node order is sorted and uploaded here; a sample queues its kernels on the handle's stream with no host
 * synchronisation.  bisbm_set_chains* clears the reference, and so does a replay merge / split that changes a chain's
 * (ka, kb); bisbm_randomize and bisbm_marginals_clear keep it, so a caller
 * can marginalise, set the reference to the arg-max, clear and marginalise again.  Multi-GPU: set the same reference on
 * every handle (or rank) before sampling, and the all-reduced histogram is aligned to that one partition.
 * Errors: BISBM_ERR_ARG for a null handle, a pool whose chains differ in (ka, kb), a reference label outside its node's
 * type range, or more blocks per type than the device's shared memory per block holds (about 1700); BISBM_ERR_STATE for a
 * histogram of another width than ka + kb (left from a pool of other K: bisbm_marginals_clear first). */
int bisbm_marginals_align(bisbm_handle* h, const uint32_t* ref_labels);
/* the permutations the last aligned sample used: map[c * (ka + kb) + g] = the global id chain c's block g was counted as
 * ([n_chains][ka + kb], computed for every chain, also those a tempering sample skips).  BISBM_ERR_STATE before any aligned
 * sample under the current reference. */
int bisbm_marginals_alignment(bisbm_handle* h, uint32_t* map);
/* ---- parallel tempering (replica exchange; no counterpart in the reference) ----------------------------------------
 * Ladder: n_rungs = R temperatures temps[0..R-1], each finite and > 0, non-decreasing; rung 0 is the cold one.  n_chains
 * must be a multiple of R: chains l R .. l R + R - 1 form ladder l, and chain l R + i starts at rung i unless rung_of_chain
 * is given (e.g. resuming from a checkpoint).  A swap exchanges the RUNGS of two chains of one ladder -- never their labels
 * or counts.  A swap round follows every swap_every full sweeps; round k of a ladder proposes the pairs (i, i+1) with
 * i = k (mod 2) (deterministic even-odd scheme), each accepted with probability min(1, exp((beta_i - beta_{i+1})(S_i -
 * S_{i+1}))), S = entropy() of the chain's current state (in estimate mode, "vary_k", with the occupied block counts, as
 * bisbm_entropy* use).  The uniform draw is Philox keyed by (swap_seed, ladder, round), a stream of its own.  The round
 * counter lives on the handle: consecutive runs neither repeat draws nor restart the parity.  Per sweep of a run: full
 * sweep -> swap round if due -> marginal sample of the rung-0 chains if due.  S, the rung maps and 1/T stay on the device;
 * a run makes no host synchronisation per round.
 * bisbm_anneal, bisbm_marginalize, bisbm_grid_search and bisbm_parallel_transition ignore any ladder.  bisbm_set_chains*
 * clears it; bisbm_randomize keeps it.  Errors: BISBM_ERR_ARG for R not dividing n_chains, a temperature <= 0, NaN,
 * infinite or decreasing, a bad rung permutation, swap_every == 0; BISBM_ERR_STATE for a run or stats call without a ladder.
 * The counters persist until the next bisbm_tempering_set; bisbm_last_timing and bisbm_sweep_launches report a run like any
 * other parallel call. */
/* n_rungs = 0 clears the ladder; rung_of_chain may be NULL (identity), else each ladder's entries are a permutation of 0..R-1 */
int bisbm_tempering_set(bisbm_handle* h, uint32_t n_rungs, const double* temps, const uint32_t* rung_of_chain);
/* sample_every = 0: no marginal samples; accept_ratio[c] = accepted moves / (sweeps x N) of this run (may be NULL) */
int bisbm_tempering_run(bisbm_handle* h, uint64_t sweeps, uint64_t swap_every, uint64_t sample_every,
                        const uint64_t* seeds, uint64_t swap_seed, uint32_t max_inflight, double* accept_ratio);
/* any pointer may be NULL.  rung_of_chain[n_chains]; swaps_tried / swaps_accepted[R-1] per adjacent pair (summed over
 * ladders); moves_tried / moves_accepted[R] per rung (a chain's moves are attributed to the rung it held while making them);
 * round_trips[n_ladders] (rung 0 -> rung R-1 -> rung 0 journeys completed by any chain of the ladder) */
int bisbm_tempering_stats(bisbm_handle* h, uint32_t* rung_of_chain, uint64_t* swaps_tried, uint64_t* swaps_accepted,
                          uint64_t* moves_tried, uint64_t* moves_accepted, uint64_t* round_trips);
/* Arithmetic of the parallel sweep's per-move evaluation (dS, Hastings factor, accept test).  The reference
 * computes transition_ratio in double (src/metropolis_hasting.cc:103-192) and so does parallel mode by default
 * (BISBM_PRECISION_FP64).  BISBM_PRECISION_FP32 evaluates the move in fp32 on the MUFU unit (|error of the log
 * acceptance ratio| <~ 2e-5); counts and commits stay exact integers either way.  Replay mode is always strict double. */
enum { BISBM_PRECISION_FP32 = 0, BISBM_PRECISION_FP64 = 1 };
int bisbm_set_precision(bisbm_handle* h, int mode);
/* Tuning options of the parallel sweep (no environment variables are read):
 *   "inflight_div"  default in-flight bound of bisbm_anneal(max_inflight = 0) = half sweep / value (default 64)
 *   "kernel"        -1 automatic; 0 force the round-1 kernel (double, counts in L2); 5 force sweep2 with counts in L2
 *                   (the kernels the automatic choice takes for hubs and for large K); other values are rejected
 *   "generic"       1: never take the Ka = Kb = 32 compile-time specialisation
 *   "spare_sms"     0: do not hand the SMs that n_groups x ctas_per_group leaves idle to the chain groups in turn (default 1;
 *                   only with max_inflight = 0: a group holding a spare CTA evaluates one more CTA's worth of moves per launch)
 *   "vary_k"        1: estimate mode (README "estimation", no code in the reference snapshot): blocks may empty and be
 *                   re-populated by the uniform part of the proposal (no "would empty block r" veto), the K-dependent
 *                   terms of the description length enter dS with the number of OCCUPIED blocks, and bisbm_entropy*
 *                   use the occupied counts too.  ka / kb of bisbm_set_chains are then upper bounds.
 *   "reserve_ka" / "reserve_kb"   minimum count-array strides of the NEXT bisbm_set_chains: room for blocks that
 *                   bisbm_replay_agg_merge with a negative diff (agg_split) adds to a chain */
int bisbm_set_option(bisbm_handle* h, const char* name, int64_t value);
/* which sweep kernel the last parallel call launched and how the half sweep was cut:
 * kernel 0 = round-1 sweep_kernel (double, counts in L2: hubs of degree > 255, K > 256 per type);
 * 2 / 3 = sweep2_kernel<float / double>, counts staged in shared memory (3 is the default);
 * 4 / 5 = sweep2_kernel<float / double>, counts in L2 (K too large for shared memory);
 * ids 1, 6 and 7 (the retired round-1 staged kernel and sweep2's thread-block-cluster form) are no longer produced;
 * slice = vertices of the visiting order per launch (the staleness bound between CTAs of one chain group) */
int bisbm_sweep_info(bisbm_handle* h, int* kernel, uint32_t* warps_per_cta, uint32_t* ctas_per_group, uint32_t* slice);
/* transition_ratio (src/metropolis_hasting.cc:103-192) for moving v to global block s in chain `chain`, evaluated by the
 * PARALLEL sweep kernel's own device code (one forced proposal through sweep2_kernel, nothing committed): dS and
 * log(accu_r) in the handle's current precision.  Cross-type targets give dS = +inf (log_accu NaN), s == r gives 0, 0. */
int bisbm_parallel_transition(bisbm_handle* h, uint32_t chain, uint32_t v, uint32_t s, double* dS, double* log_accu);
/* det_k_bisbm-style model selection in process (the caller of bin/mcmc named by reference README.md:7, one subprocess and
 * one 800 MB q-cache build per grid point there): n_points (Ka, Kb) pairs x `restarts` randomised restarts are annealed
 * as parallel chains -- bucketed by K class so that small-K chains keep the staged kernel -- and scored by entropy()
 * (src/blockmodel.cc:753-787).  Initial partitions: equal-size blocks in node order (reference `-n`), then randomised.
 * entropy / accept: [n_points * restarts], chain p * restarts + q; best_chain: index of the minimum; best_labels: [n]
 * global block ids of that chain (may be NULL); stats (may be NULL): {moves attempted, device ms, K buckets, best entropy}.
 * The buckets' pools (labels, counts) stay allocated on the graph handle for the next call with the same grid -- freeing and
 * re-allocating gigabytes per call cost more than the annealing -- unless less than a quarter of the device memory would stay
 * free; bisbm_grid_release (or bisbm_destroy of the graph handle) frees them. */
int bisbm_grid_search(bisbm_handle* graph, uint32_t n_points, const uint32_t* ka, const uint32_t* kb, uint32_t restarts,
                      double eps, int schedule, float p0, float p1, uint64_t duration, uint64_t steps_await, uint64_t seed,
                      uint32_t max_inflight, double* entropy, double* accept, uint32_t* best_chain, uint32_t* best_labels,
                      double* stats);
int bisbm_grid_release(bisbm_handle* graph);
/* the K bucket bisbm_grid_search puts a (ka, kb) point in: the bucket's (KA, KB) strides and whether its counts are staged in
 * shared memory (1) or stay in L2 (0, several times slower per move) -- what a caller needs to deal the points of a grid to
 * several GPUs in whole 32-chain groups of equal cost (host.py grid_partition) */
int bisbm_grid_k_class(const bisbm_handle* graph, uint32_t ka, uint32_t kb, uint32_t* KA, uint32_t* KB, int* staged);
/* per K bucket (= pool over the shared graph) of the last bisbm_grid_search on this graph handle, in the order they ran:
 * rows[i][8] = {KA stride, KB stride, chains, kernel id (bisbm_sweep_info), set-up ms (pool, initial partitions, counts,
 * randomise; host clock), anneal ms (device events), anneal ms (host clock), scoring + teardown ms (host clock)}.
 * n_rows = buckets of that call (may exceed max_rows; only max_rows rows are written). */
int bisbm_grid_search_report(const bisbm_handle* graph, uint32_t max_rows, double* rows, uint32_t* n_rows);
/* ---- multi-GPU: chains are partitioned over GPUs (graph replicated); the only collective is ONE all-reduce (sum, uint32)
 * of the per-node marginal histogram over NVLink.  libnccl.so.2 is loaded on first use (BISBM_ERR_STATE if absent).
 * One process per GPU: rank 0 calls bisbm_nccl_get_unique_id and hands the 128 bytes to the other ranks by any means;
 * every rank calls bisbm_nccl_init (collective), then bisbm_marginals_allreduce (collective, in place, on the handle's
 * stream; returns when the sum is complete).  One process driving several GPUs: bisbm_marginals_allreduce_local over its
 * handles (one per device). */
int bisbm_nccl_get_unique_id(uint8_t* id128);
int bisbm_nccl_init(bisbm_handle* h, int nranks, int rank, const uint8_t* id128);
int bisbm_marginals_allreduce(bisbm_handle* h);
int bisbm_marginals_allreduce_local(bisbm_handle** handles, int n);
/* device pointer + element count of the histogram (for callers that bring their own collective) */
int bisbm_marginals_device(bisbm_handle* h, void** dev_ptr, uint64_t* n_elems, uint32_t* width);
int bisbm_get_marginals(bisbm_handle* h, uint32_t* hist);          /* [n][width], global block ids */
int bisbm_marginal_argmax(bisbm_handle* h, uint32_t* labels);      /* [n] */
/* device-side sweep timing of the last parallel call: total kernel ms (CUDA events on the
 * handle's stream), kernel launches, and single-vertex moves attempted */
int bisbm_last_timing(bisbm_handle* h, double* sweep_ms, uint64_t* launches, uint64_t* moves);
/* of those launches, how many were the sweep kernel itself (one per slice of a half sweep) */
int bisbm_sweep_launches(bisbm_handle* h, uint64_t* sweep_kernel_launches);
/* stream the handle launches on (cudaStream_t as void*) */
int bisbm_stream(bisbm_handle* h, void** stream);

/* ---- state read-back (getters of blockmodel_t, src/blockmodel.hh:35-53) ---------------- */
int bisbm_info(bisbm_handle* h, uint32_t* n, uint64_t* n_edges, uint32_t* max_degree, uint32_t* n_chains);
int bisbm_get_labels(bisbm_handle* h, uint32_t chain, uint32_t* labels);          /* [n] global ids */
int bisbm_get_all_labels(bisbm_handle* h, uint32_t* labels);                     /* [n_chains][n] */
int bisbm_get_all_labels_u8(bisbm_handle* h, uint8_t* labels);                   /* [n_chains][n], ka + kb <= 256 */
int bisbm_get_m(bisbm_handle* h, uint32_t chain, int32_t* m);                    /* [K][K] symmetric */
int bisbm_get_m_r(bisbm_handle* h, uint32_t chain, int32_t* e_r);                /* [K] */
int bisbm_get_n_r(bisbm_handle* h, uint32_t chain, int32_t* n_r);                /* [K] */
int bisbm_get_eta(bisbm_handle* h, uint32_t chain, uint32_t* eta);               /* [K][max_degree+1] */
/* blockmodel_t::entropy (src/blockmodel.cc:753-787), evaluated on the device */
int bisbm_entropy(bisbm_handle* h, uint32_t chain, double* entropy);
int bisbm_entropy_all(bisbm_handle* h, double* entropy);                         /* [n_chains] */
/* number of non-empty blocks per type of every chain: ka_kb[2c], ka_kb[2c+1] (estimate mode's Ka, Kb columns) */
int bisbm_occupied_blocks(bisbm_handle* h, uint32_t* ka_kb);
/* blockmodel_t::get_entropy: running sum of accepted dS (src/blockmodel.hh:100) */
int bisbm_entropy_accum(bisbm_handle* h, uint32_t chain, double* entropy_accum);

#ifdef __cplusplus
}
#endif
#endif
