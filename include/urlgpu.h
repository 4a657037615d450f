/*
 * urlgpu.h — C ABI of the B200-native local-score engine (liburlgpu.so).
 *
 * This is the drop-in boundary for the local-score hot path of ninalu/urlearning-cpp.  All entry
 * points are extern "C", take plain pointers and sizes, return 0 on success and a negative
 * urlgpu_status on error (message via urlgpu_last_error).  There is NO CPU fallback: every scoring
 * entry point fails with URLGPU_ERR_CUDA when no sm_100 device is usable.
 *
 * What each entry point replaces in the reference (paths relative to /root/reference/urlearning/):
 *
 *   urlgpu_set_discrete      ADTree::initialize/createTree            ad_tree/ad_tree.cpp:17-31
 *                            BayesianNetwork::getConsistentRecords    base/bayesian_network.cpp:146-169
 *                            LogLikelihoodCalculator::getLogCache     scoring_function/log_likelihood_calculator.h:30-38
 *                            BICScoringFunction ctor                  scoring_function/bic_scoring_function.cpp:11-18
 *   urlgpu_set_continuous    BIC_OLS_Function ctor (standardise)      scoring_function/BIC_OLS.cpp:30-123
 *   urlgpu_score_variable    ScoreCalculator::calculateScores         scoring_function/score_calculator.cpp:33-135
 *                            (+ the per-set ScoringFunction::calculateScore calls it makes,
 *                               scoring_function/scoring_function.h:19; bic_scoring_function.cpp:32-76;
 *                               BIC_OLS.cpp:174-389; log_likelihood_calculator.cpp:22-77; ad_tree.cpp:95-164)
 *                            and, with URLGPU_PRUNE_DOMINATED, ScoreCalculator::prune
 *                                                                     scoring_function/score_calculator.cpp:150-197
 *   urlgpu_score_one         ScoringFunction::calculateScore          scoring_function/scoring_function.h:19
 *   urlgpu_contingency       ADTree::makeContab                       ad_tree/ad_tree.cpp:95-137
 *   urlgpu_spg_build/query   SparseParentBitwise::initialize/getScore  score_cache/sparse_parent_bitwise.cpp:24-110
 *   urlgpu_order_search      run_astar_on_one_scc (order-graph search) astar/astar_main.cpp:216-546
 *   urlgpu_order_search_layered  the same, for components of up to 36 variables
 *   urlgpu_order_local_search    (no counterpart: insertion hill climbing over the same orders, components of up to 256)
 *   urlgpu_order_local_search_sparse  the same climb, with SparseParentList::getScore inside the climb
 *                                                                     score_cache/sparse_parent_list.cpp:44-55
 *   urlgpu_prune             ScoreCalculator::prune                   scoring_function/score_calculator.cpp:150-197
 *   urlgpu_result_*          FloatMap iteration in scoringThread      score/score_main.cpp:187-200, base/typedefs.h:816
 *
 * varsets: the reference's varset is one uint64_t (base/typedefs.h:469,650).  Here a varset is
 * `mask_words` little-endian uint64_t words (bit i of word i/64 = variable i), so p may exceed 63.
 */
#ifndef URLGPU_H
#define URLGPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct urlgpu_ctx urlgpu_ctx;
typedef struct urlgpu_result urlgpu_result;

typedef enum {
    URLGPU_OK = 0,
    URLGPU_ERR_ARG = -1,      /* bad argument / call order */
    URLGPU_ERR_CUDA = -2,     /* CUDA runtime error or no usable device */
    URLGPU_ERR_LIMIT = -3,    /* problem exceeds an engine limit (candidate count, table size, memory) */
    URLGPU_ERR_INTERNAL = -4
} urlgpu_status;

/* URLGPU_FNML: factorized NML on the same counts as BIC (scoring_function/fnml_scoring_function.{h,cpp}: log-likelihood
 * minus sum_j log C(N_ij, r_v), no BIC penalty and no log-bound on the parent limit); needs urlgpu_set_discrete.
 * URLGPU_BDEU: BDeu on the same counts (scoring_function/bdeu_scoring_function.cpp:25-123, deCampos pruning off); the
 * `lambda` argument of the scoring calls carries the equivalent sample size (score_main.cpp -e, default 1). */
typedef enum { URLGPU_BIC = 0, URLGPU_CBIC = 1, URLGPU_FNML = 2, URLGPU_BDEU = 3 } urlgpu_score_t;

/* filter_flags of urlgpu_score_variable (bit set) */
enum {
    URLGPU_KEEP_ALL = 0,          /* store rule of the shipped `score` only (score_calculator.cpp:59,111; BIC_OLS.cpp:213-249) */
    URLGPU_PRUNE_DOMINATED = 2,   /* additionally drop S if a stored subset scores at least as well (score_calculator.cpp:150-197) */
    URLGPU_CBIC_NO_ACCEPT = 4,    /* cBIC: skip the in-line acceptance test, store every set's -the_score (diagnostics) */
    URLGPU_CBIC_ACCEPT_LITERAL = 8 /* cBIC: the acceptance test AS WRITTEN (BIC_OLS.cpp:125-172 with arma::uvec zero-filled, Armadillo >= 10.5;
                                      SURVEY.md Q5) instead of the default "clean" recursion; sets of at most 12 parents */
};

/* One context = one device + one stream.  Thread-compatible: use one context per host thread. */
int urlgpu_create(urlgpu_ctx **out, int device_id);
int urlgpu_destroy(urlgpu_ctx *ctx);
const char *urlgpu_last_error(urlgpu_ctx *ctx); /* ctx may be NULL: error of the failed urlgpu_create */
int urlgpu_device_count(void);
/* use a caller-owned stream (e.g. torch's current stream) instead of the context's own; NULL restores it */
int urlgpu_set_stream(urlgpu_ctx *ctx, void *cuda_stream);
int urlgpu_synchronize(urlgpu_ctx *ctx);

/* Data is COPIED to the device; the caller keeps ownership.  Column-major: value of variable i in record r at
 * [i*n + r].  codes are value indices < cardinality[i] (first-appearance order, base/variable.h:43-48).
 * Record limits (URLGPU_ERR_LIMIT above them): a discrete data set holds at most 2e9 records (refused here); BDeu scores
 * at most 1e8 and fNML with a child of arity >= 2 at most 238 609 293 (refused by the scoring calls: the reference's
 * regret approximation computes 9 * N in int, and its table covers N = n + 1); BIC and fNML of a constant child take
 * all 2e9.  Continuous data has no record limit. */
int urlgpu_set_discrete(urlgpu_ctx *ctx, const uint8_t *codes_colmajor, int64_t n, int p, const int32_t *cardinality);
/* same, but codes_colmajor is a DEVICE pointer on ctx's device (multi-GPU: data arrives by NCCL broadcast) */
int urlgpu_set_discrete_device(urlgpu_ctx *ctx, const uint8_t *d_codes_colmajor, int64_t n, int p, const int32_t *cardinality);
/* Several contexts on ONE device (one per host thread, the reference's -t workers) can score from a single device copy:
 * ctx borrows owner's data set (no copy).  The owner must keep it installed while borrowers score. */
int urlgpu_share_discrete(urlgpu_ctx *ctx, urlgpu_ctx *owner);
/* raw continuous data; the engine centres, scales by the sample std (N-1) and forms G = Z^T Z in FP64 */
int urlgpu_set_continuous(urlgpu_ctx *ctx, const double *x_colmajor, int64_t n, int p);
int urlgpu_set_continuous_device(urlgpu_ctx *ctx, const double *d_x_colmajor, int64_t n, int p);
/* Row-sharded protocol for data larger than one GPU (config 5: p=200, n=1e7, 8 GPUs).  Every rank holds n_local rows:
 *   urlgpu_shard_begin(rows)                         attach this rank's rows (on_device=1: x is a device pointer, used in place)
 *   urlgpu_shard_moments(NULL, s1, NULL)             -> all ranks sum s1 in rank order -> mean = S1/n_total
 *   urlgpu_shard_moments(mean, s1, s2)               -> all ranks sum -> dev = sqrt((S2 - S1^2/n_total)/(n_total-1))
 *   urlgpu_shard_finish(mean, dev, n_total)          standardise + partial Gram of the local rows
 *   urlgpu_get_gram / (all-gather, sum in rank order) / urlgpu_set_gram(G, n_total, p)
 * urlgpu_set_continuous is exactly this sequence with one shard.  The exchange steps carry p or p*p doubles. */
int urlgpu_shard_begin(urlgpu_ctx *ctx, const double *x_colmajor, int64_t n_local, int p, int on_device);
int urlgpu_shard_moments(urlgpu_ctx *ctx, const double *shift /* p or NULL */, double *sum1 /* p or NULL */, double *sum2 /* p or NULL */);
int urlgpu_shard_finish(urlgpu_ctx *ctx, const double *mean, const double *dev, int64_t n_total);
/* The Gram G = Z^T Z (p*p, symmetric) can be exported (oracle-side recomputation, multi-GPU broadcast) and
 * installed without the raw data (a rank that only scores needs G and n, not the rows). */
int urlgpu_get_gram(urlgpu_ctx *ctx, double *gram_rowmajor /* p*p */);
int urlgpu_set_gram(urlgpu_ctx *ctx, const double *gram_rowmajor, int64_t n_total, int p);

/* Score the whole candidate family of `variable`: every subset of neighbors\{variable} with 0..max_parents
 * elements (score_calculator.cpp:54-135).  `neighbors` is the 2-hop mask the reference's scoringThread builds
 * (score_main.cpp:145-155); max_parents is the EFFECTIVE limit (score_main.cpp:296-304).  Results stay on
 * the device until fetched. */
int urlgpu_score_variable(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents,
                          int score_type, double lambda, unsigned filter_flags, urlgpu_result **out);
/* Optional: enqueue the compaction of the stored entries (canonical order) behind the scoring kernels without any host
 * synchronisation.  A caller that prefetches v, scores v+1 and only then counts/fetches v keeps the GPU busy while the
 * host reads results (the reference overlaps nothing: scoringThread writes each block when its variable is done,
 * score_main.cpp:173-205).  count/fetch call it themselves when it was not called. */
int urlgpu_result_prefetch(urlgpu_result *res);
int urlgpu_result_count(urlgpu_result *res, uint64_t *n_stored);   /* stored entries (after filters) */
int urlgpu_result_scored(urlgpu_result *res, uint64_t *n_scored);  /* candidate sets scored */
/* canonical order: (|S| ascending, mask ascending as an integer).  masks: n*mask_words words. */
int urlgpu_result_fetch(urlgpu_result *res, uint64_t offset, uint64_t n, uint64_t *masks, float *scores);
int urlgpu_result_free(urlgpu_result *res);
/* The same entries into DEVICE memory: this device's, or a buffer on another GPU mapped with urlgpu_peer_open (the gather of
 * the per-variable caches to the rank that writes the .pss then runs over NVLink without touching the host).  Masks get
 * mask_words_out words; variable_shift is added to every variable index (0 unless the data set is one block of a larger one). */
int urlgpu_result_fetch_device(urlgpu_result *res, uint64_t offset, uint64_t n, int mask_words_out, int variable_shift,
                               uint64_t *d_masks, float *d_scores);
/* copy `bytes` from a device address (e.g. a board other ranks filled) into host memory */
int urlgpu_copy_to_host(urlgpu_ctx *ctx, void *dst_host, const void *src_device, uint64_t bytes);
/* page-locked host memory for large result payloads (urlgpu_result_fetch copies into it at PCIe speed; pageable
 * destinations work too but go through the driver's staging copy).  NULL on failure. */
void *urlgpu_host_alloc(uint64_t bytes);
void urlgpu_host_free(void *p);

/* (variable, parent-set range) shards — the multi-GPU unit of work SURVEY.md 8(e) / BASELINE.json north_star name.
 * The canonical order of a family (layer by layer, each layer in the reference's Gosper order, score_calculator.cpp:76-120)
 * numbers its sets 0 .. family_size-1; a contiguous range of that numbering is scored independently of the rest:
 *   urlgpu_family_size        number of sets: sum_{l<=max_parents} C(candidates, l); a family of more than 2^32 - 16 sets
 *                             is refused (URLGPU_ERR_LIMIT): the score caches index sets with 32 bits
 *   urlgpu_score_range        RAW scores of sets [first, first+count) (BIC: the score, cBIC: the_score before negation),
 *                             into a host buffer or, on_device=1, a device buffer on ctx's device (e.g. an NCCL send buffer)
 *   urlgpu_result_from_scores the variable's owner, holding all family_size raw scores (gathered from the ranks), applies
 *                             the store rule / acceptance and the optional prune; the result then behaves like any other */
int urlgpu_family_size(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type, uint64_t *n);
int urlgpu_score_range(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type,
                       double lambda, uint64_t first, uint64_t count, float *scores, int on_device);
int urlgpu_result_from_scores(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type,
                              const float *scores, uint64_t n, int on_device, unsigned filter_flags, urlgpu_result **out);
/* One of `parts` disjoint parts of a variable's family, chosen by the ENGINE so that each part is as cheap as possible: for
 * discrete BIC a sub-forest of the marginalisation forest (the root tables i with i % parts == part and everything derived
 * from them: counting and marginalising are both split), else a contiguous range.  `scores` receives all family_size
 * entries; those outside the part hold the "not scored" bit pattern 0x7fc0beef, which as an int32 is larger than any finite
 * float's pattern: an element-wise MIN over the int32 views of the parts' arrays (one NCCL all-reduce) is the complete raw
 * score array for urlgpu_result_from_scores. */
int urlgpu_score_part(urlgpu_ctx *ctx, int variable, const uint64_t *neighbors, int mask_words, int max_parents, int score_type,
                      double lambda, int part, int parts, float *scores, int on_device);

/* Peer memory for the exchange step of the range shards: instead of scoring into a local send buffer and moving the pieces
 * with an all-to-all, a rank can score a piece STRAIGHT INTO ITS OWNER'S MEMORY over NVLink.  The owner allocates its score
 * board with urlgpu_peer_alloc and publishes the 64-byte handle (any transport: one all-gather); every other rank (one
 * process per GPU) maps it with urlgpu_peer_open — CUDA IPC with lazily enabled peer access — and passes the mapped
 * address + offset as the on_device destination of urlgpu_score_range.  The scoring kernels then store through NVSwitch
 * while they compute; the only synchronisation left is a barrier before the owner filters.  No reference counterpart
 * (the reference's threads share one address space, score_main.cpp:132-171). */
#define URLGPU_PEER_HANDLE_BYTES 64
int urlgpu_peer_alloc(urlgpu_ctx *ctx, uint64_t bytes, void **dev_ptr, unsigned char handle[URLGPU_PEER_HANDLE_BYTES]);
int urlgpu_peer_open(urlgpu_ctx *ctx, const unsigned char handle[URLGPU_PEER_HANDLE_BYTES], void **dev_ptr);
int urlgpu_peer_close(urlgpu_ctx *ctx, void *dev_ptr);   /* a pointer from urlgpu_peer_open */
int urlgpu_peer_free(urlgpu_ctx *ctx, void *dev_ptr);    /* a pointer from urlgpu_peer_alloc */

/* Single parent set, same value ScoringFunction::calculateScore returns (BIC: the score; cBIC: -the_score).
 * value64 (optional): BIC: exact log-likelihood before the float rounding; cBIC: the_score in FP64. */
int urlgpu_score_one(urlgpu_ctx *ctx, int variable, const uint64_t *parents, int mask_words, int score_type,
                     double lambda, float *score, double *value64);
/* Score n_sets arbitrary (variable, parent set) pairs in one call.  Entry i is variables[i] with the parent set
 * parents[i*mask_words .. i*mask_words + mask_words): any variables, any order, duplicates allowed; a parent set that
 * names the child itself has that bit ignored (as urlgpu_score_one).  scores[i] and, if values64 is not NULL,
 * values64[i] are exactly what urlgpu_score_one returns for that entry, bit for bit (BIC / fNML / BDeu: the score and
 * the exact fixed-point log-likelihood or BDeu sum; cBIC: -the_score and the_score in FP64).  One score type per call;
 * `lambda` is cBIC's lambda or BDeu's equivalent sample size.  Raw scores only: no store rule, acceptance or prune
 * (those need a subset-closed family).  Synchronous: returns when the outputs are in host memory.  The whole list is
 * validated before anything is launched; an error about one entry names the index of the first offending entry.
 * Limits per entry are urlgpu_score_one's: BIC / fNML / BDeu at most 30 parents and 2^30 cells, cBIC at most 200
 * parents.  n_sets == 0 succeeds and does nothing; n_sets >= 2^32 is refused with URLGPU_ERR_LIMIT. */
int urlgpu_score_sets(urlgpu_ctx *ctx, uint64_t n_sets, const int32_t *variables, const uint64_t *parents, int mask_words,
                      int score_type, double lambda, float *scores, double *values64);
/* Dense contingency counts of (variable, parents): counts[x_v + r_v*paIdx], paIdx mixed radix over the parents in
 * ascending variable index, lowest index least significant (log_likelihood_calculator.cpp:61-73). */
int urlgpu_contingency(urlgpu_ctx *ctx, int variable, const uint64_t *parents, int mask_words, int32_t *counts,
                       int64_t n_cells);
/* Standalone prune of a caller-supplied cache (masks over <=30 distinct variables): keep[i]=0 iff some other
 * entry j with masks[j] subset of masks[i] has scores[j] >= scores[i] (ties: the subset wins). */
int urlgpu_prune(urlgpu_ctx *ctx, const uint64_t *masks, const float *scores, uint64_t n, int mask_words, uint8_t *keep);

/* The sparse parent graph of one variable as a device query structure (SURVEY.md 8(f) row 3): replaces
 * bestscorecalculators::SparseParentBitwise (score_cache/sparse_parent_bitwise.cpp:24-110).  Built from a variable's cache
 * with the SEARCH side's sign (scores negated on read, score_cache.cpp:151: lower is better); a query names the variables
 * allowed as parents and returns the best (lowest) score among the cached subsets of that set, FLT_MAX when there is none
 * (:104-106), optionally the winning parent set / its index in score order.  Batches of queries run one warp each. */
typedef struct urlgpu_spg urlgpu_spg;
int urlgpu_spg_build(urlgpu_ctx *ctx, const uint64_t *masks, const float *scores, uint64_t n, int mask_words, int variable_count, urlgpu_spg **out);
int urlgpu_spg_query(urlgpu_spg *spg, const uint64_t *allowed /* nq*mask_words */, uint64_t nq, float *best_scores, uint64_t *best_parents /* optional */,
                     int64_t *best_index /* optional */);
int urlgpu_spg_free(urlgpu_spg *spg);

/* The optimal DAG of one skeleton component over the order graph, layer by layer on the device: the search of
 * astar/astar_main.cpp:216-546 (run_astar_on_one_scc, ancestors = 0) with the cached-subset look-up of
 * score_cache/sparse_parent_{list,bitwise}.cpp.  Entries of variable v: masks[offsets[v]..offsets[v+1]) (mask_words words
 * each) with scores in the SEARCH side's sign (lower is better, score_cache.cpp:151).  edges: p*mask_words skeleton
 * neighbourhoods or NULL.  Writes *cost, order[0..|C|) (first = a root) and parents[v*mask_words..] for v in C.
 *
 * best(v, U) is the first entry of v, in (score, |S|, mask) order, whose parent set lies inside U (FLT_MAX if none; entries
 * with a parent outside the component never qualify).  S is reached from S\{v} if S\{v} is reached, the leaf v touches
 * S\{v} in the skeleton (or S\{v} is empty, or there is no skeleton) and g = cost(S\{v}) + best(v, S\{v}), one float32
 * addition, is not +inf; cost(S) is the least such g and the leaf the smallest v attaining it.  *cost is therefore the least
 * float32 left-to-right path sum over the admissible orders: never above A*'s goal cost, and equal to it in exact
 * arithmetic.  Among orders of equal cost the DAG may differ from A*'s.
 * Costs are kept for two adjacent layers only, indexed by colex rank inside the layer, and a leaf byte for every node.
 * Device memory, from the context's caching allocator: 2^|C| + 8*C(|C|, floor(|C|/2)) bytes for the nodes, 4*2^c_v per
 * variable for the best-parent tables (c_v = its candidate parents inside C), 16 per qualifying entry, and
 * 1328*|C| + 10960 bytes of descriptors, look-up tables, binomials and output.  (Before this layout the nodes took
 * 5*2^|C| bytes, so some calls once refused for memory now run; sweeps of 24 or more variables are faster, 1.4-2.1x from
 * 28 up, and smaller ones take about 4 us more per layer.)  Refusals, all before any launch: p < 1, mask_words outside
 * 1..4, decreasing offsets, an empty component or one naming a variable >= p, a NaN score and an entry containing its own
 * variable (URLGPU_ERR_ARG); |C| > 32 and a call that does not fit the device's free memory (URLGPU_ERR_LIMIT, with the
 * bytes split into leaves, cost layers and best-parent tables).  No admissible order, or a cost of +inf: URLGPU_ERR_ARG
 * with A*'s message "No solution found.". */
int urlgpu_order_search(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                        const float *scores, const uint64_t *edges, const uint64_t *component,
                        float *cost, int32_t *order, uint64_t *parents);

/* urlgpu_order_search with a limit of 36 variables (|C| > 36: URLGPU_ERR_LIMIT) and its messages prefixed
 * "order_search_layered: " instead of "order_search: ".  Arguments, contract, device memory and outputs are
 * urlgpu_order_search's: both run the same search and give the same bits wherever both run. */
int urlgpu_order_search_layered(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                                const float *scores, const uint64_t *edges, const uint64_t *component,
                                float *cost, int32_t *order, uint64_t *parents);

/* A DAG of one skeleton component of up to 256 variables by insertion hill climbing over its admissible orders, from
 * `restarts` random orders.  Inputs, best(v, U), the sign of the scores and the outputs cost, order and parents mean what they
 * mean for urlgpu_order_search.  An order pi of C is admissible when every pi_m, m >= 1, has a skeleton neighbour among
 * pi_0..pi_{m-1} (every order without a skeleton).  Its cost is the float32 left-to-right path sum g_0 = 0,
 * g_{m+1} = fl(g_m + best(pi_m, {pi_0..pi_{m-1}})), the objective urlgpu_order_search minimises, so *cost is never below
 * urlgpu_order_search's cost on the same input.
 * Restart r = 0..restarts-1 starts from a random admissible order drawn with splitmix64 from x = seed + 0xD1B54A32D192ED03 (r+1):
 * the first variable is element draw % |C| of C in ascending index, then, until C is placed, element draw % |F| of F, the
 * unplaced variables of C adjacent to a placed one (all unplaced ones without a skeleton), in ascending index.  It then climbs:
 * a move (i, j), i != j, takes the variable at position i out and reinserts it at position j; among the admissible results the
 * least cost is taken if it is strictly below the current cost (ties: smallest i, then smallest j), otherwise the restart ends.
 * The result is the restart with the least final cost (ties: smallest r).  restart_costs[r] and restart_moves[r] (each
 * optional, `restarts` elements) receive every restart's final cost and number of moves; a restart depends only on the input,
 * seed and r.  Device memory: 4*2^c_v per variable for the best-parent tables, 16 per qualifying entry, 8 + 5|C| per restart
 * and 80|C| of descriptors.  Refusals, all before any launch: every URLGPU_ERR_ARG refusal of urlgpu_order_search with the
 * same message after "order_local_search: "; restarts outside 1..2^20 (URLGPU_ERR_ARG); a variable with more than 32 candidate
 * parents inside C, and a call that does not fit the device's free memory (URLGPU_ERR_LIMIT, with the bytes split into
 * best-parent tables, entries and per-restart state).  No admissible order, or a best cost of +inf: URLGPU_ERR_ARG,
 * "No solution found.".  Times: the tables under ms_order_tables, the climb under ms_order_layers. */
int urlgpu_order_local_search(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                              const float *scores, const uint64_t *edges, const uint64_t *component,
                              uint32_t restarts, uint64_t seed,
                              float *cost, int32_t *order, uint64_t *parents,
                              float *restart_costs /* optional, [restarts] */, uint32_t *restart_moves /* optional, [restarts] */);

/* urlgpu_order_local_search with best(v, U) looked up in v's sorted list instead of a best-parent table: the first qualifying
 * entry, in (score, |S|, mask) order, whose parent set lies inside U (SparseParentList::getScore), so a variable may have any
 * number of candidate parents inside C.  Same arguments, contract and outputs; on every input both accept, the same cost,
 * order, parents, restart costs and restart moves, bit for bit.  Device memory: 8 ceil(|C|/64) + 4 per qualifying entry,
 * 8 + 5|C| per restart and 80|C| of descriptors; no tables.  Refusals, all before any launch: every URLGPU_ERR_ARG refusal of
 * urlgpu_order_local_search with the same message after "order_local_search_sparse: "; |C| > 256, 2^32 or more qualifying
 * entries, and a call that does not fit the device's free memory (URLGPU_ERR_LIMIT, with the bytes split into entries and
 * per-restart state).  No admissible order, or a best cost of +inf: URLGPU_ERR_ARG, "No solution found.".  Times: the climb
 * under ms_order_layers; ms_order_tables does not grow. */
int urlgpu_order_local_search_sparse(urlgpu_ctx *ctx, int p, int mask_words, const uint64_t *offsets, const uint64_t *masks,
                                     const float *scores, const uint64_t *edges, const uint64_t *component,
                                     uint32_t restarts, uint64_t seed,
                                     float *cost, int32_t *order, uint64_t *parents,
                                     float *restart_costs /* optional, [restarts] */, uint32_t *restart_moves /* optional, [restarts] */);

/* Measurement hooks: device time (CUDA events on the context's stream) and launch counts per kernel family,
 * accumulated since the last reset. */
typedef struct urlgpu_stats {
    uint64_t launches_total;
    uint64_t launches_count;   /* K1 row-count / row-bucketing kernels */
    uint64_t launches_cube;    /* K1 marginalise+score kernels */
    uint64_t launches_cbic;    /* K3 */
    uint64_t launches_accept;  /* K4 */
    uint64_t launches_prune;   /* K5 */
    uint64_t launches_other;
    double ms_count, ms_cube, ms_cbic, ms_accept, ms_prune, ms_gram;
    uint64_t sets_scored;
    double algorithmic_bytes;  /* BIC: sum over scored sets of n*(|S|+1) */
    double algorithmic_flops;  /* cBIC: sum over scored sets of k^3/3+2k^2+2k */
    double gram_flops;         /* K2: 2*n*p^2 per Gram formed */
    uint64_t launches_tree;    /* always 0: kept so the struct layout stays compatible */
    double ms_tree;            /* always 0 */
    double k1_bytes_read;      /* cube path: bytes the K1 kernels load from global memory (rows + parent tables; L2 may absorb re-reads) */
    double k1_bytes_written;   /* cube path: bytes of contingency tables the K1 kernels store */
    double ms_standardise;     /* K2: column moments + standardisation passes (HBM bound); ms_gram is the DMMA Gram kernel + combine */
    uint64_t table16_fallbacks; /* K1 cube path: variables recomputed with 32-bit tables because a cell count did not fit 16 bits */
    double ms_order_tables;    /* urlgpu_order_search(_layered), urlgpu_order_local_search: best-parent tables (fill, scatter, subset-min transform) */
    double ms_order_layers;    /* urlgpu_order_search(_layered): layer sweeps and the backtrack; urlgpu_order_local_search(_sparse): the climb */
} urlgpu_stats;
int urlgpu_stats_reset(urlgpu_ctx *ctx);
int urlgpu_stats_get(urlgpu_ctx *ctx, urlgpu_stats *out);
/* enable (1) / disable (0) per-kernel CUDA-event timing (adds a stream sync per measured region) */
int urlgpu_stats_enable_timing(urlgpu_ctx *ctx, int on);

/* Measured FP64 throughput of the context's device in TFLOP/s (register-resident probes, best of three): plain DFMA and
 * the DMMA tensor path (mma.sync.m8n8k4.f64) the Gram kernel uses.  These are the denominators bench.py divides by. */
int urlgpu_probe_fp64(urlgpu_ctx *ctx, double *dfma_tflops, double *dmma_tflops);

#ifdef __cplusplus
}
#endif
#endif
