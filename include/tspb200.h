/*
 * tspb200.h — C ABI of libtspb200.so, the B200 (sm_100a) engine for the TSP_Optimization hot path:
 * TSPLIB distance evaluation and 2-opt neighbourhood evaluation / move application.
 *
 * Plain pointers and sizes only (no torch / CUDA types).  All functions return 0 on success and a
 * non-zero TSPB200_E_* code on failure; tspb200_last_error() gives the message.  There is NO CPU
 * fallback: without a CUDA device every compute entry point fails with TSPB200_E_CUDA.
 *
 * Reference interfaces replaced (paths relative to the reference repository):
 *   calc_dist        include/distutil.h:137, src/distutil.c:73-92   -> tspb200_dist_matrix*, tspb200_tour_costs
 *   alg_2opt         include/heuristics.h:82, src/heuristics.c:438  -> tspb200_two_opt(mode = TSPB200_FI)
 *   alg_2opt_tabu    src/tabusearch.c:107 (no header)                -> tspb200_two_opt(mode = TSPB200_BI), tspb200_two_opt_tabu
 *   check_tenure     src/tabusearch.c:83-92                          -> inside tspb200_two_opt_tabu (device)
 *   reverse_path     include/utility.h:334, src/utility.c:708        -> applied on the device inside two_opt
 *   greedy           include/heuristics.h, src/heuristics.c:18       -> tspb200_nn_tour
 *   HEU_Greedy_iter  src/heuristics.c:168-205                        -> tspb200_nn_tour_batch
 *   HEU_extramileage src/heuristics.c:208-314                        -> tspb200_extra_mileage
 *   fitness          src/genetic.c:51-60                             -> tspb200_tour_costs
 * The reference-named drop-in symbols themselves (calc_dist, alg_2opt, alg_2opt_tabu, reverse_path on the
 * reference's `instance` struct) live in libtspb200_dropin.so, see tspb200_dropin.h and INTEGRATION.md.
 */
#ifndef TSPB200_H
#define TSPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* weight types: numeric values of the reference enum (include/utility.h:45-52) */
enum {
    TSPB200_EUC_2D = 0,
    TSPB200_MAX_2D = 1,
    TSPB200_MAN_2D = 2,
    TSPB200_CEIL_2D = 3,
    TSPB200_GEO = 4,
    TSPB200_ATT = 5
};

/* 2-opt modes */
enum {
    TSPB200_FI = 0, /* first improvement  == reference alg_2opt       (src/heuristics.c:438-502)  */
    TSPB200_BI = 1  /* best improvement   == reference alg_2opt_tabu  (src/tabusearch.c:107-178), NULL tabu list */
};

/* error codes */
enum {
    TSPB200_OK = 0,
    TSPB200_E_CUDA = 1,     /* CUDA runtime / no device                          */
    TSPB200_E_ARG = 2,      /* bad argument (e.g. succ[] is not a single cycle)  */
    TSPB200_E_STATE = 3,    /* call order (no instance / no tour uploaded)       */
    TSPB200_E_NCCL = 4,     /* NCCL not loadable or a collective failed          */
    TSPB200_E_UNSUPPORTED = 5,
    TSPB200_E_DEVICE_CHECK = 6 /* a device-side consistency check failed         */
};

/* status of a 2-opt run, also the reference's return convention (include/heuristics.h:6-7) */
enum {
    TSPB200_LOCAL_OPTIMUM = 0,
    TSPB200_TIME_LIMIT_EXCEEDED = 2, /* reference TIME_LIMIT_EXCEEDED */
    TSPB200_STOPPED_BY_CAP = 3       /* max_passes / max_moves reached */
};

typedef struct tspb200_ctx tspb200_ctx;

typedef struct {
    int64_t passes;     /* BI: scans performed (incl. the terminating one); FI: sweeps               */
    int64_t moves;      /* applied moves                                                             */
    int64_t evals;      /* BI: passes * n(n-3)/2 (every non-adjacent pair is evaluated every scan), scaled    */
                        /* by tiles_scanned / tiles_total when tiles were pruned (pairs excluded by the exact */
                        /* bound are not evaluations); FI: linear pairs swept (upper bound of the reference's) */
    int64_t launches;   /* kernel launches of OUR kernels inside the timed region                    */
    int64_t obj_delta;  /* sum of the applied deltas                                                 */
    double gpu_ms;      /* device time of the run, CUDA events on the engine's stream                */
    double cost;        /* tour cost after the run (BI: recomputed from scratch; FI: obj_in + delta) */
    int32_t status;     /* TSPB200_LOCAL_OPTIMUM / _TIME_LIMIT_EXCEEDED / _STOPPED_BY_CAP            */
    int32_t path;       /* 0 = FP32 filter + FP64 exact (EUC/CEIL/ATT), 1 = exact on the fly, 2 = matrix lookup */
    int64_t tiles_scanned; /* BI with exact tile pruning: tiles this rank evaluated ...                          */
    int64_t tiles_total;   /* ... out of passes * (this rank's tiles); both 0 when the scan was exhaustive        */
} tspb200_stats;

typedef struct {
    int32_t i, j;   /* node indices i<j exactly as the reference enumerates them */
    int64_t delta;
} tspb200_move;

/* ---- context ------------------------------------------------------------------------------------ */
int tspb200_create(int device, tspb200_ctx **out);
void tspb200_destroy(tspb200_ctx *ctx);
const char *tspb200_last_error(const tspb200_ctx *ctx);
/* Tuning / mode knobs. keys: "block_threads" (64|128|256), "rows_per_thread" (2|4|8|16), "tile_cols" (multiple of 4,
 * 32..1024), "grid" (blocks), "fuse_apply" (-1 auto, 0 separate apply launch, 1 the scan's last block applies the move), "seed_hint" (1 = seed each
 * pass's filter from the previous pass's runner-up moves, 0 = start every pass from delta 0),
 * "exchange" (multi-GPU: 0 = NVLink peer-memory slots when available, 1 = NCCL allreduce), "pdl" (programmatic dependent
 * launch on/off), "l2_flush_bytes" (benchmarks: write that many bytes before every BI pass and time each pass with its
 * own CUDA event pair; stats.gpu_ms is then the sum of the per-pass intervals),
 * "single_block" (tspb200_two_opt on one tour: -1 auto = one thread block with the tour in shared memory for small
 * tours [FI n <= 1536, BI n <= 160], 0 = always the grid kernels, 1 = the block kernel whenever the tour fits),
 * "force_path" (-1 auto, 0 fp32 filter, 1 exact on the fly, 2 matrix), "batch" (passes per host sync),
 * "time_limit_ms" (<=0 unlimited; checked between launch batches; on several GPUs the decision is taken collectively),
 * "prune" (exact tile pruning of the best-improvement scan: -1 auto = on for n >= 3000, 0 = exhaustive scan, 1 = on;
 * the selected moves are identical either way), "timing" (1 = accumulate the per-pass breakdown read back through
 * tspb200_get_info("tm_scan" ...), 2 = also per-block time stamps), "batch_kernel" (batched best improvement: 0 =
 * position-space block kernel where applicable, 1 = node-space kernel), "nn_grid" (tspb200_nn_tour: -1 auto = the
 * bucket-grid walk for EUC_2D / CEIL_2D / ATT with n >= 256, 0 = always the grid-wide scan, 1 = the walk whenever the metric
 * allows; same tour either way), "fi_shard_min_gap" (several GPUs, see below). */
int tspb200_set_option(tspb200_ctx *ctx, const char *key, int64_t value);
int64_t tspb200_get_info(const tspb200_ctx *ctx, const char *key);

/* ---- instance (reference: instance.nodes / num_nodes / weight_type, include/utility.h:146-160) ---- */
/* xy = n interleaved (x,y) doubles, the layout of the reference's point[] (include/utility.h:126-129). */
int tspb200_set_instance(tspb200_ctx *ctx, const double *xy, int n, int weight_type);

/* ---- distance matrix: out[i*n + j] = (int32) calc_dist(i, j)  (src/distutil.c:73-92) --------------- */
/* Builds the matrix in HBM (row pitch rounded up to 4 ints) and keeps it resident; a resident matrix is
 * what "force_path" = 2 / the GEO path gather from. gpu_ms (may be NULL) = device time of the kernel. */
int tspb200_dist_matrix_build(tspb200_ctx *ctx, double *gpu_ms);
/* Copies the resident matrix to host memory as a dense n*n int32 array. */
int tspb200_dist_matrix_get(tspb200_ctx *ctx, int32_t *out);
/* One call, host buffers: build + copy back. */
int tspb200_dist_matrix(tspb200_ctx *ctx, int32_t *out);
int tspb200_dist_matrix_free(tspb200_ctx *ctx);
/* One row, out[j] = (int32) calc_dist(i, j) for j = 0..n-1, computed on the device without a resident matrix. */
int tspb200_dist_row(tspb200_ctx *ctx, int i, int32_t *out);

/* ---- tours ---------------------------------------------------------------------------------------- */
/* succ[k] = successor of node k == reference inst->solution.edges[k].j (include/utility.h:131-134). */
int tspb200_tour_upload(tspb200_ctx *ctx, const int32_t *succ, int64_t log_cap);
int tspb200_tour_download(tspb200_ctx *ctx, int32_t *succ, double *cost);
int tspb200_tour_log(tspb200_ctx *ctx, tspb200_move *log, int64_t cap, int64_t *count);

/* Runs on the RESIDENT tour (no host<->device tour traffic): max_passes / max_moves < 0 = until the
 * local optimum. Repeated calls continue where the previous one stopped. */
int tspb200_bi_run(tspb200_ctx *ctx, int64_t max_passes, tspb200_stats *st);
int tspb200_fi_run(tspb200_ctx *ctx, int64_t max_moves, tspb200_stats *st);

/* Host-buffer entry point (what the drop-in shims call): upload succ, run, download succ.
 * *obj: FI reads it and adds the deltas (reference heuristics.c:486); BI overwrites it with the recomputed
 * cost (reference tabusearch.c:168-172). log may be NULL. */
int tspb200_two_opt(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int64_t max_iters,
                    tspb200_stats *st, tspb200_move *log, int64_t log_cap, int64_t *log_count);

/* alg_2opt_tabu WITH a tabu list (reference src/tabusearch.c:107-178, check_tenure :83-92): best improvement over the
 * pairs whose four edges (a,b), (a,a1), (b,b1), (a,b1) pass check_tenure(skip_edge[x_udir_pos(..)], iter, tenure).
 * skip_edge = the caller's n(n-1)/2 ints (in/out): entries whose tenure ran out and that a pair tested are zeroed,
 * exactly like the reference's lazy expiry.  skip_edge == NULL is plain best improvement.  n <= 46340 (the
 * reference's int edge index). */
int tspb200_two_opt_tabu(tspb200_ctx *ctx, int32_t *succ, double *obj, int32_t *skip_edge, int iter, int tenure,
                         int64_t max_passes, tspb200_stats *st, tspb200_move *log, int64_t log_cap, int64_t *log_count);

/* Batched 2-opt of `batch` independent tours of the same instance (GA offspring repair, multi-start,
 * VNS / tabu restarts): one thread block per tour, tour state in shared memory, run to the local optimum.
 * succ = batch*n successors (in/out), obj = batch doubles (in/out, same convention as tspb200_two_opt). */
int tspb200_two_opt_batch(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int batch, tspb200_stats *st);

/* Nearest-neighbour tour from `start` (reference greedy(), src/heuristics.c:18-78). */
int tspb200_nn_tour(tspb200_ctx *ctx, int start, int32_t *succ, double *cost);

/* `batch` independent nearest-neighbour tours, one per start node (reference HEU_Greedy_iter, src/heuristics.c:168-205,
 * runs greedy() from every node and keeps the first strictly better tour).  succ = batch*n successors out (may be NULL
 * when only the costs are wanted), costs = batch doubles out. */
int tspb200_nn_tour_batch(tspb200_ctx *ctx, const int32_t *starts, int batch, int32_t *succ, double *costs);

/* Extra-mileage construction (reference HEU_extramileage, src/heuristics.c:208-314): farthest pair, then cheapest
 * insertion with the reference's scan order as tie-break.  succ = n successors out. */
int tspb200_extra_mileage(tspb200_ctx *ctx, int32_t *succ, double *cost);

/* Costs of `batch` tours: as_order != 0 -> tours are visiting orders (GA chromosomes, genetic.c:51-60),
 * else successor arrays. */
int tspb200_tour_costs(tspb200_ctx *ctx, const int32_t *tours, int batch, int as_order, double *out);

/* ---- resident sessions: the perturbation steps of the reference's meta-heuristics on device-resident state --------
 * The callers of the 2-opt path alternate a small perturbation with a 2-opt run (HEU_VNS src/vns.c:103-183, tabu()
 * src/tabusearch.c:188-320, HEU_Genetic src/genetic.c:445-560).  With these entry points the tour, the n(n-1)/2-int tabu
 * list and the population stay in HBM between the steps; the caller keeps the random number generator (the reference
 * draws from glibc random()) and the control flow, only indices and costs cross the bus. */

/* Cost of the resident tour (sum of the exact integer edge lengths, reference vns.c:78-86 / tabusearch.c:168-172). */
int tspb200_tour_cost(tspb200_ctx *ctx, double *cost);
/* Device-side copies of the resident tour, slot 0 or 1 ("best solution so far", vns.c:121-122,171-173). */
int tspb200_tour_save(tspb200_ctx *ctx, int slot);
int tspb200_tour_restore(tspb200_ctx *ctx, int slot);
/* kick() (src/vns.c:11-100) on the resident tour: idx1..3 = the three tour indices (counted from node 0) the reference
 * draws with rand_choice(0, n), any order; a [b..c] [d..e] f becomes a [d..e] [b..c] f.  For idx3 = n-1 the reference reads
 * one element past its tour array; here the successor wraps to tour[0].  *cost (may be NULL) = recomputed tour cost.
 * Follow with tspb200_fi_run(ctx, -1, ..) = alg_2opt (vns.c:143): it starts a fresh sweep on the kicked tour. */
int tspb200_vns_kick(tspb200_ctx *ctx, int idx1, int idx2, int idx3, double *cost);

/* tabu() with the list in HBM: begin = CALLOC of the list (tabusearch.c:196); run = alg_2opt_tabu(inst, tabu_edge, prev,
 * iter, tenure) on the resident tour (:238), st->cost = recomputed cost; kick = the random 2-opt kick (:262-309):
 * `pairs` holds count candidate (a, b) node pairs in the order the caller drew them, the first that passes the
 * reference's adjacency and check_tenure tests is applied and its two removed edges enter the list with `iter`;
 * *accepted = its index or -1 (draw again); end = optional download of the list (n(n-1)/2 ints). n <= 46340. */
int tspb200_tabu_begin(tspb200_ctx *ctx);
int tspb200_tabu_run(tspb200_ctx *ctx, int iter, int tenure, int64_t max_passes, tspb200_stats *st);
int tspb200_tabu_kick(tspb200_ctx *ctx, const int32_t *pairs, int count, int iter, int tenure, int *accepted);
int tspb200_tabu_end(tspb200_ctx *ctx, int32_t *skip_out);

/* Resident population (GA): tours live in HBM as successor arrays.  upload with slots == NULL creates a population of
 * `count` tours; with slots it overwrites those individuals (offspring).  as_order != 0: tours are chromosomes (visiting
 * orders, genetic.c:22-26), converted on the device (from_chromosome_to_edges, genetic.c:34-44; back: :437-441).
 * costs = fitness() (genetic.c:51-60) of the listed slots (all `count` first ones when slots == NULL); two_opt = alg_2opt
 * (FI, genetic.c:435) or best improvement on the listed slots in place, obj in/out like tspb200_two_opt_batch. */
int tspb200_population_upload(tspb200_ctx *ctx, const int32_t *tours, const int32_t *slots, int count, int as_order);
int tspb200_population_download(tspb200_ctx *ctx, int32_t *tours, const int32_t *slots, int count, int as_order);
int tspb200_population_costs(tspb200_ctx *ctx, const int32_t *slots, int count, double *out);
int tspb200_population_two_opt(tspb200_ctx *ctx, int mode, const int32_t *slots, int count, double *obj, tspb200_stats *st);
/* Independent VNS chains on the resident population (reference HEU_VNS, src/vns.c:103-183), one launch for all of them: for
 * every listed slot b (the first `count` when slots == NULL) and t = 0 .. iters-1: kick the slot's tour with the three tour
 * indices kicks[(b*iters + t)*3 .. +2] (counted from node 0, any order, the rules of tspb200_vns_kick), run alg_2opt (first
 * improvement from a fresh sweep) to the local optimum, and keep the result iff its cost is strictly below the slot's
 * current cost, else go back to the slot's tour.  At return each slot holds its chain's incumbent.  A chain's whole state
 * is its slot's tour (the cost is recomputed at the start), so iters = K1 and then K2 with the next kicks equals one call
 * with K1 + K2; iters = 0 returns the current costs.  best = count doubles out (incumbent costs, may be NULL); trace =
 * count*iters doubles out (cost after each iteration's 2-opt: below the previous incumbent = accepted, may be NULL);
 * st = moves, sweeps (passes), evals, gpu_ms and launches summed over all chains and iterations.  Every triple is checked
 * first: a bad one gives TSPB200_E_ARG (naming the chain and the iteration) and leaves the population untouched.  Needs n
 * to fit one block's shared memory (28 bytes per node, as tspb200_population_two_opt) and distances < 2^24
 * (TSPB200_E_UNSUPPORTED); a slot that is not one cycle gives TSPB200_E_DEVICE_CHECK. */
int tspb200_population_vns(tspb200_ctx *ctx, const int32_t *slots, int count, const int32_t *kicks, int iters, double *best,
                           double *trace, tspb200_stats *st);
/* Independent tabu searches on the resident population (reference tabu(), src/tabusearch.c:188-320), all chains and
 * iterations in one launch.  Chain b's state: its current tour in population slot slots[b], its best tour in
 * best_slots[b], its tabu list (n(n-1)/2 ints, the reference's x_udir_pos layout), its next iteration number and its own
 * glibc random() stream.  Unlike tspb200_population_vns, the random stream lives on the device: how many pairs a kick
 * draws depends on the list.
 * begin: the 2 count slots must be distinct slots of the population; zeroes the lists (CALLOC, tabusearch.c:196), sets
 * the next iteration number to 1, copies each slot to its best slot and seeds stream b with srandom(seeds[b]).  Needs n to
 * fit one block's shared memory (28 bytes per node plus one bit), distances < 2^24 and n <= 46340; count * n(n-1)/2 * 4
 * bytes of lists must fit the device's free memory, else TSPB200_E_UNSUPPORTED naming the bytes, before anything is
 * allocated.  A begin first ends the previous chain set, so a failed begin leaves none.
 * tabu: for every chain and t = 0 .. iters-1, with tenure = tenures[b*iters + t] and iter = the chain's next iteration
 * number: alg_2opt_tabu(list, iter, tenure) to the local optimum (masked best improvement, tabusearch.c:107-178); trace[b*iters
 * + t] = the recomputed cost; if it is strictly below the best slot's cost the tour is copied there; then the random kick
 * (:262-309): pairs a = rand_choice(0, n), b = rand_choice(0, n) are drawn until one passes the tests of tspb200_tabu_kick,
 * which is applied and stamped with iter; draws[b*iters + t] = the pairs drawn; the iteration number then grows by one.  A
 * kick that would need more than max_draws (>= 1) pairs stops its chain with TSPB200_E_DEVICE_CHECK naming the chain and the
 * iteration; that chain's state is then unspecified (begin again), the other chains finish normally and the outputs are
 * filled.  The whole state is kept between calls, so iters = K1 and then K2 (with the matching tenures) equals one call with
 * K1 + K2; iters = 0 returns the best costs and changes nothing.  best = count doubles (best costs), trace = count*iters
 * doubles, draws = count*iters ints, each may be NULL; st = moves, passes and evals summed over all chains, gpu_ms, launches.
 * A slot may be overwritten with tspb200_population_upload(slots = ..): the chain continues from that tour.  No chain set,
 * a re-created population or a new instance give TSPB200_E_STATE; a slot that is not one cycle TSPB200_E_DEVICE_CHECK.
 * fetch: chain `chain`'s list (n(n-1)/2 ints, may be NULL) and next iteration number (may be NULL).  There is deliberately
 * no call that writes a list.  end: frees the chain set (so do tspb200_set_instance with another instance and destroy). */
int tspb200_population_tabu_begin(tspb200_ctx *ctx, const int32_t *slots, const int32_t *best_slots, int count,
                                  const uint32_t *seeds);
int tspb200_population_tabu(tspb200_ctx *ctx, const int32_t *tenures, int iters, int max_draws, double *best,
                            double *trace, int32_t *draws, tspb200_stats *st);
int tspb200_population_tabu_fetch(tspb200_ctx *ctx, int chain, int32_t *list_out, int32_t *next_iter);
int tspb200_population_tabu_end(tspb200_ctx *ctx);

/* One tabu search (reference tabu(), src/tabusearch.c:188-320) on the resident tour, every iteration of a call on the device:
 * the semantics of tspb200_population_tabu with one chain, for any tour the list allows (n <= 46340), not only those that
 * fit one thread block.  The masked 2-opt passes are grid-wide: the FP32-filter scan with the tabu test in its exact path
 * (the exact scan for GEO, a resident matrix or coordinates FP32 cannot hold), each preceded by the pass's lazy expiry.
 * begin: zeroes the list (CALLOC, tabusearch.c:196; an allocation of its own, shared with no other entry point), sets the
 * next iteration number to 1, seeds the search's stream with srandom(seed) and copies the resident tour to the search's
 * best tour.  Needs an uploaded tour, n <= 46340, distances < 2^24 and one GPU, else TSPB200_E_UNSUPPORTED.
 * search: for t = 0 .. iters-1, with tenure = tenures[t] and iter = the next iteration number: alg_2opt_tabu(list, iter,
 * tenure) on the resident tour to the local optimum; trace[t] = the recomputed cost; a strictly cheaper tour is copied to
 * the best tour; then the kick of tspb200_population_tabu (pairs rand_choice(0, n) twice, drawn until one passes the tests
 * of tspb200_tabu_kick; applied and stamped with iter), draws[t] = the pairs drawn; the iteration number grows by one.  A
 * kick that would need more than max_draws (>= 1) pairs gives TSPB200_E_DEVICE_CHECK naming the iteration (the search's
 * state is then unspecified: begin again).  The list, table, stream, next iteration number and best tour persist until
 * end, so iters = K1 then K2 equals one call of K1 + K2; iters = 0 changes nothing.  The current tour is the resident tour:
 * other calls may replace it (tspb200_tour_upload ..) and the search continues from the new one.  The host synchronises
 * once per batch of launches.  best (may be NULL) = the best tour's cost; trace, draws = iters entries each (may be NULL);
 * st = moves, passes, evals (passes n(n-3)/2), gpu_ms, launches.  Without begin: TSPB200_E_STATE.
 * fetch: the list (n(n-1)/2 ints), the next iteration number and the best tour's successor array; each may be NULL.
 * end: frees the search (so do tspb200_set_instance with another instance and destroy). */
int tspb200_tabu_search_begin(tspb200_ctx *ctx, uint32_t seed);
int tspb200_tabu_search(tspb200_ctx *ctx, const int32_t *tenures, int iters, int max_draws, double *best, double *trace,
                        int32_t *draws, tspb200_stats *st);
int tspb200_tabu_search_fetch(tspb200_ctx *ctx, int32_t *list_out, int32_t *next_iter, int32_t *best_succ);
int tspb200_tabu_search_end(tspb200_ctx *ctx);

/* One VNS search (HEU_VNS, reference src/vns.c:103-183) on the resident tour, every iteration of a call on the device: the
 * semantics of tspb200_population_vns with one chain, for tours of any size (not only those that fit one thread block).
 * For t = 0 .. iters-1: the kick of tspb200_vns_kick with kicks[3t .. 3t+2] on the incumbent; alg_2opt (the first-improvement
 * run of tspb200_fi_run, from a fresh sweep) to the local optimum; trace[t] = the kicked cost plus the deltas; a cost strictly
 * below the incumbent's makes that tour the incumbent, else the search goes back to the incumbent.  The incumbent at entry is
 * the resident tour (its cost is recomputed); at return the resident tour is the incumbent and *best (may be NULL) its cost.
 * Nothing else persists, so iters = K1 then K2 (with the next kicks) equals one call of K1 + K2; iters = 0 returns the
 * current cost and changes nothing.  The copy of the incumbent is the call's own (tspb200_tour_save slots are untouched).
 * Every triple is checked before anything is enqueued: a bad one gives TSPB200_E_ARG naming the iteration, with the tour
 * unchanged.  The host synchronises once per batch of launches.  trace = iters entries (may be NULL); st = moves, passes
 * (FI sweeps), evals (pairs swept), gpu_ms, launches, summed over the call.  No tour: TSPB200_E_STATE; the matrix path forced
 * without a resident matrix: TSPB200_E_STATE; several GPUs: TSPB200_E_UNSUPPORTED. */
int tspb200_vns_search(tspb200_ctx *ctx, const int32_t *kicks, int iters, double *best, double *trace, tspb200_stats *st);

/* ---- multi-GPU (one process per GPU; the caller bootstraps the id, e.g. over torch.distributed) ---- */
/* Neighbourhood sharding: with a communicator attached, tspb200_bi_run deals the pair tiles round-robin over the ranks;
 * per pass every rank's packed (delta, i, j) key is stored into every peer's exchange slots over NVLink by the scan kernel
 * itself (CUDA IPC peer memory mapped at comm_init; option "exchange" = 1 or a failed mapping falls back to one 8-byte
 * NCCL min-allreduce per pass) and every rank applies the same move to its own replica of the tour.  tspb200_fi_run
 * shards the first-improvement search the same way (segments of the pair order dealt over the ranks) whenever the previous
 * search had to sweep more than "fi_shard_min_gap" pairs (default 4 000 000; 0 = always): while moves are dense an exchange
 * per move costs more than the search, so every rank then searches alone — identical results either way. */
int tspb200_comm_unique_id(void *id128); /* 128 bytes out (ncclUniqueId), call on rank 0 */
int tspb200_comm_init(tspb200_ctx *ctx, const void *id128, int rank, int world);
int tspb200_comm_destroy(tspb200_ctx *ctx);

/* ---- host-only helpers (no device needed) ----------------------------------------------------------- */
/* Tile plan of the best-improvement scan for (n, T threads per block, R rows per thread, TJ columns per tile); T, R or
 * TJ == 0 picks the shape the engine would pick for `num_sms` SMs and `world` ranks. row_start: ntr+1 prefix sums of
 * tiles per tile-row (a tile-row = T*R tour positions); row_j0: first tile column per tile-row. Used by the CPU-side
 * sharding tests. */
int tspb200_debug_tile_plan(int n, int T, int R, int TJ, int num_sms, int world, int *out_T, int *out_R, int *out_TJ,
                            int *row_start, int *row_j0, int cap, int *ntr);
/* The same with the row-shuffle variant of the scan kernel taken into account (row_shuffle != 0: a tile-row of a 64-thread
 * shape is (T/32)(32R - 1) positions, *out_tile_rows; the shape model knows about it), i.e. the plan tspb200_tour_upload makes. */
int tspb200_debug_tile_plan_ex(int n, int T, int R, int TJ, int num_sms, int world, int row_shuffle, int *out_T, int *out_R,
                               int *out_TJ, int *out_tile_rows, int *row_start, int *row_j0, int cap, int *ntr);

/* Timing experiments: device-side debug buffers ("block_times": [grid][2] uint64 %globaltimer stamps {start, end} of every
 * block of the last best-improvement pass run with option "timing" = 2). */
int tspb200_debug_fetch(tspb200_ctx *ctx, const char *what, void *out, int64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* TSPB200_H */
