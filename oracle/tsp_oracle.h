/*
 * tsp_oracle.h — CPU restatement of the TSP_Optimization distance / 2-opt hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product:
 * only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference leg may load this library, and there only as the checker or as the
 * reported CPU baseline.  The product (libtspb200.so) never links or calls it.
 *
 * Parity status: PINNED.  This restatement is checked (tests/test_oracle.py)
 *   - against the unmodified reference compiled from /root/reference/src into
 *     oracle/_ref/libtspref.so (all-pairs distances, NN tours, FI and BI move
 *     logs and final tours on TSPLIB + synthetic instances), and
 *   - against the reference's published goldens
 *     results/constructive_heuristics_new.csv (GREEDY column) and
 *     results/constructive_heuristics_2opt_new.csv (2OPT_GREEDY column),
 *     committed as tests/golden/reference_csv_goldens.json.
 *
 * Every function cites the reference file:line (paths relative to
 * /root/reference) whose behaviour it restates.
 */
#ifndef TSP_ORACLE_H
#define TSP_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* include/utility.h:45-52 — numeric values of the reference's weight_type enum */
enum {
    ORC_EUC_2D = 0,
    ORC_MAX_2D = 1,
    ORC_MAN_2D = 2,
    ORC_CEIL_2D = 3,
    ORC_GEO = 4,
    ORC_ATT = 5
};

/* include/heuristics.h:6-7 */
#define ORC_WRONG_STARTING_NODE 1
#define ORC_TIME_LIMIT_EXCEEDED 2

/* One applied 2-opt move: node indices i<j as the reference enumerates them, and its delta. */
typedef struct {
    int32_t i;
    int32_t j;
    int64_t delta;
} orc_move;

/* Counters filled by the 2-opt drivers. */
typedef struct {
    int64_t evals;   /* evaluated (non-adjacent) pairs                                   */
    int64_t moves;   /* applied moves                                                    */
    int64_t passes;  /* BI: full scans incl. the terminating one; FI: sweeps             */
    int64_t logged;  /* entries written to the move log (<= log_cap)                     */
    int32_t status;  /* 0 = local optimum reached; 3 = stopped by max_passes / max_moves */
} orc_stats;

/* src/distutil.c:73-92 calc_dist.  xy = n interleaved (x,y) doubles (include/utility.h:126-129 point). */
double orc_dist(const double *xy, int weight_type, int integer_cost, int i, int j);

/* All-pairs calc_dist as int32, row-major n*n (no reference counterpart: the reference never
 * materialises the matrix; golden = calc_dist(i,j) for every (i,j), SURVEY.md §0 #2). */
void orc_dist_matrix(const double *xy, int n, int weight_type, int32_t *out);

/* One row of the matrix: out[j] = calc_dist(i,j). */
void orc_dist_row(const double *xy, int n, int weight_type, int i, int32_t *out);

/* src/heuristics.c:18-78 greedy(): nearest neighbour from `start`; writes succ[] (edges[k].j)
 * and returns the tour cost accumulated exactly as the reference does. Returns -1 on bad start. */
double orc_nn_tour(const double *xy, int n, int weight_type, int start, int32_t *succ);

/* src/heuristics.c:168-205 HEU_Greedy_iter(): nearest neighbour from every node, first strictly better tour kept. */
double orc_greedy_iter(const double *xy, int n, int weight_type, int32_t *succ, int32_t *best_start);

/* src/heuristics.c:208-314 HEU_extramileage(): farthest pair + cheapest insertion in the reference's scan order (n >= 2). */
double orc_extra_mileage(const double *xy, int n, int weight_type, int32_t *succ);

/* src/genetic.c:51-60 fitness(): cost of a tour given as a visiting order (chromosome). */
double orc_order_cost(const double *xy, int n, int weight_type, const int32_t *order);

/* Cost of a tour given as successor array (tabusearch.c:168-172 recompute loop). */
double orc_succ_cost(const double *xy, int n, int weight_type, const int32_t *succ);

/* src/utility.c:708-722 reverse_path(). prev may be NULL-free scratch of n ints (rebuilt in full). */
void orc_reverse_path(int n, int32_t *succ, int start_node, int end_node, int32_t *prev);

/* src/heuristics.c:438-502 alg_2opt(): first-improvement sweeps.  *obj is updated by += delta like
 * inst->solution.obj_best.  max_moves < 0 = unlimited.  log may be NULL. */
int orc_two_opt_fi(const double *xy, int n, int weight_type, int32_t *succ, double *obj,
                   int64_t max_moves, orc_move *log, int64_t log_cap, orc_stats *st);

/* src/tabusearch.c:107-178 alg_2opt_tabu(): best-improvement passes.  skip_edge (n(n-1)/2 ints) and
 * stored_prev (n ints) may be NULL.  *obj is recomputed from scratch at exit like the reference.
 * max_passes < 0 = unlimited (a capped run reports status 3 and still recomputes *obj). */
int orc_two_opt_bi(const double *xy, int n, int weight_type, int32_t *succ, double *obj,
                   int32_t *skip_edge, int32_t *stored_prev, int iter, int tenure,
                   int64_t max_passes, orc_move *log, int64_t log_cap, orc_stats *st);

/* CPU-baseline helper (bench.py only): evaluates rows [row_begin,row_end) of ONE best-improvement
 * scan (tabusearch.c:128-156, NULL mask) and returns the packed winner; threads are started by the
 * caller.  Returns the number of evaluated pairs. */
int64_t orc_bi_scan_rows(const double *xy, int n, int weight_type, const int32_t *succ,
                         int row_begin, int row_end, int64_t *best_delta, int32_t *best_i, int32_t *best_j);

/* Multi-threaded wrapper around orc_bi_scan_rows (pthreads, rows dealt round-robin in blocks).
 * Returns evaluated pairs; *seconds = wall time of the scan. */
int64_t orc_bi_scan_rows_mt(const double *xy, int n, int weight_type, const int32_t *succ,
                            int row_begin, int row_end, int threads, double *seconds,
                            int64_t *best_delta, int32_t *best_i, int32_t *best_j);

/* Every legal pair (a, b), a < b, of ONE best-improvement scan (same pairs and same delta arithmetic as
 * orc_bi_scan_rows) whose exact delta is <= H.  *out gets a malloc'ed array (free it with orc_free), in
 * (a, b) order; returns the number of pairs, -1 when out of memory. */
int64_t orc_bi_pairs_le(const double *xy, int n, int weight_type, const int32_t *succ, int64_t H, int threads,
                        orc_move **out);
void orc_free(void *p);

#ifdef __cplusplus
}
#endif
/* perturbation steps of the meta-heuristics (reference src/vns.c:11-100, src/tabusearch.c:262-309), indices handed in */
double orc_vns_kick(const double *xy, int n, int weight_type, int32_t *succ, int idx1, int idx2, int idx3);
int orc_tabu_kick(int n, int32_t *succ, int32_t *skip, const int32_t *pairs, int count, int iter, int tenure);

#endif
