/*
 * tsp_oracle.c — CPU restatement of the reference's distance / 2-opt hot path.
 * TEST INFRASTRUCTURE ONLY (see tsp_oracle.h).  Parity status: PINNED against
 * oracle/_ref (the compiled reference) and the reference's result CSVs.
 *
 * Build: gcc -O2 -fPIC -ffp-contract=off (no -march=native, no -ffast-math) so that every
 * double operation is a separately rounded IEEE-754 operation, as in the reference's x86-64 build.
 */
#include "tsp_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

/* include/distutil.h:6-7 */
static const double ORC_PI = 3.14159265358979323846264;
static const double ORC_EARTH_RAD = 6378.388;

/* src/distutil.c:4-6 nint(): truncation of x+0.5 (not a true round for negatives). */
static double round_half_trunc(double v) { return (double)(long)(v + 0.5); }

/* src/distutil.c:13-18 calc_euc2d */
static double d_euc(double ax, double ay, double bx, double by, int integer) {
    double ex = ax - bx, ey = ay - by;
    double len = sqrt(ex * ex + ey * ey);
    return integer ? round_half_trunc(len) : len;
}

/* src/distutil.c:20-31 calc_pseudo_euc (ATT) */
static double d_att(double ax, double ay, double bx, double by, int integer) {
    double ex = ax - bx, ey = ay - by;
    double r = sqrt((ex * ex + ey * ey) / 10.0);
    if (!integer) return r;
    double t = round_half_trunc(r);
    return (t < r) ? t + 1 : t;
}

/* src/distutil.c:33-37 calc_man2d — the reference takes fabs(p2.y - p2.y); the bug is the spec. */
static double d_man(double ax, double ay, double bx, double by, int integer) {
    (void)ay;
    double ex = fabs(ax - bx);
    double ey = fabs(by - by);
    return integer ? round_half_trunc(ex + ey) : ex + ey;
}

/* src/distutil.c:39-45 calc_max2d — same p2.y - p2.y bug; dmax is utility.c:12-14. */
static double d_max(double ax, double ay, double bx, double by, int integer) {
    (void)ay;
    double ex = fabs(ax - bx);
    double ey = fabs(by - by);
    if (integer) { ex = round_half_trunc(ex); ey = round_half_trunc(ey); }
    return ex > ey ? ex : ey;
}

/* src/distutil.c:47-49 calc_ceil2d — ignores the integer flag. */
static double d_ceil(double ax, double ay, double bx, double by) {
    return ceil(d_euc(ax, ay, bx, by, 0));
}

/* src/distutil.c:51-58 calc_lat_lon */
static void geo_lat_lon(double px, double py, double *lat, double *lon) {
    double deg = (double)(long)px;
    double min = px - deg;
    *lat = ORC_PI * (deg + 5.0 * min / 3.0) / 180.0;
    deg = (double)(long)py;
    min = py - deg;
    *lon = ORC_PI * (deg + 5.0 * min / 3.0) / 180.0;
}

/* src/distutil.c:60-71 calc_geo — note "+ 1.0" then nint (TSPLIB truncates; the reference rounds). */
static double d_geo(double ax, double ay, double bx, double by, int integer) {
    double lat1, lon1, lat2, lon2;
    geo_lat_lon(ax, ay, &lat1, &lon1);
    geo_lat_lon(bx, by, &lat2, &lon2);
    double q1 = cos(lon1 - lon2);
    double q2 = cos(lat1 - lat2);
    double q3 = cos(lat1 + lat2);
    double len = ORC_EARTH_RAD * acos(0.5 * ((1.0 + q1) * q2 - (1.0 - q1) * q3)) + 1.0;
    return integer ? round_half_trunc(len) : len;
}

/* src/distutil.c:73-92 calc_dist: if-chain on weight_type, anything else falls through to EUC_2D. */
double orc_dist(const double *xy, int weight_type, int integer_cost, int i, int j) {
    double ax = xy[2 * (size_t)i], ay = xy[2 * (size_t)i + 1];
    double bx = xy[2 * (size_t)j], by = xy[2 * (size_t)j + 1];
    switch (weight_type) {
        case ORC_EUC_2D: return d_euc(ax, ay, bx, by, integer_cost);
        case ORC_ATT: return d_att(ax, ay, bx, by, integer_cost);
        case ORC_MAN_2D: return d_man(ax, ay, bx, by, integer_cost);
        case ORC_MAX_2D: return d_max(ax, ay, bx, by, integer_cost);
        case ORC_CEIL_2D: return d_ceil(ax, ay, bx, by);
        case ORC_GEO: return d_geo(ax, ay, bx, by, integer_cost);
        default: return d_euc(ax, ay, bx, by, integer_cost);
    }
}

void orc_dist_row(const double *xy, int n, int weight_type, int i, int32_t *out) {
    for (int j = 0; j < n; j++) out[j] = (int32_t)orc_dist(xy, weight_type, 1, i, j);
}

void orc_dist_matrix(const double *xy, int n, int weight_type, int32_t *out) {
    for (int i = 0; i < n; i++) orc_dist_row(xy, n, weight_type, i, out + (size_t)i * n);
}

/* src/heuristics.c:18-78 greedy(): scan all unvisited i != curr, strict '<' keeps the lowest index
 * on ties (:51); closing edge added after the loop (:74).  Time limit not restated. */
double orc_nn_tour(const double *xy, int n, int weight_type, int start, int32_t *succ) {
    if (start >= n || start < 0) return -1.0;
    unsigned char *seen = (unsigned char *)calloc((size_t)n, 1);
    double total = 0.0;
    int cur = start;
    seen[start] = 1;
    for (;;) {
        int pick = -1;
        double pick_d = 1.7976931348623157e308; /* DBL_MAX */
        for (int k = 0; k < n; k++) {
            if (k == cur || seen[k]) continue;
            double d = orc_dist(xy, weight_type, 1, cur, k);
            if (d < pick_d) { pick_d = d; pick = k; }
        }
        if (pick < 0) { succ[cur] = start; break; }
        succ[cur] = pick;
        seen[pick] = 1;
        total += pick_d;
        cur = pick;
    }
    total += orc_dist(xy, weight_type, 1, cur, start);
    free(seen);
    return total;
}

/* src/heuristics.c:168-205 HEU_Greedy_iter(): greedy() from every node in index order, the first strictly better tour
 * is kept (:195).  Time limit not restated.  Returns the best cost, *best_start the node it started from. */
double orc_greedy_iter(const double *xy, int n, int weight_type, int32_t *succ, int32_t *best_start) {
    int32_t *trial = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    double best = 1.7976931348623157e308; /* DBL_MAX */
    for (int start = 0; start < n; start++) {
        double c = orc_nn_tour(xy, n, weight_type, start, trial);
        if (c < best) {
            best = c;
            if (best_start) *best_start = start;
            for (int k = 0; k < n; k++) succ[k] = trial[k];
        }
    }
    free(trial);
    return best;
}

/* src/heuristics.c:208-314 HEU_extramileage(): the two farthest nodes (strict '>' over the row-major i<j scan, :224-233),
 * then repeatedly the (unvisited node, tour edge) pair with the smallest C_ac + C_cb - C_ab — nodes in index order outside,
 * edges in edges_visited[] order inside, strict '<' (:258-277); the replaced edge keeps its slot for (a,c), (c,b) is
 * appended (:289-293).  Restated with the reference's full O(n^3) rescans.  Needs n >= 2. */
double orc_extra_mileage(const double *xy, int n, int weight_type, int32_t *succ) {
    unsigned char *seen = (unsigned char *)calloc((size_t)n, 1);
    int32_t *ea = (int32_t *)malloc(sizeof(int32_t) * (size_t)n), *eb = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    int na = 0, nb = 1;
    double far = 0.0;
    for (int i = 0; i < n; i++)
        for (int j = i + 1; j < n; j++) {
            double d = orc_dist(xy, weight_type, 1, i, j);
            if (d > far) { na = i; nb = j; far = d; }
        }
    int cnt = 0;
    ea[cnt] = na; eb[cnt] = nb; cnt++;
    ea[cnt] = nb; eb[cnt] = na; cnt++;
    succ[na] = nb;
    succ[nb] = na;
    seen[na] = seen[nb] = 1;
    double obj = 2 * orc_dist(xy, weight_type, 1, na, nb);
    while (cnt < n) {
        double best = 1.7976931348623157e308; /* DBL_MAX */
        int best_node = -1, best_slot = -1;
        for (int c = 0; c < n; c++) {
            if (seen[c]) continue;
            for (int j = 0; j < cnt; j++) {
                int a = ea[j], b = eb[j];
                double delta = orc_dist(xy, weight_type, 1, a, c) + orc_dist(xy, weight_type, 1, c, b) -
                               orc_dist(xy, weight_type, 1, a, b);
                if (delta < best) { best = delta; best_node = c; best_slot = j; }
            }
        }
        if (best_slot < 0) break;
        int a = ea[best_slot], b = eb[best_slot];
        succ[a] = best_node;
        succ[best_node] = b;
        eb[best_slot] = best_node;
        ea[cnt] = best_node; eb[cnt] = b; cnt++;
        seen[best_node] = 1;
        obj += best;
    }
    free(seen); free(ea); free(eb);
    return obj;
}

/* src/genetic.c:51-60 fitness() */
double orc_order_cost(const double *xy, int n, int weight_type, const int32_t *order) {
    double total = 0.0;
    int before = order[0];
    for (int k = 1; k < n; k++) {
        total += orc_dist(xy, weight_type, 1, before, order[k]);
        before = order[k];
    }
    total += orc_dist(xy, weight_type, 1, before, order[0]);
    return total;
}

/* src/tabusearch.c:168-172 */
double orc_succ_cost(const double *xy, int n, int weight_type, const int32_t *succ) {
    double total = 0.0;
    for (int k = 0; k < n; k++) total += orc_dist(xy, weight_type, 1, k, succ[k]);
    return total;
}

/* src/utility.c:708-722 reverse_path(): walk predecessors from start_node until end_node has been
 * re-pointed, then rebuild every predecessor from the successor array. */
void orc_reverse_path(int n, int32_t *succ, int start_node, int end_node, int32_t *prev) {
    int at = start_node;
    for (;;) {
        int before = prev[at];
        succ[at] = before;
        at = before;
        if (before == end_node) break;
    }
    for (int k = 0; k < n; k++) prev[succ[k]] = k;
}

static int32_t *build_prev(int n, const int32_t *succ) {
    int32_t *prev = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    memset(prev, 0xff, sizeof(int32_t) * (size_t)n);
    for (int k = 0; k < n; k++) prev[succ[k]] = k;
    return prev;
}

static double move_delta(const double *xy, int wt, int a, int b, int a1, int b1) {
    /* src/heuristics.c:474 == src/tabusearch.c:150 (same operand order) */
    return orc_dist(xy, wt, 1, a, b) + orc_dist(xy, wt, 1, a1, b1) - orc_dist(xy, wt, 1, a, a1) -
           orc_dist(xy, wt, 1, b, b1);
}

/* src/heuristics.c:438-502 alg_2opt() without the per-pair gettimeofday/time-limit check
 * (parity is defined with no time limit, SURVEY.md §0 #3). */
int orc_two_opt_fi(const double *xy, int n, int weight_type, int32_t *succ, double *obj,
                   int64_t max_moves, orc_move *log, int64_t log_cap, orc_stats *st) {
    orc_stats s;
    memset(&s, 0, sizeof s);
    double sweep_ref = *obj; /* best_cost, :442 */
    int32_t *prev = build_prev(n, succ);
    int stop = 0;
    while (!stop) {
        s.passes++;
        for (int a = 0; a < n - 1 && !stop; a++) {
            for (int b = a + 1; b < n; b++) {
                int a1 = succ[a], b1 = succ[b];
                if (a1 == b1 || a == b1 || b == a1) continue; /* :471 */
                s.evals++;
                double delta = move_delta(xy, weight_type, a, b, a1, b1);
                if (delta < 0) {
                    succ[a] = b;   /* :479-481 */
                    succ[a1] = b1;
                    orc_reverse_path(n, succ, b, a1, prev); /* :483 */
                    *obj += delta;                           /* :486 */
                    if (log && s.logged < log_cap) {
                        log[s.logged].i = a; log[s.logged].j = b; log[s.logged].delta = (int64_t)delta;
                        s.logged++;
                    }
                    s.moves++;
                    if (max_moves >= 0 && s.moves >= max_moves) { stop = 1; s.status = 3; break; }
                }
            }
        }
        if (stop) break;
        if (*obj >= sweep_ref) break; /* :492 */
        sweep_ref = *obj;             /* :495 */
    }
    free(prev);
    if (st) *st = s;
    return 0;
}

/* src/utility.c:17-30 x_udir_pos(), in 64-bit so that it stays defined for n > 46340. */
static int64_t tri_index(int i, int j, int n) {
    if (i > j) { int t = i; i = j; j = t; }
    return (int64_t)i * n + j - ((int64_t)(i + 1) * (i + 2)) / 2;
}

/* src/tabusearch.c:83-92 check_tenure(): lazy expiry MUTATES the entry. */
static int tenure_blocks(int32_t *slot, int iter, int tenure) {
    if (iter < 0 || tenure < 0) return 0;
    if (*slot == 0) return 0;
    if (iter - *slot > tenure) { *slot = 0; return 0; }
    return 1;
}

/* src/tabusearch.c:107-178 alg_2opt_tabu() without the per-pass time-limit check. */
int orc_two_opt_bi(const double *xy, int n, int weight_type, int32_t *succ, double *obj,
                   int32_t *skip_edge, int32_t *stored_prev, int iter, int tenure,
                   int64_t max_passes, orc_move *log, int64_t log_cap, orc_stats *st) {
    orc_stats s;
    memset(&s, 0, sizeof s);
    int32_t *prev = build_prev(n, succ);
    int best_a = 0, best_b = 0;
    for (;;) {
        if (max_passes >= 0 && s.passes >= max_passes) { s.status = 3; break; }
        s.passes++;
        double best = 0; /* mindelta, :126 */
        for (int a = 0; a < n - 1; a++) {
            for (int b = a + 1; b < n; b++) {
                int a1 = succ[a], b1 = succ[b];
                if (b == a1 || b1 == a) continue; /* :134 */
                if (skip_edge) {                  /* :137-149, '||' short-circuit order kept */
                    if (tenure_blocks(&skip_edge[tri_index(a, b, n)], iter, tenure) ||
                        tenure_blocks(&skip_edge[tri_index(a, a1, n)], iter, tenure) ||
                        tenure_blocks(&skip_edge[tri_index(b, b1, n)], iter, tenure) ||
                        tenure_blocks(&skip_edge[tri_index(a, b1, n)], iter, tenure))
                        continue;
                }
                s.evals++;
                double delta = move_delta(xy, weight_type, a, b, a1, b1);
                if (delta < best) { best = delta; best_a = a; best_b = b; } /* :151-155 strict '<' */
            }
        }
        if (best >= 0) break; /* :158 */
        int a1 = succ[best_a], b1 = succ[best_b];
        succ[best_a] = best_b; /* :161-165 */
        succ[a1] = b1;
        orc_reverse_path(n, succ, best_b, a1, prev);
        if (log && s.logged < log_cap) {
            log[s.logged].i = best_a; log[s.logged].j = best_b; log[s.logged].delta = (int64_t)best;
            s.logged++;
        }
        s.moves++;
    }
    *obj = orc_succ_cost(xy, n, weight_type, succ); /* :168-172 */
    if (stored_prev) memcpy(stored_prev, prev, sizeof(int32_t) * (size_t)n); /* :173-175 */
    free(prev);
    if (st) *st = s;
    return 0;
}

/* ---- CPU-baseline helpers (bench.py) -------------------------------------------------------- */

/* ---- the perturbation steps of the meta-heuristics (callers of the path; tests for the resident sessions) ---------- */

/* src/vns.c:11-100 kick(), with the three tour indices handed in instead of drawn (the reference draws them with
 * rand_choice at :25-31): tour[] from node 0 (:15-22), indices sorted (:34-50), a,b / c,d / e,f (:54-59), new successors
 * a->d, e->b, c->f (:60-62), cost recomputed (:78-86).  For idx3 == n-1 the reference reads tour[n] (one past its
 * calloc'ed array); f then wraps to tour[0] here, the only value that keeps the result a tour.  Returns the new cost. */
double orc_vns_kick(const double *xy, int n, int weight_type, int32_t *succ, int idx1, int idx2, int idx3) {
    int32_t *tour = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    int node = 0;
    for (int idx = 0; idx < n; idx++) { tour[idx] = node; node = succ[node]; }
    if (idx1 > idx2) { int t = idx1; idx1 = idx2; idx2 = t; }
    if (idx1 > idx3) { int t = idx1; idx1 = idx3; idx3 = t; }
    if (idx2 > idx3) { int t = idx2; idx2 = idx3; idx3 = t; }
    int a = tour[idx1], b = tour[idx1 + 1], c = tour[idx2], d = tour[idx2 + 1], e = tour[idx3];
    int f = tour[idx3 + 1 < n ? idx3 + 1 : 0];
    succ[a] = d;
    succ[e] = b;
    succ[c] = f;
    node = 0;
    for (int idx = 0; idx < n; idx++) { tour[idx] = node; node = succ[node]; }
    double cost = 0;
    int prev_node = tour[0];
    for (int i = 1; i < n; i++) { cost += orc_dist(xy, weight_type, 1, prev_node, tour[i]); prev_node = tour[i]; }
    cost += orc_dist(xy, weight_type, 1, prev_node, tour[0]);
    free(tour);
    return cost;
}

/* src/tabusearch.c:83-92 check_tenure() */
static int tenure_check(int32_t *v, int iter, int tenure) {
    if (iter < 0 || tenure < 0) return 0;
    if (*v == 0) return 0;
    if (iter - *v > tenure) { *v = 0; return 0; }
    return 1;
}

/* src/tabusearch.c:262-309, the random kick of tabu(): candidates (a, b) are taken from `pairs` in order (the reference
 * draws them with rand_choice inside the loop); skipped when a == b or the edges touch (:271-273); the first whose four
 * edges pass check_tenure (with its lazy expiry and && short-circuit, :283-290) is applied as a 2-opt move (:292-294) and
 * (a,a1), (b,b1) enter the list with `iter` (:304-307).  Returns the index of the accepted candidate or -1. */
int orc_tabu_kick(int n, int32_t *succ, int32_t *skip, const int32_t *pairs, int count, int iter, int tenure) {
    for (int c = 0; c < count; c++) {
        int a = pairs[2 * c], b = pairs[2 * c + 1];
        int a1 = succ[a], b1 = succ[b];
        if (a == b || a1 == b || b1 == a) continue;
        int64_t e1 = tri_index(a, a1, n), e2 = tri_index(b, b1, n), e3 = tri_index(a, b, n), e4 = tri_index(a1, b1, n);
        if (!tenure_check(&skip[e1], iter, tenure) && !tenure_check(&skip[e2], iter, tenure) &&
            !tenure_check(&skip[e3], iter, tenure) && !tenure_check(&skip[e4], iter, tenure)) {
            int32_t *prev = build_prev(n, succ);
            succ[a] = b;
            succ[a1] = b1;
            orc_reverse_path(n, succ, b, a1, prev);
            free(prev);
            skip[e1] = iter;
            skip[e2] = iter;
            return c;
        }
    }
    return -1;
}


int64_t orc_bi_scan_rows(const double *xy, int n, int weight_type, const int32_t *succ,
                         int row_begin, int row_end, int64_t *best_delta, int32_t *best_i, int32_t *best_j) {
    int64_t evals = 0;
    double best = 0;
    int bi = 0, bj = 0;
    if (row_end > n - 1) row_end = n - 1;
    for (int a = row_begin; a < row_end; a++) {
        for (int b = a + 1; b < n; b++) {
            int a1 = succ[a], b1 = succ[b];
            if (b == a1 || b1 == a) continue;
            evals++;
            double delta = move_delta(xy, weight_type, a, b, a1, b1);
            if (delta < best) { best = delta; bi = a; bj = b; }
        }
    }
    *best_delta = (int64_t)best; *best_i = bi; *best_j = bj;
    return evals;
}

typedef struct {
    const double *xy; int n; int wt; const int32_t *succ;
    int row_begin, row_end, tid, nthreads;
    int64_t evals, best_delta; int32_t bi, bj;
} scan_job;

#define SCAN_BLOCK_ROWS 16

static void *scan_worker(void *arg) {
    scan_job *jb = (scan_job *)arg;
    jb->evals = 0; jb->best_delta = 0; jb->bi = 0; jb->bj = 0;
    for (int r0 = jb->row_begin + jb->tid * SCAN_BLOCK_ROWS; r0 < jb->row_end; r0 += jb->nthreads * SCAN_BLOCK_ROWS) {
        int r1 = r0 + SCAN_BLOCK_ROWS < jb->row_end ? r0 + SCAN_BLOCK_ROWS : jb->row_end;
        int64_t d; int32_t i, j;
        jb->evals += orc_bi_scan_rows(jb->xy, jb->n, jb->wt, jb->succ, r0, r1, &d, &i, &j);
        if (d < jb->best_delta || (d == jb->best_delta && d < 0 && (i < jb->bi || (i == jb->bi && j < jb->bj)))) {
            jb->best_delta = d; jb->bi = i; jb->bj = j;
        }
    }
    return NULL;
}

int64_t orc_bi_scan_rows_mt(const double *xy, int n, int weight_type, const int32_t *succ,
                            int row_begin, int row_end, int threads, double *seconds,
                            int64_t *best_delta, int32_t *best_i, int32_t *best_j) {
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    pthread_t th[256];
    scan_job jobs[256];
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int t = 0; t < threads; t++) {
        scan_job jb = {xy, n, weight_type, succ, row_begin, row_end, t, threads, 0, 0, 0, 0};
        jobs[t] = jb;
        pthread_create(&th[t], NULL, scan_worker, &jobs[t]);
    }
    int64_t evals = 0, bd = 0; int32_t bi = 0, bj = 0;
    for (int t = 0; t < threads; t++) {
        pthread_join(th[t], NULL);
        evals += jobs[t].evals;
        scan_job *jb = &jobs[t];
        if (jb->best_delta < bd || (jb->best_delta == bd && bd < 0 && (jb->bi < bi || (jb->bi == bi && jb->bj < bj)))) {
            bd = jb->best_delta; bi = jb->bi; bj = jb->bj;
        }
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    if (seconds) *seconds = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
    *best_delta = bd; *best_i = bi; *best_j = bj;
    return evals;
}

/* ---- every pair at or below a threshold (tests of the FP32 filters: the pairs a filter must never reject) ---- */
typedef struct {
    const double *xy; int n; int wt; const int32_t *succ; const double *ds; double H;
    int tid, nthreads;
    orc_move *buf; int64_t len, cap;
    int64_t *block_end;  /* len after each of this thread's row blocks */
    int failed;
} pairs_job;

static void *pairs_worker(void *arg) {
    pairs_job *jb = (pairs_job *)arg;
    int k = 0;
    for (int r0 = jb->tid * SCAN_BLOCK_ROWS; r0 < jb->n - 1; r0 += jb->nthreads * SCAN_BLOCK_ROWS, k++) {
        int r1 = r0 + SCAN_BLOCK_ROWS < jb->n - 1 ? r0 + SCAN_BLOCK_ROWS : jb->n - 1;
        for (int a = r0; a < r1 && !jb->failed; a++) {
            for (int b = a + 1; b < jb->n; b++) {
                int a1 = jb->succ[a], b1 = jb->succ[b];
                if (b == a1 || b1 == a) continue;
                /* move_delta's operation order; ds[] holds the same orc_dist values it would compute */
                double delta = orc_dist(jb->xy, jb->wt, 1, a, b) + orc_dist(jb->xy, jb->wt, 1, a1, b1) - jb->ds[a] - jb->ds[b];
                if (!(delta <= jb->H)) continue;
                if (jb->len == jb->cap) {
                    int64_t nc = jb->cap ? 2 * jb->cap : 1024;
                    orc_move *nb = (orc_move *)realloc(jb->buf, sizeof(orc_move) * (size_t)nc);
                    if (!nb) { jb->failed = 1; break; }
                    jb->buf = nb;
                    jb->cap = nc;
                }
                orc_move m = {a, b, (int64_t)delta};
                jb->buf[jb->len++] = m;
            }
        }
        jb->block_end[k] = jb->len;
    }
    return NULL;
}

int64_t orc_bi_pairs_le(const double *xy, int n, int weight_type, const int32_t *succ, int64_t H, int threads,
                        orc_move **out) {
    *out = NULL;
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    double *ds = (double *)malloc(sizeof(double) * (size_t)(n > 0 ? n : 1));
    if (!ds) return -1;
    for (int a = 0; a < n; a++) ds[a] = orc_dist(xy, weight_type, 1, a, succ[a]);
    const int nblocks = n > 1 ? (n - 1 + SCAN_BLOCK_ROWS - 1) / SCAN_BLOCK_ROWS : 0;
    const int per_thread = nblocks / threads + 1;
    pthread_t th[256];
    pairs_job jobs[256];
    int failed = 0;
    for (int t = 0; t < threads; t++) {
        pairs_job jb = {xy, n, weight_type, succ, ds, (double)H, t, threads, NULL, 0, 0,
                        (int64_t *)calloc((size_t)per_thread, sizeof(int64_t)), 0};
        jobs[t] = jb;
        if (!jobs[t].block_end) { failed = 1; continue; }
        pthread_create(&th[t], NULL, pairs_worker, &jobs[t]);
    }
    int64_t total = 0;
    for (int t = 0; t < threads; t++) {
        if (!jobs[t].block_end) continue;
        pthread_join(th[t], NULL);
        failed |= jobs[t].failed;
        total += jobs[t].len;
    }
    orc_move *res = failed ? NULL : (orc_move *)malloc(sizeof(orc_move) * (size_t)(total > 0 ? total : 1));
    if (res) {  /* row block b was scanned by thread b % threads as its (b / threads)-th block */
        int64_t at = 0;
        for (int b = 0; b < nblocks; b++) {
            pairs_job *jb = &jobs[b % threads];
            const int k = b / threads;
            const int64_t lo = k ? jb->block_end[k - 1] : 0, hi = jb->block_end[k];
            memcpy(res + at, jb->buf + lo, sizeof(orc_move) * (size_t)(hi - lo));
            at += hi - lo;
        }
    }
    for (int t = 0; t < threads; t++) {
        free(jobs[t].buf);
        free(jobs[t].block_end);
    }
    free(ds);
    if (!res) return -1;
    *out = res;
    return total;
}

void orc_free(void *p) { free(p); }
