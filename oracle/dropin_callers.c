/*
 * dropin_callers.c — TEST INFRASTRUCTURE ONLY.  A C caller of the drop-in library (libtspb200_dropin.so) for
 * tests/test_gpu_dropin_link.py when the reference's own objects are not built (oracle/_ref needs a
 * deno750/TSP_Optimization checkout).  It restates the reference drivers that sit above the drop-in symbols,
 * src/heuristics.c:160 (HEU_greedy) and :572-605 (HEU_2opt_greedy, HEU_2opt_greedy_iter, HEU_2opt_extramileage:
 * constructive heuristic, then alg_2opt on its tour; plot_solution is a no-op with perf_prof set), and the instance
 * set-up of oracle/ref_shim.c, all on the reference `instance` layout the drop-in header mirrors.  Every
 * calc_dist / greedy / HEU_Greedy_iter / HEU_extramileage / alg_2opt / alg_2opt_tabu / reverse_path call resolves to
 * the drop-in, i.e. to the CUDA path.
 */
#include <stdint.h>
#include <stdlib.h>

#include "tspb200_dropin.h"

typedef tspb200_ref_instance instance;

int HEU_greedy(instance *inst) { return greedy(inst, 0); }

int HEU_2opt_greedy(instance *inst) {
    int ret = HEU_greedy(inst);
    return ret ? ret : alg_2opt(inst);
}

int HEU_2opt_greedy_iter(instance *inst) {
    int ret = HEU_Greedy_iter(inst);
    return ret ? ret : alg_2opt(inst);
}

int HEU_2opt_extramileage(instance *inst) {
    int ret = HEU_extramileage(inst);
    return ret ? ret : alg_2opt(inst);
}

/* the subset of oracle/ref_shim.c that oracle.DropinCallers drives */
instance *refshim_new(int n, const double *xy, int wt) {
    instance *inst = (instance *)calloc(1, sizeof(instance));
    inst->params.integer_cost = 1;
    inst->params.perf_prof = 1;
    inst->params.time_limit = 0; /* <=0 means unlimited, heuristics.c:458 */
    inst->params.seed = -1;
    inst->num_nodes = n;
    inst->weight_type = wt;
    inst->nodes = (tspb200_ref_point *)calloc((size_t)n, sizeof(tspb200_ref_point));
    for (int k = 0; k < n; k++) { inst->nodes[k].x = xy[2 * k]; inst->nodes[k].y = xy[2 * k + 1]; }
    inst->num_columns = (long)n * (n - 1) / 2; /* src/solver.c:268-270 */
    inst->solution.edges = (tspb200_ref_edge *)calloc((size_t)n, sizeof(tspb200_ref_edge));
    for (int k = 0; k < n; k++) { inst->solution.edges[k].i = k; inst->solution.edges[k].j = (k + 1) % n; }
    return inst;
}

void refshim_free(instance *inst) {
    if (!inst) return;
    free(inst->nodes);
    free(inst->solution.edges);
    free(inst);
}

int refshim_num_nodes(const instance *inst) { return inst->num_nodes; }
double refshim_obj(const instance *inst) { return inst->solution.obj_best; }
void refshim_set_time_limit(instance *inst, int s) { inst->params.time_limit = s; }

void refshim_get_succ(const instance *inst, int32_t *succ) {
    for (int k = 0; k < inst->num_nodes; k++) succ[k] = inst->solution.edges[k].j;
}
void refshim_set_succ(instance *inst, const int32_t *succ) {
    for (int k = 0; k < inst->num_nodes; k++) { inst->solution.edges[k].i = k; inst->solution.edges[k].j = succ[k]; }
}
