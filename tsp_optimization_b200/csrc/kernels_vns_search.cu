// kernels_vns_search.cu — the resident VNS search (reference HEU_VNS, src/vns.c:103-183) on the resident tour, every iteration
// of a call without a host round trip (tspb200_vns_search, DESIGN.md §4.9).  The host enqueues batches of
//     fi_search_kernel -> apply_move_kernel -> vns_step_kernel
// (the launches of tspb200_fi_run, plus the step) and reads the search's state once per batch.  The apply that ends a sweep
// without a move sets ctl->done: alg_2opt has returned, and the step that follows ends the iteration (cost, keep or go
// back to the incumbent) and starts the next one (kick, node-space tables, a fresh first-improvement run).  After the last
// iteration every step returns at once and ctl->done stays set, so the searches and applies return at once too.
//
// The step is one cooperative launch of one block per SM: its phases depend on each other grid-wide (the cost before the
// keep decision, the restore before the kick's gather, the gather before the scatter, the scatter before the node-space
// tables), so they are separated by grid barriers.  Every block reads `finished` and ctl->done at entry, before the first
// barrier, and nobody writes them before it: the early exit is uniform.
#include <cooperative_groups.h>

#include "tsp_state.cuh"

namespace tspb {

namespace cg = cooperative_groups;

constexpr int VS_THREADS = 512;

// start = 1: the call-start step (iters >= 1 iterations): the incumbent is the resident tour, its cost is recomputed, and the
// first kick and the first reset follow.  start = 0: the step after every apply.
__global__ void __launch_bounds__(VS_THREADS) vns_step_kernel(const VnsSearchArgs A, const InstDev I, const TourDev T, int start,
                                                              int iters) {
    __shared__ long long s_red[VS_THREADS / 32];
    __shared__ long long s_cost;
    VnsSearchDev *S = A.S;
    Ctl *ctl = T.ctl;
    const cg::grid_group grid = cg::this_grid();
    if (!start && (*((volatile int *)&S->finished) || !*((volatile int *)&ctl->done))) return;
    const int n = T.n, tid = threadIdx.x;
    const int gtid = blockIdx.x * VS_THREADS + tid, gsz = gridDim.x * VS_THREADS;
    const int t = start ? -1 : S->t;  // the iteration that ends here (-1: none)
    if (!start) iters = S->iters;
    const long long best0 = S->best;

    // 1. the position entry parked by the last late-selection apply (fi_flush_kernel), and the cost (reference vns.c:78-86;
    //    rec[].z holds the exact edge lengths, so this is the kicked cost plus the applied deltas, heuristics.c:486)
    if (gtid == 0 && ctl->fi_pend_node >= 0) {
        T.pos[ctl->fi_pend_node] = ctl->fi_pend_pos;
        ctl->fi_pend_node = -1;
    }
    long long part = 0;
    for (int p = gtid; p < n; p += gsz) part += (long long)T.rec[p].z;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) part += __shfl_xor_sync(0xffffffffu, part, m);
    if ((tid & 31) == 0) s_red[tid >> 5] = part;
    __syncthreads();
    if (tid == 0) {
        long long c = 0;
        for (int w = 0; w < VS_THREADS / 32; ++w) c += s_red[w];
        A.part[blockIdx.x] = c;
    }
    grid.sync();

    // 2. keep the tour if it is strictly cheaper than the incumbent (vns.c:167-176), else go back to the incumbent; the
    //    next kick's blocks X and Y are gathered from whichever of the two is the incumbent now
    if (tid < 32) {
        long long c = 0;
        for (int b = tid; b < (int)gridDim.x; b += 32) c += A.part[b];
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) c += __shfl_xor_sync(0xffffffffu, c, m);
        if (tid == 0) s_cost = c;
    }
    __syncthreads();
    const long long cost = s_cost;
    const bool keep = start || cost < best0;
    const float4 *src_rec = keep ? T.rec : A.inc_rec;
    const int *src_pos = keep ? T.pos : A.inc_pos;
    float4 *dst_rec = keep ? A.inc_rec : T.rec;
    int *dst_pos = keep ? A.inc_pos : T.pos;
    for (int p = gtid; p <= n; p += gsz) dst_rec[p] = src_rec[p];
    for (int p = gtid; p < n; p += gsz) dst_pos[p] = src_pos[p];
    const bool last = t + 1 >= iters;
    if (gtid == 0) {
        if (!start) A.trace[t] = cost;
        if (keep) S->best = cost;
        if (last) {
            S->t = iters;
            S->finished = 1;
        }
    }
    if (last) return;
    // kick() (vns.c:11-100) with the sorted tour indices of iteration t + 1, as vns_kick_gather_kernel / _scatter_kernel
    // (kernels_session.cu): tour index k is position (pos[0] + k) mod n, X = tour[i1+1..i2] and Y = tour[i2+1..i3] trade
    // places, f wraps to tour index 0 for i3 = n-1
    const int *kk = A.kicks + 3 * (t + 1);
    const int i1 = kk[0], L1 = kk[1] - i1, L2 = kk[2] - kk[1], L = L1 + L2;
    const int base = src_pos[0];
    auto wrap = [n](int p) {
        if (p >= n) p -= n;
        if (p >= n) p -= n;
        return p;
    };
    for (int k = gtid; k < L; k += gsz) A.scratch[k] = src_rec[wrap(base + i1 + 1 + k)];
    grid.sync();

    // 3. scatter: Y then X behind a; every read goes to the scratch or to positions outside the rewritten range
    const float4 *scr = A.scratch;
    auto from = [&](int k) { return k < L2 ? scr[L1 + k] : scr[k - L2]; };
    for (int k = gtid; k <= L; k += gsz) {
        if (k == L) {  // node a: new successor d = first node of Y
            const int pa = wrap(base + i1);
            T.rec[pa].z = (float)dist_nodes(I, node_of(T.rec[pa]), node_of(scr[L1]));
            continue;
        }
        const float4 r = from(k);
        float ds = r.z;
        if (k == L - 1) {  // node c: new successor f
            ds = (float)dist_nodes(I, node_of(r), node_of(T.rec[wrap(base + i1 + 1 + L)]));
        } else if (k == L2 - 1) {  // node e: new successor b
            ds = (float)dist_nodes(I, node_of(r), node_of(from(k + 1)));
        }
        const int p = wrap(base + i1 + 1 + k);
        T.rec[p] = make_float4(r.x, r.y, ds, r.w);
        T.pos[node_of(r)] = p;
        if (p == 0) {  // rec[n] mirrors rec[0]
            *reinterpret_cast<float2 *>(&T.rec[n].x) = make_float2(r.x, r.y);
            T.rec[n].w = r.w;
        }
    }
    grid.sync();

    // 4. node-space tables of the kicked tour (rebuild_node_space_kernel), and a fresh first-improvement run as
    //    prepare_run(reset_fi_cursor = true, cap = -1) starts it
    for (int p = gtid; p < n; p += gsz) {
        const float4 rp = T.rec[p];
        const float4 rn = T.rec[p + 1];
        const float4 rv = T.rec[p == 0 ? n - 1 : p - 1];
        const int k = node_of(rp);
        T.nrec[k] = make_float4(rp.x, rp.y, rn.x, rn.y);
        T.nlnk[k] = make_float4(rp.z, rn.w, rv.z, rv.w);
        T.npxy[k] = make_float2(rv.x, rv.y);
    }
    if (gtid == 0) {
        S->t = t + 1;
        if (start) {
            S->iters = iters;
            S->finished = 0;
            ctl->max_moves = -1;
        }
        ctl->cur_i = 0;
        ctl->cur_j = 1;
        ctl->sweep_moves = 0;
        ctl->fi_found = FI_NONE;
        ctl->fi_seg = 0;
        ctl->fi_pend_node = -1;
        ctl->fi_mode[0] = ctl->fi_mode[1] = 0;
        ctl->fi_sel[0] = ctl->fi_sel[1] = FI_NONE;
        ctl->ap_valid = 0;
        ctl->done_reason = DONE_NONE;
        ctl->done = 0;
    }
}

cudaError_t launch_vns_step(const VnsSearchArgs &a, const InstDev &I, const TourDev &T, int start, int iters, int num_sms,
                            cudaStream_t st) {  // one block per SM: co-resident, as the grid barrier needs
    VnsSearchArgs args = a;
    InstDev inst = I;
    TourDev tour = T;
    void *params[] = {&args, &inst, &tour, &start, &iters};
    return cudaLaunchCooperativeKernel((const void *)vns_step_kernel, dim3(num_sms), dim3(VS_THREADS), params, 0, st);
}

}  // namespace tspb
