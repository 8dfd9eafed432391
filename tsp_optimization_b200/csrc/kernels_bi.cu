// kernels_bi.cu — the kernels of a best-improvement pass other than the scan itself (reference src/tabusearch.c:107-178):
// the NCCL decode, the grid-wide apply (+ first-improvement late selection), exact tile pruning (boxes, filter), the rank
// alignment barrier of the benchmarks, the exact / tabu-masked scan — and the dispatch to the scan kernel's instantiations
// (kernels_bi_scan.cuh, compiled in kernels_bi_s64.cu / _p64.cu / _128.cu / _256.cu).
#include "tsp_state.cuh"

namespace tspb {

// NCCL variant of the multi-GPU exchange: after ncclAllReduce(min) of ctl->packed every rank decodes the same winning key
// and publishes the move for its own replica of the tour.
__global__ void bi_decode_packed_kernel(const TourDev tour) {
    Ctl *ctl = tour.ctl;
    if (ctl->done) { ctl->ap_valid = 0; return; }
    int delta, i, j;
    key_unpack(ctl->packed, &delta, &i, &j);
    ctl->passes += 1;
    publish_move(tour, i, j, delta);
    if (delta >= 0) { ctl->done = 1; ctl->done_reason = DONE_OPTIMUM; }
}

// Grid-wide application of the published move (see apply_swap_range).
// seed: number of block_best[] entries (the scan's grid size) to re-evaluate as seeds of the next pass's filter, 0 = none
// NODE: also keep the node-space view of the first-improvement search current (see apply_swap_range)
// fi_late (first improvement, searches that were not sharded): 1 + parity — nobody has published a move; every thread reads the search's winner
// ctl->fi_sel[parity] = (i << 32) | j and the two positions itself (two round trips, one more than reading a published
// move, instead of the search kernel's whole "last block" tail), global thread 0 — which applies swap 0 and therefore
// holds the four edge lengths of the move — logs it and advances the sweep.
template <bool NODE>
__global__ void __launch_bounds__(256) apply_move_kernel(const InstDev inst, const TourDev tour, int seed, int timing, int fi_late) {
    __shared__ int s_last;
    Ctl *ctl = tour.ctl;
    pdl_launch_dependents();
    pdl_wait();
    // (a sharded search — several GPUs, ctl->fi_mode — has published its move itself: the classic path below)
    if (NODE && fi_late && blockIdx.x == 0 && threadIdx.x == 0) ctl->fi_sel[(fi_late - 1) ^ 1] = FI_NONE;  // the next search's word
    if (NODE && fi_late && *((volatile int *)&ctl->fi_mode[fi_late - 1]) == 0) {
        const int gtid = blockIdx.x * 256 + threadIdx.x;
        const unsigned long long f = *((volatile unsigned long long *)&ctl->fi_sel[fi_late - 1]);
        int done = 0, i0 = 0, j0 = 0;
        if (gtid == 0) {  // only thread 0 may look at these: it is also the one that rewrites them below
            done = *((volatile int *)&ctl->done);
            i0 = *((volatile int *)&ctl->cur_i);
            j0 = *((volatile int *)&ctl->cur_j);
        }
        long long delta = 0;
        int i = 0, j = 0;
        int2 park = make_int2(-1, 0);
        if (f != FI_NONE) {  // (after `done` the searches return at once and the word stays FI_NONE)
            i = (int)(f >> 32);
            j = (int)(f & 0xffffffffull);
            // pos[i] (a, outside the reversed path) is not touched by this launch; pos[j] (b) would be, by swap 0: parked instead
            apply_swap_range<true>(inst, tour, tour.pos[i], tour.pos[j], gtid, gridDim.x * 256, &delta, &park);
        }
        if (gtid == 0 && !done) {
            ctl->fi_pend_node = park.x;
            ctl->fi_pend_pos = park.y;
            if (f != FI_NONE) {
                if (delta >= 0) ctl->error = 1;  // cannot happen: the searching thread saw delta < 0
                ctl->moves += 1;                 // reference heuristics.c:476-486
                ctl->obj_delta += delta;
                const long long lc = ctl->log_count;
                if (tour.log && lc < tour.log_cap) {
                    MoveRec mr;
                    mr.i = i; mr.j = j; mr.delta = delta;
                    tour.log[lc] = mr;
                }
                ctl->log_count = lc + 1;
            }
            ctl->ap_valid = 0;
            fi_advance(tour, f, i0, j0);
        }
        // (This launch's own word is reset by the next apply launch — also by the no-op launches that follow a finished run
        // inside a batch, or the launch after them would find this move again.)
        return;
    }
    if (!ctl->ap_valid) return;
    if (timing && threadIdx.x == 0) atomicMin(&ctl->tm_apply_first, globaltimer_ns());
    apply_swap_range<NODE>(inst, tour, ctl->ap_pa, ctl->ap_pb, blockIdx.x * 256 + threadIdx.x, gridDim.x * 256);
    if (timing) {
        __syncthreads();
        if (threadIdx.x == 0) atomicMax(&ctl->tm_apply_end, globaltimer_ns());
    }
    if (!seed) return;
    // last block done: seed the next pass's filter (BI only).  Every block winner of the pass that just ended is re-evaluated in
    // the tour as it is NOW; the best one that is still a legal move bounds the next pass's minimum, so every block of the
    // next scan starts with a tight threshold instead of re-discovering its own local winner through the exact path
    // (~700 exact-path calls per pass at n = 10 000 without it, a handful with it).
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned tk = atomicAdd(&ctl->apply_ticket, 1u);
        s_last = (tk == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (threadIdx.x == 0) ctl->apply_ticket = 0;
    int best = 0;
    for (int c = threadIdx.x; c < seed; c += 256) {
        const long long d = legal_move_delta_cg(inst, tour, key_load_cg(&tour.block_best[c]));
        if (d < best) best = (int)d;
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, m));
    if ((threadIdx.x & 31) == 0 && best < 0) atomicMin(&ctl->hint, best);
}

// ---- exact tile pruning (DESIGN.md §4.8) ---------------------------------------------------------------------------
// For a tile (tile-row I, tile-column J) every pair it holds satisfies
//     delta_exact >= 2 * scale * bd(I, J) - 1 - maxds(I) - maxds(J)
// where bd is the distance between the bounding boxes of the positions of tile-row I (TI positions + the successor of
// the last one) and of tile-column J (TJ positions + successor), maxds the largest edge length ds among them, scale = 1
// (EUC_2D / CEIL_2D; an integer distance is never more than 1/2 below the real one) or 1/sqrt(10) (ATT).  A tile whose bound
// exceeds `hint` — the exact delta of some legal move, i.e. an upper bound of the pass minimum — can hold neither the
// argmin nor a tie (a tie needs delta == minimum <= hint), so skipping it cannot change the selected move: the move log
// stays the reference's bit for bit, only the number of evaluated pairs drops.  The bound is evaluated in FP32 from the
// FP32 records, and W + 1 is subtracted from it: W = 1 + 4 eps (EUC_2D) or 0.125 + 4 eps (CEIL_2D, ATT), DESIGN.md §3,
// with eps = dmax 2^-20 + 4 dc (tspb200_set_instance).  The "- 1" of the bound above is the rounding of the two exact
// distances; the 4 eps of W cover the FP32 side: the coordinate rounding of the boxes (<= 2 sqrt(2) dc per distance) and
// the roundings of the few operations below (sqrtf and the product 2 bd scale: a few ulp of 2 dmax, then one rounding per
// subtraction: together < dmax 2^-20 = eps).  The scale constants lie below 1/sqrt(10) and 1.
__global__ void __launch_bounds__(64) tile_boxes_kernel(const InstDev inst, const TourDev tour, int TI, int TJ, int ntr, int ncb,
                                                        int ncb2, int nseed) {
    __shared__ float s_r[2][5];
    Ctl *ctl = tour.ctl;
    pdl_launch_dependents();
    pdl_wait();
    if (*((volatile int *)&ctl->done)) return;
    const int n = tour.n;
    const int tid = threadIdx.x;
    const int b = blockIdx.x;
    if (b >= ntr + ncb + ncb2) {
        // every block winner of the previous pass that is still a legal move bounds this pass's minimum
        const int c = (b - ntr - ncb - ncb2) * 64 + tid;
        if (c < nseed) {
            const long long d = legal_move_delta_cg(inst, tour, key_load_cg(&tour.block_best[c]));
            if (d < 0) atomicMin(&ctl->hint, (int)d);
        }
        return;
    }
    const bool is_row = b < ntr, is_coarse = b >= ntr + ncb;
    const int start = is_row ? b * TI : (is_coarse ? (b - ntr - ncb) * PRUNE_GROUP * TJ : (b - ntr) * TJ);
    const int len = is_row ? TI : (is_coarse ? PRUNE_GROUP * TJ : TJ);
    const int end = min(start + len, n);  // inclusive: the successor of the last position (position n mirrors position 0)
    float xmin = TSPB_BIG, ymin = TSPB_BIG, xmax = -TSPB_BIG, ymax = -TSPB_BIG, mds = -TSPB_BIG;
    for (int p = start + tid; p <= end; p += 64) {
        const float4 r = __ldcg(&tour.rec[p]);
        xmin = fminf(xmin, r.x); xmax = fmaxf(xmax, r.x);
        ymin = fminf(ymin, r.y); ymax = fmaxf(ymax, r.y);
        if (p < start + len && p < n) mds = fmaxf(mds, r.z);
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
        xmin = fminf(xmin, __shfl_xor_sync(0xffffffffu, xmin, m));
        ymin = fminf(ymin, __shfl_xor_sync(0xffffffffu, ymin, m));
        xmax = fmaxf(xmax, __shfl_xor_sync(0xffffffffu, xmax, m));
        ymax = fmaxf(ymax, __shfl_xor_sync(0xffffffffu, ymax, m));
        mds = fmaxf(mds, __shfl_xor_sync(0xffffffffu, mds, m));
    }
    if ((tid & 31) == 0) {
        float *o = s_r[tid >> 5];
        o[0] = xmin; o[1] = ymin; o[2] = xmax; o[3] = ymax; o[4] = mds;
    }
    __syncthreads();
    if (tid == 0) {
        const float4 box = make_float4(fminf(s_r[0][0], s_r[1][0]), fminf(s_r[0][1], s_r[1][1]), fmaxf(s_r[0][2], s_r[1][2]),
                                       fmaxf(s_r[0][3], s_r[1][3]));
        const float m = fmaxf(s_r[0][4], s_r[1][4]);
        if (is_row) { tour.rowbox[b] = box; tour.rowmaxds[b] = m; }
        else if (is_coarse) { tour.colbox2[b - ntr - ncb] = box; tour.colmaxds2[b - ntr - ncb] = m; }
        else { tour.colbox[b - ntr] = box; tour.colmaxds[b - ntr] = m; }
    }
}

// Two-level filter, one block per tile-row: first the coarse boxes (PRUNE_GROUP tile-columns each — a superset of their
// tiles' boxes, so a dead group has only dead tiles), then the tiles of the surviving groups.  With a few per cent of the
// tiles alive the second level touches a small fraction of the ~3*10^5 tiles of a 100 000-node tour.  Live tiles of this rank
// (tile ids rank, rank + world, ...) are appended to tour.live / live_lb.
__device__ __forceinline__ float tile_lower_bound(const float4 rb, float rmax, const float4 cb, float cmax, float scale, float W) {
    const float dx = fmaxf(0.f, fmaxf(rb.x - cb.z, cb.x - rb.z));
    const float dy = fmaxf(0.f, fmaxf(rb.y - cb.w, cb.y - rb.w));
    const float bd = sqrtf(fmaf(dy, dy, dx * dx)) * scale;
    return 2.0f * bd - rmax - cmax - W - 1.0f;
}

__global__ void __launch_bounds__(128) tile_filter_kernel(const BiArgs A) {
    extern __shared__ int s_groups[];
    __shared__ int s_ng;
    Ctl *ctl = A.tour.ctl;
    pdl_launch_dependents();
    pdl_wait();
    if (*((volatile int *)&ctl->done)) return;
    const int I = blockIdx.x;
    const int rs = A.tile_row_start[I], cnt = A.tile_row_start[I + 1] - rs, j0 = A.tile_row_j0[I];
    const float hint = (float)__ldcg(&ctl->hint);
    const float4 rb = __ldcg(&A.tour.rowbox[I]);
    const float rmax = __ldcg(&A.tour.rowmaxds[I]);
    const float scale = (A.inst.metric == M_ATT) ? 0.31622773f : 0.99999905f;  // just below 1/sqrt(10) and 1
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid == 0) s_ng = 0;
    __syncthreads();
    const int K0 = j0 / PRUNE_GROUP, K1 = (j0 + cnt - 1) / PRUNE_GROUP;
    for (int K = K0 + tid; K <= K1; K += 128) {
        const float lb2 = tile_lower_bound(rb, rmax, __ldcg(&A.tour.colbox2[K]), __ldcg(&A.tour.colmaxds2[K]), scale, A.inst.W);
        if (!(lb2 > hint)) s_groups[atomicAdd(&s_ng, 1)] = K;
    }
    __syncthreads();
    const int total = s_ng * PRUNE_GROUP;
    for (int w = tid; w < ((total + 31) & ~31); w += 128) {
        bool live = false;
        float lb = 0.f;
        int t = 0;
        if (w < total) {
            const int J = s_groups[w / PRUNE_GROUP] * PRUNE_GROUP + (w % PRUNE_GROUP);
            t = rs + (J - j0);
            if (J >= j0 && J < j0 + cnt && t % A.world == A.rank) {
                lb = tile_lower_bound(rb, rmax, __ldcg(&A.tour.colbox[J]), __ldcg(&A.tour.colmaxds[J]), scale, A.inst.W);
                live = !(lb > hint);
            }
        }
        const unsigned mask = __ballot_sync(0xffffffffu, live);
        if (mask) {
            unsigned base = 0;
            if (lane == __ffs(mask) - 1) base = atomicAdd(&ctl->live_count, (unsigned)__popc(mask));
            base = __shfl_sync(0xffffffffu, base, __ffs(mask) - 1);
            if (live) {
                const unsigned idx = base + __popc(mask & ((1u << lane) - 1u));
                A.tour.live[idx] = make_int2(t, __float_as_int(lb));
            }
        }
    }
}

cudaError_t launch_tile_prune(const BiArgs &a, int TI, int grid_bi, bool pdl, cudaStream_t st) {
    const int ncb = (a.tour.n - 1) / a.TJ + 1;
    const int ncb2 = (ncb + PRUNE_GROUP - 1) / PRUNE_GROUP;
    const int nseed = grid_bi;
    const int gb = a.ntr + ncb + ncb2 + (nseed + 63) / 64;
    cudaError_t e = launch_maybe_pdl(tile_boxes_kernel, dim3(gb), dim3(64), 0, st, pdl, a.inst, a.tour, TI, a.TJ, a.ntr, ncb, ncb2, nseed);
    if (e != cudaSuccess) return e;
    if (a.ntr == 0) return cudaSuccess;
    return launch_maybe_pdl(tile_filter_kernel, dim3((unsigned)a.ntr), dim3(128), sizeof(int) * (size_t)(ncb2 + 2), st, pdl, a);
}

// ---- cross-rank alignment barrier (benchmarks): every rank bumps its counter in every peer's XchgMem and waits until all
// peers' counters reached the same value.  Launched between the L2 flush and the start event of a timed pass, so that the
// ranks enter the pass together whatever their flushes took.
__global__ void rank_align_kernel(const XchgDev X, int rank, int world, Ctl *ctl) {
    __shared__ unsigned s_e;
    const int tid = threadIdx.x;
    if (tid == 0) {
        s_e = *X.align_epoch + 1u;
        *X.align_epoch = s_e;
    }
    __syncthreads();
    if (tid < world) {
        const unsigned long long e = s_e;
        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(&X.peer[tid]->align[rank]), "l"(e) : "memory");
        const unsigned long long *src = &X.peer[rank]->align[tid];
        const long long t0 = clock64();
        for (;;) {
            unsigned long long got;
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(got) : "l"(src) : "memory");
            if (got >= e) break;
            if (clock64() - t0 > 20000000000ll) {
                ctl->error = 2;
                break;
            }
        }
    }
}

cudaError_t launch_rank_align(const XchgDev &x, int rank, int world, Ctl *ctl, cudaStream_t st) {
    rank_align_kernel<<<1, 32, 0, st>>>(x, rank, world, ctl);
    return cudaGetLastError();
}

// ---- generic exact pass (any metric, incl. GEO / matrix lookup / oversized coordinates) ------------
// Same argmin, every delta evaluated exactly (FP64 on the fly or int32 matrix gather).  One block per
// group of rows; not the throughput path.
//
// MASK = true adds the tabu list of reference src/tabusearch.c:137-149: for every non-adjacent pair the four
// edges (a,b), (a,a1), (b,b1), (a,b1) are tested with check_tenure() (:83-92) under the reference's
// short-circuit order, INCLUDING its side effect — an entry whose tenure has run out is zeroed when (and only
// when) a pair actually tests it.  iter and tenure are constant during one alg_2opt_tabu call, so an entry's
// verdict never depends on whether it was already zeroed: the set of zeroed entries is the union over all
// tested pairs and does not depend on evaluation order, which is what makes the parallel scan exact.
// Zeroed indices are appended to a list so that the host can replay them on the caller's array.
struct TabuArgs {
    int *skip;                 // n(n-1)/2 ints, device copy of the caller's tabu list
    int iter, tenure;
    long long *zl;             // indices zeroed by lazy expiry
    unsigned long long *zl_count;
    long long zl_cap;
};

// reference src/utility.c:17-30 x_udir_pos (evaluated in 64 bits; the reference's int overflows for n > 46341)
__device__ __forceinline__ long long udir_pos(int i, int j, int n) {
    if (i > j) { const int t = i; i = j; j = t; }
    return (long long)i * n + j - ((long long)(i + 1) * (i + 2)) / 2;
}

// reference src/tabusearch.c:83-92 check_tenure
__device__ __forceinline__ bool tabu_check(const TabuArgs &T, long long e) {
    if (T.iter < 0 || T.tenure < 0) return false;
    const int v = *((volatile int *)&T.skip[e]);
    if (v == 0) return false;
    if (T.iter - v > T.tenure) {
        if (atomicExch(&T.skip[e], 0) != 0) {
            const unsigned long long k = atomicAdd(T.zl_count, 1ull);
            if ((long long)k < T.zl_cap) T.zl[k] = e;
        }
        return false;
    }
    return true;
}

template <bool MASK>
__device__ __forceinline__ void bi_scan_exact_body(const InstDev &inst, const TourDev &tour, int rank, int world, int fuse_apply,
                                                   const TabuArgs &tabu) {
    __shared__ MoveKey s_keys[8];
    __shared__ int s_last;
    Ctl *ctl = tour.ctl;
    if (ctl->done) {
        if (blockIdx.x == 0 && threadIdx.x == 0) ctl->ap_valid = 0;
        return;
    }
    const int n = tour.n;
    const int tid = threadIdx.x;
    const float4 *rec = tour.rec;
    MoveKey best = key_none();
    for (int p = rank + world * (int)blockIdx.x; p < n - 2; p += world * (int)gridDim.x) {
        const float4 rp = rec[p];
        const int u = node_of(rp), u1 = node_of(rec[p + 1]);
        const long long dsp = (long long)rp.z;
        for (int q = p + 2 + tid; q < n; q += 256) {
            if (p == 0 && q == n - 1) continue;
            const float4 rq = rec[q];
            const int v = node_of(rq), v1 = node_of(rec[q + 1]);
            if (MASK) {
                // a = min(u,v) as the reference enumerates the pair; a1 / b1 are the successors of a / b
                const int a = min(u, v), b = max(u, v);
                const int a1 = (u < v) ? u1 : v1, b1 = (u < v) ? v1 : u1;
                if (tabu_check(tabu, udir_pos(a, b, n)) || tabu_check(tabu, udir_pos(a, a1, n)) ||
                    tabu_check(tabu, udir_pos(b, b1, n)) || tabu_check(tabu, udir_pos(a, b1, n)))
                    continue;
            }
            long long delta = dist_nodes(inst, u, v) + dist_nodes(inst, u1, v1) - dsp - (long long)rq.z;
            if (delta < 0 && delta <= best.delta) {
                MoveKey k;
                k.delta = (int)delta; k.i = min(u, v); k.j = max(u, v); k.pad = 0;
                if (key_less(k, best)) best = k;
            }
        }
    }
    best = key_warp_min(best);
    if ((tid & 31) == 0) s_keys[tid >> 5] = best;
    __syncthreads();
    if (tid < 32) {
        MoveKey k = (tid < 8) ? s_keys[tid] : key_none();
        k = key_warp_min(k);
        if (tid == 0) {
            tour.block_best[blockIdx.x] = k;
            __threadfence();
            unsigned tk = atomicAdd(&ctl->ticket, 1u);
            s_last = (tk == gridDim.x - 1);
        }
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    MoveKey k = key_none();
    for (int b = tid; b < (int)gridDim.x; b += 256) {
        MoveKey o = key_load_cg(&tour.block_best[b]);
        if (key_less(o, k)) k = o;
    }
    k = key_warp_min(k);
    if ((tid & 31) == 0) s_keys[tid >> 5] = k;
    __syncthreads();
    k = s_keys[0];
    for (int w = 1; w < 8; ++w)
        if (key_less(s_keys[w], k)) k = s_keys[w];
    if (tid == 0) {
        ctl->last = k;
        ctl->ticket = 0;
        ctl->launches += 1;
        if (!fuse_apply) {
            ctl->packed = (k.delta < 0) ? key_pack(k.delta, k.i, k.j) : KEY_PACK_NONE;
        } else {
            ctl->passes += 1;
            publish_move(tour, k.i, k.j, k.delta);
            if (k.delta >= 0) { ctl->done = 1; ctl->done_reason = DONE_OPTIMUM; }
        }
    }
}


template <bool MASK>
__global__ void __launch_bounds__(256) bi_scan_exact_kernel(const InstDev inst, const TourDev tour, int rank, int world,
                                                            int fuse_apply, const TabuArgs tabu) {
    bi_scan_exact_body<MASK>(inst, tour, rank, world, fuse_apply, tabu);
}

// The resident tabu search's masked pass for instances without the FP32 path: iter and tenure of the running call come from
// the search's device state.  The pass's own lazy expiry finds nothing left to zero (ts_expire_kernel ran before it).
__global__ void __launch_bounds__(256) bi_scan_exact_search_kernel(const InstDev inst, const TourDev tour, TabuArgs tabu,
                                                                   const TabuSearchDev *S) {
    tabu.iter = S->cur_iter;
    tabu.tenure = S->cur_tenure;
    bi_scan_exact_body<true>(inst, tour, 0, 1, 1, tabu);
}

// ---- host-side launchers -----------------------------------------------------------------------------
// rows (moves) of one tile for a block of `threads` threads with `rows_per_thread` rows each
int bi_tile_rows(int threads, int rows_per_thread, int row_shuffle) {
    return row_shuffle ? (threads / 32) * (32 * rows_per_thread - 1) : threads * rows_per_thread;
}
// the shuffle variant is built for the 64-thread shapes (the ones the shape model picks)
bool bi_shuffle_supported(int threads, int rows_per_thread) {
    return threads == 64 && (rows_per_thread == 2 || rows_per_thread == 4 || rows_per_thread == 8);
}

// supported (threads, rows per thread) shapes; anything else is rejected by tspb200_set_option
bool bi_shape_supported(int threads, int rows_per_thread) {
    if (threads == 256) return rows_per_thread == 2 || rows_per_thread == 4 || rows_per_thread == 8 || rows_per_thread == 16;
    if (threads == 128) return rows_per_thread == 4 || rows_per_thread == 8 || rows_per_thread == 16;
    if (threads == 64) return rows_per_thread == 2 || rows_per_thread == 4 || rows_per_thread == 8;
    return false;
}

// the scan kernel's instantiations live in four translation units (kernels_bi_scan.cuh)
cudaError_t launch_bi_scan_s64(const BiArgs &a, int R, int grid, bool pdl, cudaStream_t st);   // 64 threads, row shuffle
cudaError_t launch_bi_scan_p64(const BiArgs &a, int R, int grid, bool pdl, cudaStream_t st);   // 64 threads, plain
cudaError_t launch_bi_scan_128(const BiArgs &a, int R, int grid, bool pdl, cudaStream_t st);
cudaError_t launch_bi_scan_256(const BiArgs &a, int R, int grid, bool pdl, cudaStream_t st);

cudaError_t launch_bi_scan(const BiArgs &a, int threads, int rows_per_thread, int grid, bool pdl, cudaStream_t st) {
    if (a.row_shuffle) return threads == 64 ? launch_bi_scan_s64(a, rows_per_thread, grid, pdl, st) : cudaErrorInvalidValue;
    if (threads == 256) return launch_bi_scan_256(a, rows_per_thread, grid, pdl, st);
    if (threads == 128) return launch_bi_scan_128(a, rows_per_thread, grid, pdl, st);
    if (threads == 64) return launch_bi_scan_p64(a, rows_per_thread, grid, pdl, st);
    return cudaErrorInvalidValue;
}

cudaError_t launch_bi_scan_exact(const InstDev &inst, const TourDev &tour, int rank, int world, int fuse_apply,
                                 int grid, cudaStream_t st) {
    bi_scan_exact_kernel<false><<<grid, 256, 0, st>>>(inst, tour, rank, world, fuse_apply, TabuArgs{});
    return cudaGetLastError();
}

cudaError_t launch_bi_scan_tabu(const InstDev &inst, const TourDev &tour, int *skip, int iter, int tenure, long long *zl,
                                unsigned long long *zl_count, long long zl_cap, int grid, cudaStream_t st) {
    TabuArgs t;
    t.skip = skip; t.iter = iter; t.tenure = tenure; t.zl = zl; t.zl_count = zl_count; t.zl_cap = zl_cap;
    bi_scan_exact_kernel<true><<<grid, 256, 0, st>>>(inst, tour, 0, 1, 1, t);
    return cudaGetLastError();
}

cudaError_t launch_bi_scan_exact_search(const InstDev &inst, const TourDev &tour, TabuSearchDev *S, int *list, int grid,
                                        cudaStream_t st) {
    TabuArgs t;
    t.skip = list; t.iter = 0; t.tenure = 0; t.zl = nullptr; t.zl_count = &S->zl_count; t.zl_cap = 0;
    bi_scan_exact_search_kernel<<<grid, 256, 0, st>>>(inst, tour, t, S);
    return cudaGetLastError();
}

cudaError_t launch_bi_decode_packed(const TourDev &tour, cudaStream_t st) {
    bi_decode_packed_kernel<<<1, 1, 0, st>>>(tour);
    return cudaGetLastError();
}

// grid sized for one swap per thread (at most n/2 swaps), capped at 4 blocks per SM
// node_space: the first-improvement runs keep their node-space tables current inside the same launch
cudaError_t launch_apply_move(const InstDev &inst, const TourDev &tour, int num_sms, int seed, int timing, bool pdl,
                              bool node_space, int fi_late, cudaStream_t st) {
    int grid = (tour.n / 2 + 255) / 256;
    if (grid < 1) grid = 1;
    if (grid > 4 * num_sms) grid = 4 * num_sms;
    if (node_space) return launch_maybe_pdl(apply_move_kernel<true>, dim3(grid), dim3(256), 0, st, pdl, inst, tour, seed, timing, fi_late);
    return launch_maybe_pdl(apply_move_kernel<false>, dim3(grid), dim3(256), 0, st, pdl, inst, tour, seed, timing, 0);
}

}  // namespace tspb
