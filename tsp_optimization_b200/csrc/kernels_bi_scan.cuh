// kernels_bi_scan.cuh — the best-improvement scan kernel: best-improvement 2-opt pass (reference src/tabusearch.c:107-178 alg_2opt_tabu with a
// NULL tabu list): one launch = one full scan of all n(n-3)/2 non-adjacent pairs + argmin + apply.
//
// The scan runs in POSITION space.  For positions p<q with u=node(p), v=node(q) the reference pair is
// (i,j) = (min(u,v), max(u,v)); its two removed edges are (node(p),node(p+1)) and (node(q),node(q+1))
// whichever of u,v is the smaller index, and
//     delta = D[p][q] + D[p+1][q+1] - ds[p] - ds[q],      D[p][q] = d(node(p), node(q)).
// Each D value is therefore used by two pairs, (p,q) and (p-1,q-1): a thread owns R consecutive rows
// and marches along the columns, so it needs R+1 distances per R evaluated moves — R of its own and
// the first one of the thread below, which the SHUF variants fetch from the next lane with a shuffle.
//
// Arithmetic: FP32 (2 FADD, FMUL, FFMA, MUFU.SQRT per distance) as a FILTER: Q = D1 + D2 - ds_p is
// compared with thr + ds_q where thr = (best exact delta so far) + W.  W bounds the worst FP32/rounding
// excess (DESIGN.md §3), so the true argmin always passes; every pair that passes is re-evaluated in
// FP64 with the reference's exact operation order and only those exact integer deltas enter the
// (delta, i, j) argmin.  Column records are staged in shared memory by TMA bulk copies (UBLKCP),
// double-buffered across tiles.
//
// Stage-1 prefilter (bi_scan_kernel, exhaustive scans of large tours): a bound on the sum of squared distances, evaluated as
// a 4-term dot product (four packed FMAs per two moves, no square root), decides first; only its hits meet the square-root
// filter above (see pf_bound and pf_dot_const below).
// bi_scan_sqrt_kernel is the square-root filter alone (pruned passes, smaller shares per rank, option "prefilter" = 0).
//
// Header: the kernels are templates over the block shape and the instance flags (104 square-root instantiations, 52 prefilter
// ones: exhaustive only); they are compiled in
// four translation units (kernels_bi_s64.cu, kernels_bi_p64.cu, kernels_bi_128.cu, kernels_bi_256.cu) so that a clean build
// compiles them in parallel (make -j4).  kernels_bi.cu holds the dispatch and the other kernels of a pass.
#pragma once
#include "tsp_state.cuh"

namespace tspb {



template <bool ATT>
__device__ __forceinline__ float dist32(float ax, float ay, float bx, float by) {
    float dx = ax - bx;
    float dy = ay - by;
    float s = fmaf(dy, dy, dx * dx);
    if (ATT) s *= 0.1f;
    return sqrt_approx(s);
}


// distances from R+1 consecutive rows to one column point: rows 0..R-1 in R/2 packed pairs, row R scalar
// LAST: how D[R] — the distance from the row just below this thread's rows, i.e. the first row of the next lane — is
// obtained: 1 = computed here (scalar, the (R+1)-th square root of the column), 2 = taken from the next lane with one
// shuffle (SHUF kernels: the lanes of a warp own adjacent row groups, so that distance is lane+1's D[0]), 0 = not needed.
template <int R, bool ATT, int LAST>
__device__ __forceinline__ void column_dists(const f32x2 (&xr2)[R / 2], const f32x2 (&yr2)[R / 2], float xrl, float yrl,
                                             float cx, float cy, float (&D)[R + 1]) {
    const f32x2 cxx = f2pack(cx, cx), cyy = f2pack(cy, cy);
#pragma unroll
    for (int k = 0; k < R / 2; ++k) {
        f32x2 dx = f2sub(xr2[k], cxx);
        f32x2 dy = f2sub(yr2[k], cyy);
        f32x2 s = f2fma(dy, dy, f2mul(dx, dx));
        if (ATT) s = f2mul(s, f2pack(0.1f, 0.1f));
        D[2 * k] = sqrt_approx(f2lo(s));
        D[2 * k + 1] = sqrt_approx(f2hi(s));
    }
    if (LAST == 1) {
        D[R] = dist32<ATT>(xrl, yrl, cx, cy);
    } else if (LAST == 2) {
        D[R] = __shfl_down_sync(0xffffffffu, D[0], 1);
    } else {
        D[R] = 0.f;
    }
}

// ---- stage-1 prefilter (option "prefilter", DESIGN.md §3) ----------------------------------------------------
// The FP32 filter above asks D1 + D2 <= ds_p + ds_q + thr (D1 = D(p,q), D2 = D(p+1,q+1)) and needs a square root per
// distance.  With a = ds_p + h, b = ds_q + h, h = (thr + E) / 2, every pair that filter can pass has d1 + d2 <= a + b
// (d = the real distance between the FP32 coordinates; E bounds the filter's own FP32 error and the roundings of a, b),
// hence, since a + b >= d1 + d2 >= 0,
//     s1 + s2 = d1^2 + d2^2 <= (d1 + d2)^2 <= (a + b)^2 <= 2 a|a| + 2 b|b|        (s = dx^2 + dy^2; ATT: d^2 = s / 10)
// — the last step is 2a^2 + 2b^2 - (a+b)^2 = (a-b)^2 >= 0 for a, b >= 0 and, for b < 0 <= a + b, (a - 3b)(a + b) >= 0.
// So every such pair has  s1 + s2 - pf_bound(ds_p) - pf_bound(ds_q) <= 0  in real arithmetic, where
// pf_bound(x) >= 2g (x + h)|x + h| (g = 1, ATT: 10) is an FP32 value with a relative slack PF_REL over its own roundings and
// an absolute one (PF_ABS) for flushed denormals.
// Stage 1 evaluates that left-hand side in expanded form, as a 4-term dot product.  With X' = x - c (the instance's
// translation BiArgs::pf_cx / pf_cy, exact for every coordinate, so s is unchanged), P = point(p), P1 = point(p+1),
// Q = point(q), Q1 = point(q+1):
//     s1 + s2 - pf_p - pf_q = A_p + B_q + w_p . v_q,      w_p = -2 (X'_p, Y'_p, X'_p+1, Y'_p+1),  v_q = (X'_q, Y'_q, X'_q+1, Y'_q+1)
//     A_p = |P'|^2 + |P1'|^2 - pf_p   (row constant),      B_q = |Q'|^2 + |Q1'|^2 - pf_q   (column constant)
// The column loop does 4 FMAs per move from A_p, folds the rows with a minimum and adds B_q once per column; a block is a hit
// when its minimum is <= 0.  pf_dot_const lowers A_p and B_q by the rounding margins of that chain (see there), so no pair
// the square-root filter can pass is rejected.  Padding rows / columns (ds = -BIG) give pf = -inf, hence A = +inf /
// B = +inf: never a hit, never a NaN (their coordinates are finite).
// Stage 2 re-runs the square-root filter on the hitting lane's R x BI_CB block (bi_refilter_warp); only what survives it
// reaches bi_cold_warp, so the exact path sees the same pairs as without the prefilter.
//
// PF_REL: each constant rounds < 3 ulp; inflating it by 2^-16 of 2g (x + h)^2 keeps it above 2g (x + h)|x + h|.
// PF_ABS: flush-to-zero can move a product or a sum by < 2^-126 each.
constexpr float PF_REL = 0x1p-16f;
constexpr float PF_ABS = 0x1p-100f;

// upper bound of 2g (ds + h)|ds + h|, g = 10 for ATT (its distances are sqrt(s / 10)), else 1
template <bool ATT>
__device__ __forceinline__ float pf_bound(float ds, float h) {
    const float a = ds + h;
    return fmaf(a * (ATT ? 20.f : 2.f), fmaf(PF_REL, a, fabsf(a)), PF_ABS);
}

// DOT_REL: the four roundings of the FMA chain are < 4.01 ulp of |A| + sum |w_i v_i| <= |A| + |P^|^2 + |Q^|^2 (AM-GM,
// P^ = (P', P1'), Q^ = (Q', Q1')), so that error splits into a row part and a column part.  Each constant also carries the
// roundings of its norm (< 4.01 ulp), of nrm - pf (1 ulp), of the margin's sum and FMA (< 2 ulp), all relative to
// K = nrm + |pf|: < 15 ulp of K for the row, < 11 for the column.  Both are lowered by 2^-19 = 32 ulp of K (DESIGN.md §3).
// DOT_ABS: flushed or gradual-underflow results, < 2^-126 per operation.
constexpr float DOT_REL = 0x1p-19f;
constexpr float DOT_ABS = 0x1p-100f;

// stage-1 row / column constant: nrm - pf lowered by its margin; +inf for padding (pf = -inf)
__device__ __forceinline__ float pf_dot_const(float nrm, float pf) {
    const float t = nrm - pf;
    return pf == -INFINITY ? t : fmaf(-DOT_REL, nrm + fabsf(pf), t) - DOT_ABS;
}

// ---- cold path ------------------------------------------------------------------------------------------
// Exact re-evaluation of one filter hit: the R x BI_CB pairs (rows p0..p0+R-1) x (columns Q0+jj0 .. +BI_CB-1) of ONE
// thread whose FP32 block minimum passed the threshold.  WARP-COOPERATIVE: the whole warp is converged at the call (the
// hot loop has no divergent branch, the hit test is a ballot), so the 32 lanes take one pair each — column records
// from shared memory, row records from L2 — re-apply the FP32 filter, evaluate the survivors exactly (FP64 with the reference's
// operation order, reference src/tabusearch.c:150 / src/distutil.c) and reduce the best exact (delta, i, j) key with
// shuffles.  A hit costs a few hundred cycles instead of a serial walk over 32 pairs by a single lane.
constexpr int BI_CB = 4;  // columns per filter check (the prefilter reads its column constants as one float4 per check)

template <int R, bool ATT, bool EXACT32>
__device__ __noinline__ MoveKey bi_cold_warp(const InstDev I, const float4 *rec, const float4 *sc, int n, int p0, int Q0,
                                             int jj0, float thr TSPB_PROBE_ARG(int own_rows)) {
    const int lane = threadIdx.x & 31;
    MoveKey best = key_none();
#pragma unroll 1
    for (int base = 0; base < R * BI_CB; base += 32) {
        const int idx = base + lane;
        const int r = idx / BI_CB, c = idx % BI_CB;
        const int p = p0 + r, q = Q0 + jj0 + c;
        if (idx < R * BI_CB && q >= p + 2 && q <= n - 1 && !(p == 0 && q == n - 1)) {  // reference tabusearch.c:134
            const float4 rp = __ldg(&rec[p]), rp1 = __ldg(&rec[p + 1]);  // row records: one L2 round trip for the warp
            const float4 c0 = sc[jj0 + c], c1 = sc[jj0 + c + 1];
            const float dsq = c0.z;
            const float qv = (dist32<ATT>(rp.x, rp.y, c0.x, c0.y) - rp.z) + dist32<ATT>(rp1.x, rp1.y, c1.x, c1.y);
            if (qv <= thr + dsq TSPB_PROBE_OR(I.probe_on)) {
                const int u = node_of(rp), v = node_of(c0);
                long long d1, d2;
                if (EXACT32) {
                    d1 = exact_dist(I.metric, make_double2((double)rp.x, (double)rp.y), make_double2((double)c0.x, (double)c0.y));
                    d2 = exact_dist(I.metric, make_double2((double)rp1.x, (double)rp1.y), make_double2((double)c1.x, (double)c1.y));
                } else {
                    d1 = exact_dist(I.metric, I.pt64[u], I.pt64[v]);
                    d2 = exact_dist(I.metric, I.pt64[node_of(rp1)], I.pt64[node_of(c1)]);
                }
                const long long delta = d1 + d2 - (long long)rp.z - (long long)dsq;
#if TSPB_FILTER_PROBE
                if (I.probe_on) {  // every pair, passed or not; rows the calling lane owns only; no key (the threshold stays pinned)
                    if (r < own_rows && delta <= I.probe_H) probe_record(I, u, v, delta, qv, thr, qv <= thr + dsq);
                    continue;
                }
#endif
                if (delta < 0) {
                    MoveKey k;
                    k.delta = (int)delta; k.i = min(u, v); k.j = max(u, v); k.pad = 0;
                    if (key_less(k, best)) best = k;
                }
            }
        }
    }
    __syncwarp();
    return key_warp_min(best);
}

// Stage 2 of the prefilter: does any pair of the R x BI_CB block pass bi_cold_warp's square-root filter?  Same pairs,
// same expression, one pair per lane; inline, so the kernel's own code keeps the MUFU.SQRT of the filter.  Warp-uniform.
template <int R, bool ATT>
__device__ __forceinline__ bool bi_refilter_warp(const float4 *rec, const float4 *sc, int n, int p0, int Q0, int jj0, float thr) {
    const int lane = threadIdx.x & 31;
    bool pass = false;
#pragma unroll
    for (int base = 0; base < R * BI_CB; base += 32) {
        const int idx = base + lane;
        const int r = idx / BI_CB, c = idx % BI_CB;
        const int p = p0 + r, q = Q0 + jj0 + c;
        if (idx < R * BI_CB && q >= p + 2 && q <= n - 1 && !(p == 0 && q == n - 1)) {
            const float4 rp = __ldg(&rec[p]), rp1 = __ldg(&rec[p + 1]);
            const float4 c0 = sc[jj0 + c], c1 = sc[jj0 + c + 1];
            const float qv = (dist32<ATT>(rp.x, rp.y, c0.x, c0.y) - rp.z) + dist32<ATT>(rp1.x, rp1.y, c1.x, c1.y);
            pass |= qv <= thr + __ldg(&rec[q].z);
        }
    }
    return __any_sync(0xffffffffu, pass);
}

// BI_THREADS x R rows per tile: 256 x 8 for big instances; smaller blocks (64 / 128 threads, up to 8 per SM) give
// mid-size instances (n ~ 10^4: only ~20 k evaluations per warp and pass) enough tiles to fill 148 SMs while keeping
// R = 8 rows per thread, i.e. 1.125 sqrt per evaluated move.
//
// Shared memory per block (dynamic): two column buffers (TJ+2 records) filled by TMA bulk copies, one mbarrier per stage,
// plus the tile tables.  Row records go straight from L2 into registers: a thread's R+1 rows are 16*(R+1) contiguous bytes,
// and reading them through shared memory would put all lanes of a quarter-warp on the same banks (stride 16*R bytes).
//
// SHUF: a warp owns 32 R - 1 consecutive rows instead of 32 R: lane L holds rows p0 .. p0+R-1 with p0 = warp base + L R, the
// distance of the row below its last one is lane L+1's first distance of the same column (one SHFL instead of a square root
// and four FP32 instructions), and lane 31's last row — whose lower neighbour lives in another warp — is masked out and
// scanned again as the first row of the next warp.  R square roots per R moves (minus 1/32R): the algorithmic minimum.
#ifndef TSPB_BI_MINBLOCKS64
// Resident 64-thread blocks per SM the compiler must leave room for (register cap 65536 / (64 x this)).  Measured on B200,
// 64 x 8 x 256 row-shuffle kernel at n = 100 000 (profiles/r2_blocks_per_sm_ab.jsonl): 8 blocks (100 registers) 1288 us per
// pass, 10 blocks (94 registers, no spills) 1276 us — and 184 vs 189 us for one rank's share of eight —, 12 blocks (80
// registers, spills) 1321 us.  engine.cu (bi_blocks_per_sm) sizes the grid to match.  The pruned variants (more live state: they
// would spill under the lower cap) keep 8.
#define TSPB_BI_MINBLOCKS64 10
#endif
// PF: stage-1 prefilter (bi_scan_kernel: exhaustive scans with a large share of pairs per rank, engine.cu) or the square-root
// filter alone (bi_scan_sqrt_kernel: pruned passes, smaller shares, option "prefilter" = 0).
template <int BI_THREADS, int R, bool ATT, bool EXACT32, bool PRUNED, bool SHUF, bool PF>
__device__ __forceinline__ void bi_scan_body(const BiArgs &A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bars[2];
    __shared__ int s_hint;
    __shared__ int s_last;
    __shared__ MoveKey s_keys[BI_THREADS / 32];
    __shared__ int s_ap[3];

    Ctl *ctl = A.tour.ctl;
    const int tid = threadIdx.x;
    // Programmatic dependent launch: let the apply kernel queue up behind us right away, and do everything that does not
    // depend on the previous kernel (barrier init, the static tile tables) before waiting for it.
    pdl_launch_dependents();
    const int n = A.inst.n;
    const int TJ = A.TJ;
    constexpr int TI = SHUF ? (BI_THREADS / 32) * (32 * R - 1) : BI_THREADS * R;  // rows (moves) of a tile
    const float W = A.inst.W;
    const float4 *rec = A.tour.rec;
    float4 *scols0 = reinterpret_cast<float4 *>(smem_raw);
    float4 *scols1 = scols0 + (TJ + 2);
    const unsigned col_bytes = (unsigned)(TJ + 1) * 16u;

    // PF: the stage-1 column operands of the current tile, written after its bulk copy has landed (one stage: the end-of-tile
    // barrier orders the next tile's writes after this one's reads).  s_v[j] = {X'_j, X'_j, Y'_j, Y'_j}, so one LDS.128 gives
    // both broadcast pairs of the packed FMAs; s_b[j] = B_j.
    float4 *s_v = scols1 + (TJ + 2);                                       // [TJ+2] (PF only)
    float *s_b = reinterpret_cast<float *>(s_v + (TJ + 2));                // [TJ+4] (PF only)
    // tile tables -> shared memory (one coalesced L2 round trip instead of a dependent chain per binary-search step)
    int *s_rs = PF ? reinterpret_cast<int *>(s_b + (TJ + 4))
                   : reinterpret_cast<int *>(scols1 + (TJ + 2));  // [ntr+1] prefix sums of tiles per tile-row
    int *s_rj = s_rs + (A.ntr + 1);                          // [ntr]   first tile column of each tile-row
    __shared__ float s_pfthr;                                // PF: the block's threshold of the tile's bounds
    for (int k = tid; k <= A.ntr; k += BI_THREADS) {
        s_rs[k] = A.tile_row_start[k];
        if (k < A.ntr) s_rj[k] = A.tile_row_j0[k];
    }
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    pdl_wait();  // the previous kernel of the stream (apply / upload) is complete and its writes are visible
    // everything the prologue needs from global memory is requested at once (ONE L2 round trip instead of a chain of four
    // dependent ones, ~0.5 us each: at n = 10 000 a pruned pass has one small tile per block and nothing to hide them behind)
    const int done = *((volatile int *)&ctl->done);
    const int hint0 = *((volatile int *)&ctl->hint);
    const unsigned live_count0 = PRUNED ? __ldcg(&ctl->live_count) : 0u;
    int2 live_first = make_int2(0, 0);
    if (PRUNED && tid == 0) live_first = __ldcg(&A.tour.live[blockIdx.x]);  // in bounds whatever live_count is (engine.cu)
    if (tid == 0) s_hint = hint0;
    if (done) {  // local optimum already reached: later launches of the same batch return at once
        if (blockIdx.x == 0 && tid == 0) ctl->ap_valid = 0;
        return;
    }
    if (A.timing && tid == 0) {
        const unsigned long long t = globaltimer_ns();
        atomicMin(&ctl->tm_scan_first, t);
        if (A.timing == 2) {
            A.dbg[2 * blockIdx.x] = t;
            if (PRUNED) {  // phase stamps: pruned variants only, so that the exhaustive (headline) kernel's code is not touched
                for (int k = 0; k < 8; ++k) A.dbg[8192 + 8 * blockIdx.x + k] = 0;
                A.dbg[8192 + 8 * blockIdx.x] = t;
            }
        }
    }
    __syncthreads();

    // This block's own winner of the previous pass is most likely still a legal move: its exact delta now is a valid
    // bound for this pass (see seed_hint_from_candidates).  One thread re-evaluates it while the first tile is in
    // flight; the result tightens s_hint / ctl->hint asynchronously.
    if (A.seed_hint && tid == BI_THREADS - 32) {
        const MoveKey c = key_load_cg(&A.tour.block_best[blockIdx.x]);
        const long long d = legal_move_delta_cg(A.inst, A.tour, c);
        if (d < 0) {
            atomicMin(&s_hint, (int)d);
            atomicMin(&ctl->hint, (int)d);
        }
    }

    MoveKey best = key_none();
    float thr = (float)s_hint + W;
    int pend_hint = 0;  // tid 0: value of ctl->hint fetched 64 columns ago
    // PF: tid 0 keeps it in shared memory instead: in a register it would be live across the hit handling of every block,
    // and the 96-register prefilter kernels for coordinates FP32 cannot hold would spill it to local memory
    __shared__ int s_pend_hint;
    if (PF && tid == 0) s_pend_hint = 0;

    // Tiles are DRAWN, not dealt: ctl->tile_next counts this rank's tiles handed out beyond the first wave (rank r owns
    // the tile ids r, r + world, ...; every tile costs the same — masked and padded pairs are computed too), so the blocks
    // run dry within one tile of each other whatever slows some of them down (exact-path calls, the far die's L2
    // latency).  Static dealing left the SMs idle ~10 % of a pass once a pass is only ~5 tiles deep (8 ranks).
    // [stage] = {P0, Q0, valid, columns}, written by thread 0 one tile ahead.  The 4th word (the tile width, TJ for every tile)
    // keeps a stage 16 bytes; with the 12-byte layout ptxas moved the hot loop's counter and shared-memory addresses from the
    // uniform datapath into vector registers (+5 % pass time at n = 100 000; tests/test_codegen.py watches the SASS)
    __shared__ __align__(16) int s_tile[2][4];

    // tile id -> (tile row I, tile column J)
    auto decode = [&](int t, int &P0, int &Q0) {
        int lo = 0, hi = A.ntr - 1;
        while (lo < hi) {
            int mid = (lo + hi + 1) >> 1;
            if (s_rs[mid] <= t) lo = mid; else hi = mid - 1;
        }
        P0 = lo * TI;
        Q0 = (s_rj[lo] + (t - s_rs[lo])) * TJ;
    };
    // thread 0: take the next tile, start the bulk copy of its column records, publish it for stage b.  A block's first
    // tile is its block index (no atomic on the critical path of the prologue); the following ones are drawn from the
    // counter, which therefore counts from gridDim.x.  tiles_rank <= gridDim.x (one wave, n <~ 10^4) never touches it.
    // Exact tile pruning (A.pruned): the tiles come from this rank's live list (tile_filter_kernel); a live tile whose lower
    // bound meanwhile exceeds the best exact delta found in this pass is dropped at the draw (it cannot hold the argmin
    // nor a tie: ties need delta == best).
    // Exact tile pruning (PRUNED): the tiles come from this rank's live list (tile_filter_kernel); a live tile whose lower
    // bound meanwhile exceeds the best exact delta found in this pass is dropped at the draw (it cannot hold the argmin nor
    // a tie: ties need delta == best).  The exhaustive kernel keeps the loop-free draw: a loop inside this thread-0-only
    // region makes the compiler give up the uniform datapath for the hot loop's counter and shared-memory addresses
    // (+4 % pass time at n = 100 000, measured).
    const long long tiles_rank = PRUNED ? (long long)live_count0
                                        : ((long long)A.ntiles - A.rank + A.world - 1) / A.world;
    unsigned scanned = 0;  // thread 0: tiles this block really scanned (statistics of the pruned mode)
    unsigned next_raw = 0; // thread 0, pruned mode: ticket requested one draw ahead
    auto draw = [&](int b, bool first) {
        int P = 0, Q = 0, valid = 0;
        if (!PRUNED) {
            long long kl = first ? (long long)blockIdx.x : tiles_rank;
            if (!first && tiles_rank > (long long)gridDim.x) kl = (long long)gridDim.x + (long long)atomicAdd(&ctl->tile_next, 1u);
            if (kl < tiles_rank) {
                decode((int)((long long)A.rank + (long long)A.world * kl), P, Q);
                valid = 1;
            }
        } else {
            // pruned tiles are small (a few us): the ticket of the NEXT draw is requested as soon as this one is taken, so the
            // atomic's L2 round trip overlaps the tile instead of preceding it
            const bool counted = tiles_rank > (long long)gridDim.x;
            for (;;) {
                long long kl = first ? (long long)blockIdx.x : (counted ? (long long)gridDim.x + (long long)next_raw : tiles_rank);
                if (kl >= tiles_rank) break;
                const int2 ent = first ? live_first : __ldcg(&A.tour.live[kl]);
                first = false;
                if (counted) next_raw = atomicAdd(&ctl->tile_next, 1u);
                if (__int_as_float(ent.y) > (float)(*((volatile int *)&s_hint))) continue;
                decode(ent.x, P, Q);
                valid = 1;
                scanned += 1;
                break;
            }
        }
        if (valid) {
            mbar_expect_tx(&bars[b], col_bytes);
            tma_load_1d(b ? scols1 : scols0, rec + Q, col_bytes, &bars[b]);
        }
        s_tile[b][0] = P;
        s_tile[b][1] = Q;
        s_tile[b][2] = valid;
        s_tile[b][3] = TJ;
    };

    if (tid == 0) draw(0, true);
    __syncthreads();
    int P0 = s_tile[0][0], Q0 = s_tile[0][1], NCv = s_tile[0][3];
    bool have = s_tile[0][2] != 0;
    if (PRUNED && A.timing == 2 && tid == 0) A.dbg[8192 + 8 * blockIdx.x + 1] = globaltimer_ns();  // first tile drawn, its copy in flight

    for (int it = 0; have; ++it) {
        const int buf = it & 1;
        const unsigned parity = (unsigned)(it >> 1) & 1u;
        const float4 *sc = buf ? scols1 : scols0;
        // prefetch the next tile into the other stage (its slot in s_tile / scols was last read two tiles ago; only the bulk
        // copy writes scols, so no proxy fence is needed)
        if (tid == 0) draw(buf ^ 1, false);

        // rows of this thread: p0 .. p0+R-1 in packed pairs (+ successor row p0+R, scalar)
        const int p0 = SHUF ? P0 + (tid >> 5) * (32 * R - 1) + (tid & 31) * R : P0 + tid * R;
        f32x2 xr2[R / 2], yr2[R / 2], cp2[R / 2];
        float xrl, yrl;
#pragma unroll
        for (int k = 0; k < R / 2; ++k) {
            const float4 v0 = __ldg(&rec[p0 + 2 * k]), v1 = __ldg(&rec[p0 + 2 * k + 1]);
            // "+ 0" is a real FADD2 (not an identity for -0.0, so it is never folded): its 64-bit result is an aligned
            // register pair that stays live across the column loop, instead of being re-packed with MOVs per step.
            // PF: the translated coordinates X' = x - c (exact, see pf_dot_const)
            const f32x2 zero2 = f2pack(0.f, 0.f);
            if (PF) {
                xr2[k] = f2sub(f2pack(v0.x, v1.x), f2pack(A.pf_cx, A.pf_cx));
                yr2[k] = f2sub(f2pack(v0.y, v1.y), f2pack(A.pf_cy, A.pf_cy));
            } else {
                xr2[k] = f2add(f2pack(v0.x, v1.x), zero2);
                yr2[k] = f2add(f2pack(v0.y, v1.y), zero2);
            }
            cp2[k] = f2sub(zero2, f2pack(v0.z, v1.z));  // padding rows carry ds = -BIG -> cp = +BIG -> never a candidate
        }
        if (!SHUF) {
            const float4 v = __ldg(&rec[p0 + R]);
            xrl = PF ? v.x - A.pf_cx : v.x;
            yrl = PF ? v.y - A.pf_cy : v.y;
        } else {
            // PF: the row below this lane's rows is the next lane's first one (lane 31 gets its own: finite, and masked)
            xrl = PF ? __shfl_down_sync(0xffffffffu, f2lo(xr2[0]), 1) : 0.f;
            yrl = PF ? __shfl_down_sync(0xffffffffu, f2lo(yr2[0]), 1) : 0.f;
            // lane 31's last row has its lower neighbour in another warp: never a candidate here (it is the next warp's first
            // row).  PF: -ds = BIG gives pf = -inf, hence A = +inf (pf_dot_const)
            if ((tid & 31) == 31) cp2[R / 2 - 1] = f2pack(f2lo(cp2[R / 2 - 1]), TSPB_BIG);
        }
        thr = fminf(thr, (float)(*((volatile int *)&s_hint)) + W);

        mbar_wait(&bars[buf], parity);
        if (PRUNED && A.timing == 2 && tid == 0 && it == 0) A.dbg[8192 + 8 * blockIdx.x + 2] = globaltimer_ns();  // rows and columns of the first tile are here

        // PF: stage-1 operands of this tile (see pf_dot_const), from ONE threshold for the whole block (thread 0's snapshot;
        // every thread's thr is lowered to it, so h bounds every lane's (thr + E) / 2 until the end of the tile, when thr may
        // have fallen: an older, larger h only admits more pairs).  Row pair k = rows (2k, 2k+1): w0 = -2 X', w1 = -2 Y' of
        // those rows, w2 = -2 X', w3 = -2 Y' of the rows below them (2k+1, 2k+2), A2 = the row constants.  The column operands
        // go to s_v / s_b once per tile; the bulk-copied records keep the original coordinates and ds for stages 2 and 3.
        f32x2 w0[R / 2], w1[R / 2], w2[R / 2], w3[R / 2], A2[R / 2];
        if (PF) {
            if (tid == 0) s_pfthr = (float)(*((volatile int *)&s_hint)) + W;
            __syncthreads();
            thr = fminf(thr, s_pfthr);
            const float h = 0.5f * (s_pfthr + A.pf_slack);
            for (int j = tid; j <= NCv; j += BI_THREADS) {
                const float4 c = sc[j];
                const float x = c.x - A.pf_cx, y = c.y - A.pf_cy;
                s_v[j] = make_float4(x, x, y, y);
                if (j < NCv) {
                    const float4 c1 = sc[j + 1];
                    const float x1 = c1.x - A.pf_cx, y1 = c1.y - A.pf_cy;
                    s_b[j] = pf_dot_const(fmaf(y, y, x * x) + fmaf(y1, y1, x1 * x1), pf_bound<ATT>(c.z, h));
                }
            }
            const f32x2 m2 = f2pack(-2.f, -2.f);
#pragma unroll
            for (int k = 0; k < R / 2; ++k) {
                const f32x2 x1 = f2pack(f2hi(xr2[k]), k + 1 < R / 2 ? f2lo(xr2[(k + 1) % (R / 2)]) : xrl);
                const f32x2 y1 = f2pack(f2hi(yr2[k]), k + 1 < R / 2 ? f2lo(yr2[(k + 1) % (R / 2)]) : yrl);
                const f32x2 nrm = f2add(f2fma(yr2[k], yr2[k], f2mul(xr2[k], xr2[k])), f2fma(y1, y1, f2mul(x1, x1)));
                w0[k] = f2mul(xr2[k], m2);
                w1[k] = f2mul(yr2[k], m2);
                w2[k] = f2mul(x1, m2);
                w3[k] = f2mul(y1, m2);
                // cp2 holds -ds (padding / masked rows: -BIG -> pf = -inf -> A = +inf)
                A2[k] = f2pack(pf_dot_const(f2lo(nrm), pf_bound<ATT>(-f2lo(cp2[k]), h)),
                               pf_dot_const(f2hi(nrm), pf_bound<ATT>(-f2hi(cp2[k]), h)));
            }
            __syncthreads();
        }

        // pairs with q < p+2 exist in this tile?  (mask them; they are mirrored / adjacent pairs)
        const bool diag = (Q0 < P0 + TI + 1);
        const int NC = PRUNED ? NCv : TJ;  // columns of this tile
        // first column of the scan: D0 -> U2 (kept per variant so that the regular tile's shared-memory addressing stays uniform)
        // PF: the column operands of q (qx, qy: {X'_q, X'_q}, {Y'_q, Y'_q}) and of q + 1 (vnext).  The 64-thread kernels (96
        // registers) read them from s_v at the start of every BI_CB block and carry them within it only: nothing of the
        // columns stays live across the hit handling (a noinline call), which keeps them free of spills.  The larger blocks
        // have registers to spare and carry them from block to block (CARRY), which keeps their addressing uniform.
        constexpr bool CARRY = BI_THREADS != 64;
        float4 c0, cnext, vnext;
        f32x2 U2[R / 2], qx, qy;
#define BI_INIT(JB)                                                                                    \
    if constexpr (PF) {                                                                                \
        if (CARRY) {                                                                                   \
            const float4 v0 = s_v[(JB)];                                                               \
            qx = f2pack(v0.x, v0.y);                                                                   \
            qy = f2pack(v0.z, v0.w);                                                                   \
            vnext = s_v[(JB) + 1];                                                                     \
        }                                                                                              \
    } else {                                                                                           \
        c0 = sc[(JB)];                                                                                 \
        cnext = sc[(JB) + 1];                                                                          \
        float D0[R + 1];                                                                               \
        column_dists<R, ATT, SHUF ? 0 : 1>(xr2, yr2, xrl, yrl, c0.x, c0.y, D0);                        \
        _Pragma("unroll") for (int k = 0; k < R / 2; ++k) U2[k] = f2add(f2pack(D0[2 * k], D0[2 * k + 1]), cp2[k]); \
    }
#define UU(r_) (((r_) & 1) ? f2hi(U2[(r_) >> 1]) : f2lo(U2[(r_) >> 1]))

// one column: R+1 fresh distances -> R move deltas Q[r] = (D[p_r][q] - ds_p) + D[p_r+1][q+1]; the filter quantity
// min_r Q[r] - ds_q is folded into the running block minimum M (no branch, no per-pair state kept).
// PF: acc = A_p + w_p . v_q, four packed FMAs per row pair; min_r acc + B_q is folded into M (bq: B of this block's columns)
#define BI_COL(DIAG, jj_, c_)                                                                          \
    if constexpr (PF) {                                                                                \
        const float4 v1 = vnext;                                                                       \
        if (CARRY) vnext = s_v[(jj_) + 2]; /* prefetched one column ahead */                           \
        else if ((c_) + 1 < BI_CB) vnext = svj[(c_) + 2]; /* ... within the block */                   \
        const f32x2 q1x = f2pack(v1.x, v1.y), q1y = f2pack(v1.z, v1.w);                                \
        float m = TSPB_BIG;                                                                            \
        _Pragma("unroll") for (int k = 0; k < R / 2; ++k) {                                            \
            f32x2 acc = f2fma(w0[k], qx, A2[k]);                                                       \
            acc = f2fma(w1[k], qy, acc);                                                               \
            acc = f2fma(w2[k], q1x, acc);                                                              \
            acc = f2fma(w3[k], q1y, acc);                                                              \
            float a0 = f2lo(acc), a1 = f2hi(acc);                                                      \
            if (DIAG) {                                                                                \
                a0 = (qrel0 + (jj_) >= 2 * k + 2) ? a0 : TSPB_BIG;                                     \
                a1 = (qrel0 + (jj_) >= 2 * k + 3) ? a1 : TSPB_BIG;                                     \
            }                                                                                          \
            m = fminf(m, fminf(a0, a1));                                                               \
        }                                                                                              \
        M = fminf(M, m + bq[(c_)]);                                                                    \
        qx = q1x;                                                                                      \
        qy = q1y;                                                                                      \
    } else {                                                                                           \
        const float4 c1 = cnext;                                                                       \
        cnext = sc[(jj_) + 2]; /* prefetched one column ahead */                                       \
        float Dn[R + 1];                                                                               \
        column_dists<R, ATT, SHUF ? 2 : 1>(xr2, yr2, xrl, yrl, c1.x, c1.y, Dn);                        \
        float m = TSPB_BIG;                                                                            \
        _Pragma("unroll") for (int r = 0; r < R; ++r) {                                                \
            float qv = UU(r) + Dn[r + 1];                                                              \
            if (DIAG) qv = (qrel0 + (jj_) >= r + 2) ? qv : TSPB_BIG;                                   \
            m = fminf(m, qv);                                                                          \
        }                                                                                              \
        M = fminf(M, m - c0.z);                                                                        \
        _Pragma("unroll") for (int k = 0; k < R / 2; ++k)                                              \
            U2[k] = f2add(f2pack(Dn[2 * k], Dn[2 * k + 1]), cp2[k]);                                   \
        c0 = c1;                                                                                       \
    }

// BI_CB columns, then ONE filter check per warp (ballot); hits are resolved one lane at a time by the whole warp
// (PF: a stage-1 hit first goes through stage 2, the square-root filter, and only its survivors to the exact path)
#define BI_BLOCK(DIAG)                                                                                 \
    for (int jj = 0; jj < NC; jj += BI_CB) {                                                           \
        float M = TSPB_BIG;                                                                            \
        const float4 b4 = PF ? *reinterpret_cast<const float4 *>(s_b + jj) : make_float4(0.f, 0.f, 0.f, 0.f); \
        const float bq[BI_CB] = {b4.x, b4.y, b4.z, b4.w};                                              \
        /* s_v + jj, spelled from s_b + jj: this form keeps the addresses in uniform registers */      \
        const float4 *svj = reinterpret_cast<const float4 *>(s_b + 4 * jj) - (TJ + 2);                 \
        if (PF && !CARRY) {                                                                            \
            const float4 v0 = svj[0];                                                                  \
            qx = f2pack(v0.x, v0.y);                                                                   \
            qy = f2pack(v0.z, v0.w);                                                                   \
            vnext = svj[1];                                                                            \
        }                                                                                              \
        _Pragma("unroll") for (int c = 0; c < BI_CB; ++c) { BI_COL(DIAG, jj + c, c) }                  \
        unsigned hits = __ballot_sync(0xffffffffu, M <= (PF ? 0.f : thr));                             \
        while (hits) {                                                                                 \
            const int L = __ffs(hits) - 1;                                                             \
            const float thrL = __shfl_sync(0xffffffffu, thr, L);                                       \
            const int pL = p0 + (L - (tid & 31)) * R;                                                  \
            bool cold = true;                                                                          \
            if (PF) {                                                                                  \
                if ((tid & 31) == L) atomicAdd(&ctl->pf_hits, 1ull);                                   \
                cold = bi_refilter_warp<R, ATT>(rec, sc, n, pL, Q0, jj, thrL);                         \
            }                                                                                          \
            if (cold) {                                                                                \
                const MoveKey nb = bi_cold_warp<R, ATT, EXACT32>(A.inst, rec, sc, n, pL, Q0, jj, thrL                   \
                                                                 TSPB_PROBE_ARG(SHUF && L == 31 ? R - 1 : R)); \
                if ((tid & 31) == L) {                                                                 \
                    atomicAdd(&ctl->cold_calls, 1ull);                                                 \
                    if (key_less(nb, best)) {                                                          \
                        best = nb;                                                                     \
                        atomicMin(&s_hint, nb.delta);                                                  \
                        atomicMin(&ctl->hint, nb.delta);                                               \
                    }                                                                                  \
                }                                                                                      \
                /* an exact delta of a real move bounds the minimum for every lane: tighten all, drop stale hits */ \
                if (nb.delta < 0) thr = fminf(thr, (float)nb.delta + W);                               \
            }                                                                                          \
            hits &= hits - 1;                                                                          \
            if (!PF) hits &= __ballot_sync(0xffffffffu, M <= thr);                                     \
        }                                                                                              \
        /* every 64 columns: pick up what the other warps / blocks found (tid 0 swaps in the ctl->hint value it */ \
        /* requested 64 columns ago, so nobody waits for L2)                                                    */ \
        if ((jj & 63) == 64 - BI_CB) {                                                                 \
            if (tid == 0) {                                                                            \
                const int ph = PF ? s_pend_hint : pend_hint;                                           \
                if (ph < 0) atomicMin(&s_hint, ph);                                                    \
                if (PF) s_pend_hint = __ldcg(&ctl->hint);                                              \
                else pend_hint = __ldcg(&ctl->hint);                                                   \
            }                                                                                          \
            thr = fminf(thr, (float)(*((volatile int *)&s_hint)) + W);                                 \
        }                                                                                              \
    }

        const int qrel0 = Q0 - p0;  // q - p0 at jj = 0
        if (!diag) {
            BI_INIT(0)
            BI_BLOCK(false)
        } else {
            BI_INIT(0)
            BI_BLOCK(true)
        }
#undef BI_INIT
#undef BI_BLOCK
#undef BI_COL
#undef UU

        __syncthreads();  // every thread is done with this stage before the next prefetch overwrites it
        if (PRUNED && A.timing == 2 && tid == 0) {
            if (it == 0) A.dbg[8192 + 8 * blockIdx.x + 3] = globaltimer_ns();  // first tile scanned
            A.dbg[8192 + 8 * blockIdx.x + 5] = (unsigned long long)(it + 1);
        }
        // publish the best exact delta to the other blocks (fire and forget; theirs arrive through pend_hint above)
        if (tid == 0 && s_hint < 0) atomicMin(&ctl->hint, s_hint);
        P0 = s_tile[buf ^ 1][0];
        Q0 = s_tile[buf ^ 1][1];
        have = s_tile[buf ^ 1][2] != 0;
        NCv = s_tile[buf ^ 1][3];
    }

    // ---- block argmin -> grid argmin ("last block done") -------------------------------------------
    // packed_tail: every block folds its key into ctl->pass_min with ONE 64-bit atomicMin, so the last block only has to
    // read that word (instead of reducing gridDim.x keys: ~3 us of every pass at 1184 blocks).
    best = key_warp_min(best);
    if ((tid & 31) == 0) s_keys[tid >> 5] = best;
    __syncthreads();
    if (tid < 32) {
        MoveKey k = (tid < BI_THREADS / 32) ? s_keys[tid] : key_none();
        k = key_warp_min(k);
        if (tid == 0) {
            A.tour.block_best[blockIdx.x] = k;
            if (A.packed_tail && k.delta < 0) atomicMin(&ctl->pass_min, key_pack(k.delta, k.i, k.j));
            if (PRUNED && scanned) atomicAdd(&ctl->tiles_scanned, (unsigned long long)scanned);
            if (A.timing) {
                const unsigned long long t = globaltimer_ns();
                atomicMin(&ctl->tm_blk_end_min, t);
                if (A.timing == 2) {
                    A.dbg[2 * blockIdx.x + 1] = t;
                    if (PRUNED) A.dbg[8192 + 8 * blockIdx.x + 4] = t;  // block key folded, about to take the ticket
                }
            }
            __threadfence();
            unsigned tk = atomicAdd(&ctl->ticket, 1u);
            s_last = (tk == gridDim.x - 1);
            if (PRUNED && A.timing == 2) A.dbg[8192 + 8 * blockIdx.x + 6] = globaltimer_ns();  // ticket taken
        }
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    unsigned long long t_ticket = 0;
    if (A.timing && tid == 0) {
        t_ticket = globaltimer_ns();
        const unsigned long long t_first = ctl->tm_scan_first, ap0 = ctl->tm_apply_first, ap1 = ctl->tm_apply_end;
        ctl->tm_acc[TM_SCAN] += t_ticket - t_first;
        ctl->tm_acc[TM_SPREAD] += t_ticket - ctl->tm_blk_end_min;
        if (ap1 != 0 && ap0 != ~0ull) {  // the previous pass applied a move
            ctl->tm_acc[TM_GAP] += t_first > ap1 ? t_first - ap1 : 0;
            ctl->tm_acc[TM_APPLY] += ap1 - ap0;
            ctl->tm_acc[TM_APPLY_GAP] += ap0 > ctl->tm_publish ? ap0 - ctl->tm_publish : 0;
        }
        ctl->tm_acc[TM_COUNT] += 1;
        ctl->tm_scan_first = ~0ull;
        ctl->tm_blk_end_min = ~0ull;
        ctl->tm_apply_first = ~0ull;
        ctl->tm_apply_end = 0;
    }

    MoveKey k = key_none();
    int rounds = 1;
    if (A.packed_tail) {
        if (tid == 0) {
            const unsigned long long pk = __ldcg(&ctl->pass_min);
            ctl->pass_min = KEY_PACK_NONE;
            if (pk < KEY_PACK_NONE) {
                key_unpack(pk, &k.delta, &k.i, &k.j);
                k.pad = 0;
            }
            ctl->cand[0] = k;
        }
    } else {
        MoveKey mine = key_none();
        for (int b = tid; b < (int)gridDim.x; b += BI_THREADS) {
            MoveKey o = key_load_cg(&A.tour.block_best[b]);
            if (key_less(o, mine)) mine = o;
        }
        // CTL_NCAND rounds of "block-wide minimum, then retire it": round 0 is the winner of the pass, the rest are
        // runner-ups kept as seeds for the next pass's filter (seed_hint_from_candidates)
        rounds = (A.seed_hint >= 2) ? CTL_NCAND : 1;
#pragma unroll 1
        for (int round = 0; round < rounds; ++round) {
            MoveKey m = key_warp_min(mine);
            if ((tid & 31) == 0) s_keys[tid >> 5] = m;
            __syncthreads();
            m = s_keys[0];
#pragma unroll
            for (int w = 1; w < BI_THREADS / 32; ++w)
                if (key_less(s_keys[w], m)) m = s_keys[w];
            __syncthreads();
            if (round == 0) k = m;
            if (tid == 0) ctl->cand[round] = m;
            if (m.delta < 0 && mine.i == m.i && mine.j == m.j) mine = key_none();
        }
    }

    if (tid == 0) {
        ctl->ncand = rounds;
        ctl->last = k;
        ctl->ticket = 0;
        ctl->tile_next = 0;
        ctl->live_count = 0;
        ctl->hint = 0;
        ctl->launches += 1;
        if (!A.fuse_apply) {
            // multi-GPU: this rank's key for the exchange (peer memory below, or NCCL + the decode kernel)
            ctl->packed = (k.delta < 0) ? key_pack(k.delta, k.i, k.j) : KEY_PACK_NONE;
        } else {
            ctl->passes += 1;
            publish_move(A.tour, k.i, k.j, k.delta);
            if (k.delta >= 0) { ctl->done = 1; ctl->done_reason = DONE_OPTIMUM; }  // reference src/tabusearch.c:158: mindelta >= 0 -> stop
            s_ap[0] = ctl->ap_pa;
            s_ap[1] = ctl->ap_pb;
            s_ap[2] = k.delta < 0;
            if (A.timing) {
                const unsigned long long now = globaltimer_ns();
                ctl->tm_publish = now;
                ctl->tm_acc[TM_TAIL] += now - t_ticket;
            }
        }
    }
    // Multi-GPU exchange over peer memory, fused into this kernel's tail (xchg_min): thread r stores this rank's key word
    // into rank r's slot array (NVLink peer store), then polls this rank's LOCAL slot r until rank r's word of the same
    // epoch has arrived; the block takes the minimum — every rank gets the same winner — and publishes the move for its
    // own replica of the tour.  No collective launch and no tour data on the wire.
    if (!A.fuse_apply && A.xchg.enabled) {
        __shared__ unsigned long long s_xkey[XCHG_MAX_WORLD];
        __shared__ unsigned long long s_mine;
        __shared__ int s_err;
        if (tid == 0) {
            s_mine = ctl->packed;
            s_err = 0;
        }
        __syncthreads();
        unsigned long long wait_ns = 0;
        const unsigned long long win = xchg_min(A.xchg, A.rank, A.world, s_mine, s_xkey, &s_err, A.timing ? &wait_ns : nullptr);
        if (tid == 0) {
            int delta, i, j;
            key_unpack(win, &delta, &i, &j);
            if (s_err) {
                ctl->error = 2;
                ctl->done = 1;
                ctl->done_reason = DONE_OPTIMUM;
                ctl->ap_valid = 0;
            } else {
                ctl->passes += 1;
                publish_move(A.tour, i, j, delta);
                if (delta >= 0) { ctl->done = 1; ctl->done_reason = DONE_OPTIMUM; }
            }
            if (A.timing) {
                const unsigned long long now = globaltimer_ns();
                ctl->tm_publish = now;
                ctl->tm_acc[TM_TAIL] += now - t_ticket;
                ctl->tm_acc[TM_XWAIT] += wait_ns;
            }
        }
    }
    // fuse_apply == 2: this (last) block also applies the move, saving the apply launch — every other block has
    // finished reading rec[] before it took its ticket.  Used for mid-size tours where a launch costs more than the swap.
    if (A.fuse_apply == 2) {
        __syncthreads();  // s_ap[] (thread 0 knows the winner; in packed_tail mode nobody else does)
        if (!s_ap[2]) return;
        apply_swap_range<false>(A.inst, A.tour, s_ap[0], s_ap[1], tid, BI_THREADS);
        if (tid == 0) ctl->ap_valid = 0;
        __threadfence();
        __syncthreads();
        if (A.seed_hint) seed_hint_from_candidates(A.inst, A.tour, tid);
    }
}


#define TSPB_BI_BOUNDS \
    __launch_bounds__(BI_THREADS, (R >= 16 ? (BI_THREADS == 256 ? 1 : 384 / BI_THREADS) : (BI_THREADS == 64 && !PRUNED ? TSPB_BI_MINBLOCKS64 : 512 / BI_THREADS)))
template <int BI_THREADS, int R, bool ATT, bool EXACT32, bool PRUNED, bool SHUF>
__global__ void TSPB_BI_BOUNDS bi_scan_kernel(const BiArgs A) {
    bi_scan_body<BI_THREADS, R, ATT, EXACT32, PRUNED, SHUF, true>(A);
}
template <int BI_THREADS, int R, bool ATT, bool EXACT32, bool PRUNED, bool SHUF>
__global__ void TSPB_BI_BOUNDS bi_scan_sqrt_kernel(const BiArgs A) {
    bi_scan_body<BI_THREADS, R, ATT, EXACT32, PRUNED, SHUF, false>(A);
}
#undef TSPB_BI_BOUNDS

// ---- host-side launchers -----------------------------------------------------------------------------
template <int T, int R, bool SHUF>
static inline cudaError_t launch_bi_tr(const BiArgs &a, int grid, bool pdl, cudaStream_t st) {
    // two column stages, the prefilter's column operands (bi_scan_body: s_v, s_b), the tile tables
    const size_t smem = (size_t)2 * (a.TJ + 2) * sizeof(float4) + (size_t)(2 * a.ntr + 2) * sizeof(int) +
                        (a.prefilter ? (size_t)(a.TJ + 2) * sizeof(float4) + (size_t)(a.TJ + 4) * sizeof(float) : 0);
    const bool att = (a.inst.metric == M_ATT);
    const bool ex = a.inst.exact32 != 0;
    auto go = [&](auto kern) -> cudaError_t {
        if (smem > 48 * 1024) {  // opt in to more dynamic shared memory than the default limit (never at the supported tile widths)
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        if (!pdl) {
            kern<<<grid, T, smem, st>>>(a);
            return cudaGetLastError();
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(T);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, kern, a);
    };
#if TSPB_BI_PREFILTER_PRUNED
    if (a.prefilter && a.pruned) {
        if (att && ex) return go(bi_scan_kernel<T, R, true, true, true, SHUF>);
        if (att) return go(bi_scan_kernel<T, R, true, false, true, SHUF>);
        if (ex) return go(bi_scan_kernel<T, R, false, true, true, SHUF>);
        return go(bi_scan_kernel<T, R, false, false, true, SHUF>);
    }
#endif
    if (a.prefilter && !a.pruned) {  // the prefilter serves exhaustive scans only (engine.cu, tspb200_bi_run)
        if (att && ex) return go(bi_scan_kernel<T, R, true, true, false, SHUF>);
        if (att) return go(bi_scan_kernel<T, R, true, false, false, SHUF>);
        if (ex) return go(bi_scan_kernel<T, R, false, true, false, SHUF>);
        return go(bi_scan_kernel<T, R, false, false, false, SHUF>);
    }
    if (a.pruned) {
        if (att && ex) return go(bi_scan_sqrt_kernel<T, R, true, true, true, SHUF>);
        if (att) return go(bi_scan_sqrt_kernel<T, R, true, false, true, SHUF>);
        if (ex) return go(bi_scan_sqrt_kernel<T, R, false, true, true, SHUF>);
        return go(bi_scan_sqrt_kernel<T, R, false, false, true, SHUF>);
    }
    if (att && ex) return go(bi_scan_sqrt_kernel<T, R, true, true, false, SHUF>);
    if (att) return go(bi_scan_sqrt_kernel<T, R, true, false, false, SHUF>);
    if (ex) return go(bi_scan_sqrt_kernel<T, R, false, true, false, SHUF>);
    return go(bi_scan_sqrt_kernel<T, R, false, false, false, SHUF>);
}


}  // namespace tspb
