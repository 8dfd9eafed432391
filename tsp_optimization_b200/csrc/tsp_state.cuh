// tsp_state.cuh — device-resident instance / tour state and the block-wide move application.
//
// HBM layout (DESIGN.md §2).  A tour lives on the device in two views that are kept in sync:
//   position space  rec[p] = {x, y, ds, node}   p = 0..n-1 in visiting order (forward orientation),
//                   ds = exact integer d(node_p, node_{p+1}) stored as float, node id in the 4th word;
//                   rec[n] mirrors rec[0]'s coordinates with ds = -BIG (wrap-around successor of p=n-1);
//                   everything after is padding with ds = -BIG (never a candidate).
//                   pos[node] = p.
//   node space      nrec[k] = {x_k, y_k, x_succ(k), y_succ(k)}, nlnk[k] = {d(k, succ k), succ k, d(pred k, k), pred k},
//                   npxy[k] = {x_pred(k), y_pred(k)}  (first-improvement search only: it scans node-index order).
//                   Doubly linked so that a reversal is a LOCAL update of every node on the reversed path — its successor
//                   and predecessor halves trade places — which the apply kernel does in the same pass as the swap.
// The reference keeps edges[k].j = succ(k) and a prev[] array (reference include/utility.h:131-145,
// src/heuristics.c:444-448); succ[] is rebuilt from rec[] when a tour is downloaded.
#pragma once
#include "tsp_device.cuh"

namespace tspb {

#ifndef TSPB_FILTER_PROBE
// 1: the filter probe build (make OUT=../lib/probe EXTRA=-DTSPB_FILTER_PROBE=1; tests/test_gpu_filter_probe.py).  Option
// "probe" = H <= -1 pins the threshold of the next best-improvement pass at H + W (nothing lowers it: the cold paths record
// and return no key, no seed tightens the hint), and the cold paths record every pair of their R x 4 block whose exact
// delta is <= H.  The product build keeps it 0: none of this exists there.
#define TSPB_FILTER_PROBE 0
#endif

#if TSPB_FILTER_PROBE
struct ProbeRec {  // one pair seen by a cold path: node ids i < j, exact delta, the FP32 filter value, threshold and verdict
    int i, j, delta;
    float qv, thr;
    int passed, pad0, pad1;
};
#define TSPB_PROBE_ARG(x) , x
#define TSPB_PROBE_OR(x) || (x)
#else
#define TSPB_PROBE_ARG(x)
#define TSPB_PROBE_OR(x)
#endif

struct InstDev {
    int n;
    int metric;             // reference weight_type value
    int exact32;            // every coordinate is exactly representable in FP32
    int fp32_ok;            // FP32 filter path usable (metric in EUC/CEIL/ATT, |coords| small enough)
    int int_coords;         // every coordinate is an integer (and exact32): rounding decisions reduce to exact compares
    float W;                // filter window (see DESIGN.md §3): candidate iff Q <= best + W
    float band;             // matrix kernel guard band, relative to r
    const double2 *pt64;    // node-indexed exact points (GEO: lat/lon radians)
    const float2 *pt32;     // node-indexed FP32 points
    const int *dmat;        // optional n x ld int32 distance matrix (matrix mode), else nullptr
    long long dmat_ld;
#if TSPB_FILTER_PROBE
    int probe_on;                    // the threshold is pinned at probe_H + W and the cold paths record
    int probe_H;
    ProbeRec *probe_rec;             // [probe_cap]
    unsigned long long *probe_count; // records appended (beyond probe_cap: counted, not written)
    long long probe_cap;
#endif
};

#if TSPB_FILTER_PROBE
__device__ __forceinline__ void probe_record(const InstDev &I, int u, int v, long long delta, float qv, float thr, bool passed) {
    const unsigned long long k = atomicAdd(I.probe_count, 1ull);
    if ((long long)k < I.probe_cap) {
        ProbeRec r;
        r.i = min(u, v); r.j = max(u, v); r.delta = (int)delta;
        r.qv = qv; r.thr = thr; r.passed = passed ? 1 : 0; r.pad0 = r.pad1 = 0;
        I.probe_rec[k] = r;
    }
}
#endif

struct MoveRec {  // one applied move, as logged for parity tests
    int i, j;
    long long delta;
};

struct Ctl {
    int done;                       // 1 = local optimum reached (all later launches return at once)
    int error;                      // device-side consistency check failed
    unsigned ticket;                // block completion counter of the current launch
    int hint;                       // best exact delta found so far in the current BI pass (<= 0)
    long long passes;               // BI: completed scans; FI: completed sweeps
    long long moves;                // applied moves
    long long obj_delta;            // sum of applied deltas
    long long launches;             // kernel launches that did work
    long long sweep_moves;          // FI: moves applied in the current sweep
    int cur_i, cur_j;               // FI cursor (next pair to look at, node-index order)
    unsigned long long fi_found;    // FI: min linear index i*n+j of an improving pair in this launch
    unsigned long long packed;      // multi-GPU: this rank's packed best key for the NCCL min-allreduce
    long long log_count;
    long long max_moves;            // FI only: stop after this many moves (<0 = unlimited)
    long long pairs_swept;          // FI: linear pairs covered (statistics only)
    MoveKey last;                   // last selected key
    int ap_pa, ap_pb, ap_valid;     // move to apply: positions of a and b (published by the selecting kernel)
    unsigned apply_ticket;          // block completion counter of the apply launch
    unsigned fi_seg;                // FI: next segment of the row-major pair order to hand to a block
    unsigned tile_next;             // BI: this rank's tiles handed out so far in the current pass
    MoveKey cand[4];                // runner-up moves of the last BI pass: re-evaluated after the apply to seed `hint`
    int ncand;
    unsigned long long cold_calls;  // statistics: filter hits that went through the exact (cold) path
    unsigned long long pf_hits;     // statistics: stage-1 prefilter hits (warp ballot blocks), each re-checked by the FP32 filter
    unsigned long long pass_min;    // BI: packed (delta,i,j) minimum of the running pass (one atomicMin per block)
    int done_reason;                // why `done` is set: DONE_OPTIMUM or DONE_CAP (a capped run may be continued)
    // first improvement on several GPUs: 1 = the next search deals its segments over the ranks and exchanges the winner,
    // 0 = every rank searches alone from the cursor (identical results, no exchange).  Decided after every search from the
    // number of pairs it had to sweep — the same number on every rank — so all ranks always agree.
    int fi_shard;
    // single GPU ("late selection"): the search kernels only fold their hits into fi_sel[parity of the launch]; the apply
    // launch that follows reads the winner itself, applies it and does the bookkeeping, so the search kernel has no
    // "last block" tail.  The other parity's word is reset by that apply launch for the next search.
    unsigned long long fi_sel[2];
    // ... every thread of that apply launch reads pos[b] to find the range, so the ONE position entry the launch itself would
    // overwrite under their eyes — pos[b], written by swap 0 — is parked here and stored by the next search launch (which never
    // reads pos[]) or by fi_flush_kernel at the end of the run.
    int fi_pend_node, fi_pend_pos;   // fi_pend_node < 0: nothing parked
    int fi_mode[2];                  // per launch parity: 1 = that search was sharded and published its move itself (several GPUs)
    long long fi_shard_min_gap;     // pairs swept by the last search above which the next one is sharded
    // exact tile pruning (DESIGN.md §4.8): this rank's live tiles of the coming pass, built by tile_filter_kernel
    unsigned live_count;            // entries in TourDev::live
    unsigned long long tiles_scanned, tiles_skipped;  // statistics over all pruned passes
    // per-pass timing breakdown (option "timing"): %globaltimer stamps of the running pass and accumulated intervals
    unsigned long long tm_scan_first, tm_blk_end_min, tm_apply_first, tm_apply_end, tm_publish;
    unsigned long long tm_acc[8];   // see TM_* below
};
constexpr int CTL_NCAND = 4;
constexpr int PRUNE_GROUP = 16;  // tile-columns per coarse box of the two-level tile filter
enum { DONE_NONE = 0, DONE_OPTIMUM = 1, DONE_CAP = 2 };
// tm_acc slots, all in ns summed over passes: gap between the previous apply's end and the first scan block's start,
// scan (first block start -> last block's ticket), spread (first block end -> last block end), tail (ticket -> move
// published, includes the exchange), exchange wait alone, publish -> first apply block, apply duration, pass count
enum { TM_GAP = 0, TM_SCAN = 1, TM_SPREAD = 2, TM_TAIL = 3, TM_XWAIT = 4, TM_APPLY_GAP = 5, TM_APPLY = 6, TM_COUNT = 7 };

struct TourDev {
    int n;
    int alloc;        // entries allocated in rec
    float4 *rec;
    int *pos;
    float4 *nrec;     // node space (first improvement): {x, y, x_succ, y_succ}
    float4 *nlnk;     //   {ds = d(k, succ), succ (int bits), pds = d(pred, k), pred (int bits)}
    float2 *npxy;     //   {x_pred, y_pred}
    Ctl *ctl;
    MoveKey *block_best;
    MoveRec *log;
    long long log_cap;
    // exact tile pruning: bounding boxes {xmin, ymin, xmax, ymax} and largest edge length of every tile-row (TI positions
    // + the successor of the last one) and tile-column (TJ positions + successor); live tile ids + their lower bounds
    float4 *rowbox, *colbox, *colbox2;   // colbox2: groups of PRUNE_GROUP consecutive tile-columns (first level of the filter)
    float *rowmaxds, *colmaxds, *colmaxds2;
    int2 *live;       // {tile id, lower bound of the tile's deltas (float bits)}: one 8-byte load per draw
};

#define FI_NONE 0xffffffffffffffffull

#ifndef TSPB_BI_PREFILTER_PRUNED
// 1: pruned passes run the stage-1 prefilter kernel too.  Measurement builds only (make EXTRA=-DTSPB_BI_PREFILTER_PRUNED=1
// OUT=...): it is slower there (profiles/r3_prefilter_pruned.jsonl), so the product build keeps it 0.
#define TSPB_BI_PREFILTER_PRUNED 0
#endif

__device__ __forceinline__ int node_of(const float4 &r) { return __float_as_int(r.w); }

// distance between two nodes by id, exact (matrix lookup when a matrix is resident).
__device__ __forceinline__ long long dist_nodes(const InstDev &I, int u, int v) {
    if (I.dmat) return (long long)I.dmat[(long long)u * I.dmat_ld + v];
    return exact_dist(I.metric, I.pt64[u], I.pt64[v]);
}

// Application of the 2-opt move (i,j), i<j node ids, exactly as the reference does it:
//   a=i, b=j, a1=succ[a], b1=succ[b]; succ[a]=b; succ[a1]=b1; reverse_path(b, a1)
// (reference src/heuristics.c:476-483, src/tabusearch.c:161-165, src/utility.c:708-722): the FORWARD path
// a1 -> ... -> b is reversed, wrap-around included, never "the shorter side", so the orientation of the
// tour — and with it the (i,j) -> (a1,b1) mapping of every later move — stays the reference's.
// In position space that is an in-place reversal of the cyclic range [pa+1, pb], pa = pos[a], pb = pos[b].
//
// The selecting kernel publishes (pa, pb) in Ctl; this routine is then run by a whole GRID (gtid of gthreads
// threads) with no synchronisation at all: every swap t touches only positions s+t and e-t, the edge-length
// reversal touches only the .z words of s..e-1, and the thread that owns swap 0 knows all four end nodes
// (a, a1, b, b1) from its own loads, so it also writes the two new edge lengths.
// NODE = true (first improvement) also keeps the node-space view current, with no extra launch and no extra
// synchronisation: on the reversed path a1..b every node's successor and predecessor trade places, which touches only
// that node's own node-space words; the thread that swaps positions s+t and e-t owns the two nodes it moves (the middle
// node of an odd-length path gets an iteration of its own), and the thread of swap 0 — which holds a1 and b and reads a
// and b1 anyway — writes the four boundary links (a -> b, a1 -> b1 and their back links).
__device__ __forceinline__ void node_flip(const TourDev &T, int k) {
    const float4 r = T.nrec[k];
    const float4 l = T.nlnk[k];
    const float2 p = T.npxy[k];
    T.nrec[k] = make_float4(r.x, r.y, p.x, p.y);
    T.nlnk[k] = make_float4(l.z, l.w, l.x, l.y);
    T.npxy[k] = make_float2(r.z, r.w);
}

// delta_out (may be null): the thread of swap 0 — global thread 0 — stores the exact delta of the move it applied,
// d(a,b) + d(a1,b1) - d(a,a1) - d(b,b1), from the edge lengths it reads and writes anyway.
// park_pos_b (may be null): swap 0 does NOT store pos[b]; the thread gets {b, new position of b} back instead (see Ctl::fi_pend_*).
template <bool NODE>
__device__ __forceinline__ void apply_swap_range(const InstDev &I, const TourDev &T, int pa, int pb, int gtid, int gthreads,
                                                 long long *delta_out = nullptr, int2 *park_pos_b = nullptr) {
    const int n = T.n;
    float4 *rec = T.rec;
    int s = pa + 1;
    if (s >= n) s -= n;
    int len = pb - pa;
    if (len < 0) len += n;  // number of nodes on the path a1..b
    const int e = pb;
    const int half = len >> 1;         // record swaps: positions s+t <-> e-t
    const int mhalf = (len - 1) >> 1;  // inner edge lengths (positions s .. e-1) reversed among themselves: s+t <-> e-1-t
    const int iters = NODE ? half + (len & 1) : half;
    // One iteration = record swap t AND edge-length swap t, all loads issued before the first store: one L2 round trip.
    // No two threads touch the same word: swap t owns {x,y,node} of s+t and e-t and the edge lengths of s+t and e-1-t.
    for (int t = gtid; t < iters; t += gthreads) {
        int A = s + t;
        if (A >= n) A -= n;
        if (NODE && t == half) {  // middle node of an odd-length path: it stays where it is, only its links flip
            node_flip(T, node_of(rec[A]));
            continue;
        }
        int B = e - t;
        if (B < 0) B += n;
        int Bm = B - 1;
        if (Bm < 0) Bm += n;
        const bool dsw = t < mhalf;
        const float2 xa = *reinterpret_cast<const float2 *>(&rec[A].x);
        const float wa = rec[A].w;
        const float2 xb = *reinterpret_cast<const float2 *>(&rec[B].x);
        const float wb = rec[B].w;
        float za = 0.f, zc = 0.f;
        if (dsw) {
            za = rec[A].z;
            zc = rec[Bm].z;
        }
        const int ka = __float_as_int(wa), kb = __float_as_int(wb);
        float4 nra, nla, nrb, nlb;
        float2 npa, npb;
        if (NODE) {  // second (dependent) round trip, issued before the stores below
            nra = T.nrec[ka]; nla = T.nlnk[ka]; npa = T.npxy[ka];
            nrb = T.nrec[kb]; nlb = T.nlnk[kb]; npb = T.npxy[kb];
        }
        *reinterpret_cast<float2 *>(&rec[A].x) = xb;
        rec[A].w = wb;
        *reinterpret_cast<float2 *>(&rec[B].x) = xa;
        rec[B].w = wa;
        if (dsw) {
            rec[A].z = zc;
            rec[Bm].z = za;
        }
        if (park_pos_b && t == 0) *park_pos_b = make_int2(kb, A);
        else T.pos[kb] = A;
        T.pos[ka] = B;
        if (A == 0) {  // rec[n] mirrors rec[0] (wrap-around successor of position n-1)
            *reinterpret_cast<float2 *>(&rec[n].x) = xb;
            rec[n].w = wb;
        }
        if (B == 0) {
            *reinterpret_cast<float2 *>(&rec[n].x) = xa;
            rec[n].w = wa;
        }
        if (t == 0) {
            // new edges: (a, b) at position pa and (a1, b1) at position pb; a and b1 are outside the range
            int pb1 = pb + 1;
            if (pb1 >= n) pb1 -= n;
            float4 ra, rb1;
            int na, nb1;
            if (NODE) {
                ra = rec[pa];
                rb1 = (pb1 == pa) ? ra : rec[pb1];
                na = node_of(ra);
                nb1 = node_of(rb1);
            } else {
                na = node_of(rec[pa]);
                nb1 = (pb1 == pa) ? na : node_of(rec[pb1]);
            }
            const float dab = (float)dist_nodes(I, na, kb);
            const float da1b1 = (float)dist_nodes(I, ka, nb1);
            if (delta_out) *delta_out = (long long)dab + (long long)da1b1 - (long long)rec[pa].z - (long long)rec[pb].z;  // nobody else writes these two
            rec[pa].z = dab;
            rec[pb].z = da1b1;
            if (NODE) {
                // ka = a1 (was at s), kb = b (was at e):  a -> b -> ... -> a1 -> b1
                T.nrec[ka] = make_float4(nra.x, nra.y, rb1.x, rb1.y);                       // a1: successor b1, predecessor = old successor
                T.nlnk[ka] = make_float4(da1b1, __int_as_float(nb1), nla.x, nla.y);
                T.npxy[ka] = make_float2(nra.z, nra.w);
                T.nrec[kb] = make_float4(nrb.x, nrb.y, npb.x, npb.y);                       // b: successor = old predecessor, predecessor a
                T.nlnk[kb] = make_float4(nlb.z, nlb.w, dab, __int_as_float(na));
                T.npxy[kb] = make_float2(ra.x, ra.y);
                *reinterpret_cast<float2 *>(&T.nrec[na].z) = xb;                            // a: successor b
                *reinterpret_cast<float2 *>(&T.nlnk[na].x) = make_float2(dab, __int_as_float(kb));
                *reinterpret_cast<float2 *>(&T.nlnk[nb1].z) = make_float2(da1b1, __int_as_float(ka));  // b1: predecessor a1
                T.npxy[nb1] = xa;
            }
        } else if (NODE) {
            T.nrec[ka] = make_float4(nra.x, nra.y, npa.x, npa.y);
            T.nlnk[ka] = make_float4(nla.z, nla.w, nla.x, nla.y);
            T.npxy[ka] = make_float2(nra.z, nra.w);
            T.nrec[kb] = make_float4(nrb.x, nrb.y, npb.x, npb.y);
            T.nlnk[kb] = make_float4(nlb.z, nlb.w, nlb.x, nlb.y);
            T.npxy[kb] = make_float2(nrb.z, nrb.w);
        }
    }
}

// Bookkeeping done by ONE thread of the selecting kernel once the move (i,j,delta) is known: publishes the
// positions for the apply launch, counts, logs.  delta >= 0 means "no move".
__device__ __forceinline__ void publish_move(const TourDev &T, int i, int j, long long delta) {
    Ctl *ctl = T.ctl;
    if (delta < 0) {
        ctl->ap_pa = T.pos[i];
        ctl->ap_pb = T.pos[j];
        ctl->ap_valid = 1;
        ctl->moves += 1;
        ctl->obj_delta += delta;
        const long long lc = ctl->log_count;
        if (T.log && lc < T.log_cap) {
            MoveRec mr;
            mr.i = i; mr.j = j; mr.delta = delta;
            T.log[lc] = mr;
        }
        ctl->log_count = lc + 1;
    } else {
        ctl->ap_valid = 0;
    }
}

// Exact delta of the move (i,j) in the CURRENT tour, from node ids (used to re-derive the delta of a
// selected move and as a device-side consistency check).
__device__ __forceinline__ long long move_delta_nodes(const InstDev &I, const TourDev &T, int i, int j) {
    const int n = T.n;
    int pa = T.pos[i], pb = T.pos[j];
    int pa1 = pa + 1; if (pa1 >= n) pa1 -= n;
    int pb1 = pb + 1; if (pb1 >= n) pb1 -= n;
    int a1 = node_of(T.rec[pa1]), b1 = node_of(T.rec[pb1]);
    return dist_nodes(I, i, j) + dist_nodes(I, a1, b1) - (long long)T.rec[pa].z - (long long)T.rec[pb].z;
}

// Seeding the filter of the NEXT best-improvement pass.  The runner-up moves of the pass that just ended are mostly
// still legal after the winner was applied; the exact delta of any legal move is a valid upper bound of the next
// pass's minimum, so `hint` may start there instead of at 0 and the FP32 filter is tight from the first tile on
// (without it every thread climbs through a series of "record" candidates, each a trip through the cold path).
// Called by the last block of the apply launch; all loads bypass L1 (other blocks just rewrote rec[] / pos[]).
// Exact delta of candidate move c in the CURRENT tour, or 0 when c is not a legal move any more (bad indices, the pair
// became adjacent — e.g. it IS the move just applied).  All loads bypass L1 (another block may just have rewritten
// rec[] / pos[]).
__device__ __forceinline__ long long legal_move_delta_cg(const InstDev &I, const TourDev &T, const MoveKey c) {
    const int n = T.n;
    if (c.delta >= 0 || c.i < 0 || c.j >= n || c.i >= c.j) return 0;
    const int pa = __ldcg(&T.pos[c.i]), pb = __ldcg(&T.pos[c.j]);
    int d = pa - pb;
    if (d < 0) d = -d;
    if (d <= 1 || d == n - 1) return 0;
    int pa1 = pa + 1; if (pa1 >= n) pa1 -= n;
    int pb1 = pb + 1; if (pb1 >= n) pb1 -= n;
    const float4 ra = __ldcg(&T.rec[pa]), rb = __ldcg(&T.rec[pb]);
    const int a1 = node_of(__ldcg(&T.rec[pa1])), b1 = node_of(__ldcg(&T.rec[pb1]));
    return dist_nodes(I, c.i, c.j) + dist_nodes(I, a1, b1) - (long long)ra.z - (long long)rb.z;
}

// Called by the last block of the apply launch with t = thread index.
__device__ __forceinline__ void seed_hint_from_candidates(const InstDev &I, const TourDev &T, int t) {
    Ctl *ctl = T.ctl;
    if (t >= ctl->ncand) return;
    const long long delta = legal_move_delta_cg(I, T, ctl->cand[t]);
    if (delta < 0) atomicMin(&ctl->hint, (int)delta);
}

// ---- first improvement: what follows a search (shared by the search kernel's last block and the apply launch) --------
// The first improving pair travels as (i << 32) | j: the same order as the reference's row-major enumeration.
__device__ __forceinline__ unsigned long long fi_key(int i, int j) { return ((unsigned long long)(unsigned)i << 32) | (unsigned)j; }
// number of pairs (i<j) in rows 0..r-1 of the row-major enumeration: sum_{q<r} (n-1-q)
__device__ __forceinline__ long long fi_pairs_before_row(long long r, long long n) { return r * (n - 1) - r * (r - 1) / 2; }

// Counters, cursor and sweep end once the first improving pair f at or after the cursor (i0, j0) is known (FI_NONE: none left
// in this sweep), reference src/heuristics.c:476-496.  One thread.  The move itself is published / applied by the caller.
__device__ __forceinline__ void fi_advance(const TourDev &T, unsigned long long f, int i0, int j0) {
    Ctl *ctl = T.ctl;
    const int n = T.n;
    int ci = 0, cj = 0;
    bool sweep_end = false;
    const long long A0 = fi_pairs_before_row(i0, n) + (j0 - i0 - 1);
    long long gap;
    if (f != FI_NONE) {
        const int i = (int)(f >> 32), j = (int)(f & 0xffffffffull);
        ctl->sweep_moves += 1;
        gap = fi_pairs_before_row(i, n) + (j - i - 1) - A0 + 1;
        ci = i;
        cj = j + 1;
        if (cj >= n) { ci = i + 1; cj = ci + 1; }
        if (ci >= n - 1) sweep_end = true;
    } else {
        sweep_end = true;
        ctl->ap_valid = 0;
        gap = (long long)n * (n - 1) / 2 - A0;
    }
    ctl->pairs_swept += gap;
    ctl->fi_shard = gap > ctl->fi_shard_min_gap;
    ctl->launches += 1;
    if (sweep_end) {
        ctl->passes += 1;
        if (ctl->sweep_moves == 0) {  // reference heuristics.c:492: the sweep brought no gain
            ctl->done = 1;
            ctl->done_reason = DONE_OPTIMUM;
        }
        ctl->sweep_moves = 0;
        ci = 0;
        cj = 1;
    }
    if (ctl->max_moves >= 0 && ctl->moves >= ctl->max_moves && !ctl->done) {  // a capped run may be continued later
        ctl->done = 1;
        ctl->done_reason = DONE_CAP;
    }
    ctl->cur_i = ci;
    ctl->cur_j = cj;
    ctl->fi_seg = 0;
}

// ---- kernel argument blocks shared by the kernel translation units and engine.cu ----------------------
// ---- multi-GPU argmin exchange over NVLink peer memory ------------------------------------------------------
// Every rank owns 2 x XCHG_MAX_WORLD 64-bit slots (double-buffered by the parity of the exchange epoch) plus XCHG_MAX_WORLD
// alignment counters.  In the tail of its scan kernel a rank STORES ONE 64-bit word — its packed (delta,i,j) key shifted
// left by two, with a 2-bit generation number derived from the epoch in the low bits — into slot [epoch&1][rank] of EVERY
// peer (plain st.global on pointers mapped with cudaIpcOpenMemHandle, i.e. NVLink writes through NVSwitch) and then polls
// its LOCAL slots until all `world` words carry the generation of this epoch.  Key and "arrived" flag travel in the same
// word, so no fence and no second store are needed.  No collective launch, no tour data on the wire: 8 bytes per peer
// and pass.  A rank can be at most one exchange ahead of a peer (it cannot finish exchange k+1 without that peer's word
// of exchange k+1), so two buffers suffice; successive words in one buffer are 2 epochs apart, i.e. their generations
// ((epoch >> 1) + 1) & 3 differ, and the zero-initialised slot never matches the first expected generation (1).
constexpr int XCHG_MAX_WORLD = 16;
struct XchgMem {
    unsigned long long slot[2][XCHG_MAX_WORLD];
    unsigned long long align[XCHG_MAX_WORLD];  // monotonically increasing barrier counters (rank_align_kernel)
};
struct XchgDev {
    XchgMem *peer[XCHG_MAX_WORLD];   // peer[r] = rank r's XchgMem (peer[rank] = own, local pointer)
    unsigned *epoch;                 // this rank's exchange epoch (device word, monotonically increasing, never reset)
    unsigned *align_epoch;           // this rank's alignment-barrier epoch
    int enabled;
};

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Block-wide: every rank contributes `key62` (< 2^62) and gets the minimum over all ranks.  Threads 0..world-1 each serve
// one peer; `s_x` is a shared array of XCHG_MAX_WORLD words.  Returns the minimum in thread 0 (other threads: undefined);
// *err is set to 2 when a peer did not deliver within ~10 s.  `wait_ns` (may be null) accumulates thread 0's polling time.
__device__ __forceinline__ unsigned long long xchg_min(const XchgDev &X, int rank, int world, unsigned long long key62,
                                                       unsigned long long *s_x, int *err, unsigned long long *wait_ns) {
    __shared__ unsigned s_epoch;
    const int tid = threadIdx.x;
    if (tid == 0) {
        const unsigned e = *X.epoch + 1u;
        *X.epoch = e;
        s_epoch = e;
    }
    __syncthreads();
    if (tid < world) {
        const unsigned e = s_epoch;
        const unsigned long long gen = (unsigned long long)(((e >> 1) + 1u) & 3u);
        const unsigned long long word = (key62 << 2) | gen;
        unsigned long long *dst = &X.peer[tid]->slot[e & 1u][rank];
        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(word) : "memory");
        const unsigned long long *src = &X.peer[rank]->slot[e & 1u][tid];
        const long long t0 = clock64();
        const unsigned long long g0 = (wait_ns && tid == 0) ? globaltimer_ns() : 0ull;
        unsigned long long got;
        for (;;) {
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(got) : "l"(src) : "memory");
            if ((got & 3ull) == gen) break;
            if (clock64() - t0 > 20000000000ll) {  // ~10 s: a peer died; fail loudly instead of hanging the GPU
                *err = 2;
                got = ~0ull;
                break;
            }
        }
        s_x[tid] = got >> 2;
        if (wait_ns && tid == 0) *wait_ns += globaltimer_ns() - g0;
    }
    __syncthreads();
    unsigned long long win = ~0ull;
    if (tid == 0) {
        win = s_x[0];
        for (int r = 1; r < world; ++r) win = s_x[r] < win ? s_x[r] : win;
    }
    return win;
}

struct BiArgs {
    InstDev inst;
    TourDev tour;
    const int *tile_row_start;  // [ntr+1] prefix sums of tiles per tile-row
    const int *tile_row_j0;     // [ntr] first tile column of each tile-row
    int ntr;
    int ntiles;
    int TJ;          // columns per tile (even)
    int rank, world; // tiles are dealt round-robin over ranks (multi-GPU neighbourhood sharding)
    int fuse_apply;  // 0: the last block only publishes this rank's key (multi-GPU); 1: it publishes the move for the
                     // apply launch; 2: it also applies the move itself
    int seed_hint;   // 0 = none, 1 = this block's previous winner re-evaluated at the start of the scan, 2 = also runner-ups
    int packed_tail; // 1: blocks fold their key into ctl->pass_min with one 64-bit atomicMin (n <= 2^17, seed_hint < 2)
    int pruned;      // 1: tiles come from the live list built by tile_filter_kernel (exact tile pruning)
    int row_shuffle; // 1: SHUF kernels (a warp owns 32 R - 1 rows, the distance below a lane's rows comes from the next lane)
    int prefilter;   // 1: stage-1 prefilter on squared distances in front of the FP32 filter (kernels_bi_scan.cuh)
    float pf_slack;  // prefilter: linear slack E of its row and column bounds (4 eps, DESIGN.md §3)
    float pf_cx, pf_cy;  // prefilter: translation of the coordinates, exact for every one of them (0 if none is)
    int timing;      // 1: accumulate the per-pass breakdown in ctl->tm_acc; 2: also dump per-block {start, end} stamps
    unsigned long long *dbg;        // timing == 2: [gridDim.x][2] globaltimer stamps of the last pass
    XchgDev xchg;    // fuse_apply == 0: how this rank's key reaches the other ranks (enabled = 0 -> NCCL allreduce of ctl->packed)
};

struct NnArgs {
    InstDev inst;
    int start;
    int *succ;                       // out
    unsigned char *visited;          // n bytes, zeroed by the launcher
    unsigned long long *slots;       // [3] packed (dist << 32 | idx) winners, rotating; init to ~0
    unsigned *barrier;               // grid barrier counter, zeroed by the launcher
    long long *cost;                 // out: accumulated cost
};

}  // namespace tspb
