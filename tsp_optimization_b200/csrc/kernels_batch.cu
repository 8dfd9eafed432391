// kernels_batch.cu — batched 2-opt: one thread block drives one tour to its 2-opt local optimum with the
// whole tour state in shared memory (28 bytes per node), no host round trips.  This is the path for
// independent tour batches (GA offspring repair — reference src/genetic.c:426-443 calls alg_2opt on a
// mutated offspring; multi-start; VNS src/vns.c:143 and tabu restarts) and for small TSPLIB instances,
// where a grid-wide launch per move would be pure latency.
//
// Both modes replay the reference bit for bit:
//   FI  reference src/heuristics.c:438-502: row-major (i<j) sweep, every improving move applied at once,
//       the scan continues at (i, j+1); sweeps repeat until one brings no gain.
//   BI  reference src/tabusearch.c:107-178 (NULL tabu list): full scan, strict '<' argmin == lowest (i,j)
//       among equal deltas, apply, repeat until no negative delta.
// Evaluation is in node space (the enumeration order IS the node order); FP32 filter + FP64 exact check
// as in the grid-wide kernels.
#include "tsp_state.cuh"

namespace tspb {

constexpr int BATCH_THREADS = 256;

struct BatchSmem {
    float *sx, *sy, *dsn;  // node space: coordinates, d(k, succ k)
    float *dsp;            // position space: d(order[p], order[p+1]) — what a reversal permutes without recomputing
    int *succ, *order, *pos;
};

template <bool ATT>
__device__ __forceinline__ float bt_dist32(float ax, float ay, float bx, float by) {
    float dx = ax - bx, dy = ay - by;
    float s = fmaf(dy, dy, dx * dx);
    if (ATT) s *= 0.1f;
    return sqrt_approx(s);
}

__device__ __forceinline__ long long bt_exact(const InstDev &I, const BatchSmem &S, bool exact32, int u, int v) {
    if (I.dmat) return (long long)I.dmat[(long long)u * I.dmat_ld + v];
    if (exact32)
        return exact_dist(I.metric, make_double2((double)S.sx[u], (double)S.sy[u]), make_double2((double)S.sx[v], (double)S.sy[v]));
    return exact_dist(I.metric, I.pt64[u], I.pt64[v]);
}

// exact delta of pair (i,j) or "skip" (adjacent) -> returns false
template <bool ATT, bool EXACT32, bool FP32_OK>
__device__ __forceinline__ bool bt_eval(const InstDev &I, const BatchSmem &S, int i, int j, float xi, float yi, int si,
                                        float xsi, float ysi, float dsi, float thr, long long &delta) {
    const int sj = S.succ[j];
    if (sj == i || si == j || si == sj) return false;  // reference heuristics.c:471 / tabusearch.c:134
    const float dsj = S.dsn[j];
    if (FP32_OK) {
        float q = bt_dist32<ATT>(xi, yi, S.sx[j], S.sy[j]) + bt_dist32<ATT>(xsi, ysi, S.sx[sj], S.sy[sj]) - dsi - dsj;
        if (q > thr) return false;
    }
    delta = bt_exact(I, S, FP32_OK && EXACT32, i, j) + bt_exact(I, S, FP32_OK && EXACT32, si, sj) - (long long)dsi - (long long)dsj;
    return true;
}

// block-wide application of move (i,j) on the shared-memory tour (same orientation rule as apply_swap_range): the forward
// path a1..b is reversed in place.  Edge lengths inside the path are only PERMUTED (position-space dsp[] reversed among
// themselves); just the two new edges (a,b) and (a1,b1) are evaluated.
__device__ __forceinline__ void bt_apply(const InstDev &I, const BatchSmem &S, bool exact32, int n, int i, int j) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int pa = S.pos[i], pb = S.pos[j];
    const int a1 = S.succ[i], b1 = S.succ[j];
    __syncthreads();
    int s = pa + 1; if (s >= n) s -= n;
    int len = pb - pa; if (len < 0) len += n;
    const int e = pb;
    const int half = len >> 1, mhalf = (len - 1) >> 1;
    for (int t = tid; t < half; t += nt) {
        int A = s + t; if (A >= n) A -= n;
        int B = e - t; if (B < 0) B += n;
        const int ua = S.order[A], ub = S.order[B];
        S.order[A] = ub; S.order[B] = ua;
        S.pos[ub] = A; S.pos[ua] = B;
        if (t < mhalf) {
            int Bm = B - 1; if (Bm < 0) Bm += n;
            const float za = S.dsp[A], zc = S.dsp[Bm];
            S.dsp[A] = zc; S.dsp[Bm] = za;
        }
    }
    if (tid == 0) {
        S.dsp[pa] = (float)bt_exact(I, S, exact32, i, j);
        S.dsp[pb] = (float)bt_exact(I, S, exact32, a1, b1);
    }
    __syncthreads();
    // nodes at positions pa .. pb got a new successor
    for (int t = tid; t <= len; t += nt) {
        int P = pa + t; if (P >= n) P -= n;
        int Pn = P + 1; if (Pn >= n) Pn -= n;
        const int k = S.order[P];
        S.succ[k] = S.order[Pn];
        S.dsn[k] = S.dsp[P];
    }
    __syncthreads();
}

template <bool ATT, bool EXACT32, bool FP32_OK>
__global__ void __launch_bounds__(BATCH_THREADS) two_opt_batch_kernel(const InstDev I, int mode, int *succ_all, const int *slots,
                                                                      long long *obj_out, long long *counters, int batch,
                                                                      MoveRec *log, long long log_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_hits[BATCH_THREADS / 32];
    __shared__ int s_err;
    __shared__ MoveKey s_keys[BATCH_THREADS / 32];
    const int n = I.n;
    const int tid = threadIdx.x;
    BatchSmem S;
    S.sx = reinterpret_cast<float *>(smem_raw);
    S.sy = S.sx + n;
    S.dsn = S.sy + n;
    S.dsp = S.dsn + n;
    S.succ = reinterpret_cast<int *>(S.dsp + n);
    S.order = S.succ + n;
    S.pos = S.order + n;
    const bool ex32 = FP32_OK && EXACT32;
    const float W = I.W;

    for (int b = blockIdx.x; b < batch; b += gridDim.x) {
        int *gsucc = succ_all + (long long)(slots ? slots[b] : b) * n;  // slots: tours of a resident population
        for (int k = tid; k < n; k += BATCH_THREADS) {
            float2 p = I.pt32[k];
            S.sx[k] = p.x; S.sy[k] = p.y;
            S.succ[k] = gsucc[k];
        }
        if (tid == 0) s_err = 0;
        __syncthreads();
        if (tid == 0) {  // visiting order from node 0; also validates the cycle
            int at = 0;
            for (int p = 0; p < n; ++p) {
                if (at < 0 || at >= n || (p > 0 && at == 0)) { s_err = 1; break; }
                S.order[p] = at;
                S.pos[at] = p;
                at = S.succ[at];
            }
            if (at != 0) s_err = 1;
        }
        __syncthreads();
        long long moves = 0, passes = 0, evals = 0, objd = 0;
        if (!s_err && n >= 4) {
            for (int k = tid; k < n; k += BATCH_THREADS) {
                const float d = (float)bt_exact(I, S, ex32, k, S.succ[k]);
                S.dsn[k] = d;
                S.dsp[S.pos[k]] = d;
            }
            __syncthreads();
            if (mode == 1) {
                // ---------------- best improvement ----------------
                for (;;) {
                    MoveKey best = key_none();
                    float thr = W;
                    const int warp = tid >> 5, lane = tid & 31;
                    for (int i = warp; i < n - 1; i += BATCH_THREADS / 32) {
                        const float xi = S.sx[i], yi = S.sy[i], dsi = S.dsn[i];
                        const int si = S.succ[i];
                        const float xsi = S.sx[si], ysi = S.sy[si];
                        for (int j = i + 1 + lane; j < n; j += 32) {
                            long long delta;
                            if (!bt_eval<ATT, EXACT32, FP32_OK>(I, S, i, j, xi, yi, si, xsi, ysi, dsi, thr, delta)) continue;
                            if (delta < 0 && delta <= (long long)best.delta) {
                                MoveKey k;
                                k.delta = (int)delta; k.i = i; k.j = j; k.pad = 0;
                                if (key_less(k, best)) { best = k; thr = (float)k.delta + W; }
                            }
                        }
                    }
                    best = key_warp_min(best);
                    if (lane == 0) s_keys[warp] = best;
                    __syncthreads();
                    best = s_keys[0];
#pragma unroll
                    for (int w = 1; w < BATCH_THREADS / 32; ++w)
                        if (key_less(s_keys[w], best)) best = s_keys[w];
                    __syncthreads();
                    passes++;
                    if (best.delta >= 0) break;
                    if (log && tid == 0 && moves < log_cap) {
                        MoveRec mr;
                        mr.i = best.i; mr.j = best.j; mr.delta = best.delta;
                        log[moves] = mr;
                    }
                    bt_apply(I, S, ex32, n, best.i, best.j);
                    moves++;
                    objd += best.delta;
                }
                evals = passes * ((long long)n * (n - 3) / 2);
            } else {
                // ---------------- first improvement ----------------
                // The reference's sweep is a linear scan of the pairs in row-major order from a cursor.  The block scans a
                // WINDOW of that linear order per step: chunks of 32 consecutive pairs (crossing row ends) are dealt to the
                // 8 warps round-robin, K chunks per warp, each warp stopping at its first improving pair; the smallest
                // linear offset over the warps is the reference's "first improving pair at or after the cursor".  K
                // doubles while nothing is found (long quiet stretches cost few barriers) and resets after a move (tours
                // far from the optimum improve every few hundred pairs), so the work past the hit is bounded by the gap.
                constexpr int NW = BATCH_THREADS / 32;
                const int warp = tid >> 5, lane = tid & 31;
                int ci = 0, cj = 1;      // cursor (row, column)
                long long lin_prev = 1;  // statistics: linear index i*n+j of the cursor after the last move / sweep start
                long long sweep_moves = 0;
                int K = 1;
                const float thr = -1.0f + W;
                // (row, column) of the pair `k` places after the cursor; row >= n-1 means "past the end of the sweep"
                auto locate = [&](int k, int &row, int &j) {
                    row = ci;
                    long long jj = (long long)cj + k;
                    while (row < n - 1 && jj >= n) {
                        jj -= n;
                        row += 1;
                        jj += row + 1;
                    }
                    j = (int)jj;
                };
                for (;;) {
                    int myhit = 0x7fffffff;
                    // this lane's pair of the warp's first chunk; later chunks are 32*NW pairs further along the linear
                    // order, reached by walking (row, column) forward instead of locating from the cursor again
                    int row, j;
                    locate(32 * warp + lane, row, j);
                    for (int q = 0; q < K; ++q) {
                        bool hit = false;
                        const bool valid = row < n - 1;
                        if (valid) {
                            const int si = S.succ[row];
                            long long delta;
                            if (bt_eval<ATT, EXACT32, FP32_OK>(I, S, row, j, S.sx[row], S.sy[row], si, S.sx[si], S.sy[si], S.dsn[row], thr, delta))
                                hit = delta < 0;
                        }
                        const unsigned m = __ballot_sync(0xffffffffu, hit);
                        if (m) {
                            myhit = 32 * (warp + q * NW) + __ffs(m) - 1;
                            break;
                        }
                        if (!__any_sync(0xffffffffu, valid)) break;  // the whole chunk lies past the end of the sweep
                        long long jj = (long long)j + 32 * NW;
                        while (row < n - 1 && jj >= n) {
                            jj -= n;
                            row += 1;
                            jj += row + 1;
                        }
                        j = (int)jj;
                    }
                    if (lane == 0) s_hits[warp] = myhit;
                    __syncthreads();
                    int first = s_hits[0];
#pragma unroll
                    for (int w = 1; w < NW; ++w) first = min(first, s_hits[w]);
                    __syncthreads();  // s_hits[] is rewritten by the next step
                    bool sweep_end = false;
                    if (first != 0x7fffffff) {
                        int fi, fj;
                        locate(first, fi, fj);
                        const int si = S.succ[fi], sj = S.succ[fj];
                        const long long fdelta = bt_exact(I, S, ex32, fi, fj) + bt_exact(I, S, ex32, si, sj) - (long long)S.dsn[fi] -
                                                 (long long)S.dsn[fj];
                        evals += (long long)fi * n + fj - lin_prev + 1;  // linear pairs swept, like the grid kernel
                        if (log && tid == 0 && moves < log_cap) {
                            MoveRec mr;
                            mr.i = fi; mr.j = fj; mr.delta = fdelta;
                            log[moves] = mr;
                        }
                        bt_apply(I, S, ex32, n, fi, fj);
                        moves++; sweep_moves++;
                        objd += fdelta;
                        ci = fi; cj = fj + 1;
                        if (cj >= n) { ci = fi + 1; cj = ci + 1; }
                        lin_prev = (long long)ci * n + cj;
                        if (ci >= n - 1) sweep_end = true;
                        K = 1;
                    } else {
                        int nr, nj;
                        locate(32 * NW * K, nr, nj);
                        ci = nr; cj = nj;
                        if (ci >= n - 1) {
                            sweep_end = true;
                            evals += (long long)(n - 1) * n - lin_prev;
                        }
                        if (K < 16) K *= 2;
                    }
                    if (sweep_end) {
                        passes++;
                        if (sweep_moves == 0) break;  // reference heuristics.c:492
                        sweep_moves = 0;
                        ci = 0; cj = 1;
                        lin_prev = 1;
                        K = 1;
                    }
                }
            }
        } else if (!s_err) {
            passes = 1;
        }
        // write back
        long long cost_part = 0;
        for (int k = tid; k < n; k += BATCH_THREADS) {
            gsucc[k] = S.succ[k];
            if (!s_err && n >= 4) cost_part += (long long)S.dsn[k];
        }
        if (mode == 1) {
            // reference tabusearch.c:168-172: cost recomputed from scratch
            if (!s_err && n < 4)
                for (int k = tid; k < n; k += BATCH_THREADS) cost_part += bt_exact(I, S, ex32, k, S.succ[k]);
            for (int m = 16; m > 0; m >>= 1) cost_part += __shfl_xor_sync(0xffffffffu, cost_part, m);
            __shared__ long long s_cost[BATCH_THREADS / 32];
            if ((tid & 31) == 0) s_cost[tid >> 5] = cost_part;
            __syncthreads();
            if (tid == 0) {
                long long c = 0;
                for (int w = 0; w < BATCH_THREADS / 32; ++w) c += s_cost[w];
                obj_out[b] = c;
            }
        } else if (tid == 0) {
            obj_out[b] = objd;
        }
        if (tid == 0) {
            counters[4 * b + 0] = moves;
            counters[4 * b + 1] = passes;
            counters[4 * b + 2] = evals;
            counters[4 * b + 3] = s_err;
        }
        __syncthreads();
    }
}

template <bool ATT, bool EXACT32, bool FP32_OK>
static cudaError_t launch_batch_t(const InstDev &I, int mode, int *succ, const int *slots, long long *obj, long long *counters,
                                  int batch, int num_sms, cudaStream_t st, int *launched, MoveRec *log, long long log_cap) {
    size_t smem = (size_t)I.n * 28 + 16;
    auto kern = two_opt_batch_kernel<ATT, EXACT32, FP32_OK>;
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, BATCH_THREADS, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorInvalidValue;
    int grid = num_sms * occ;
    if (grid > batch) grid = batch;
    kern<<<grid, BATCH_THREADS, smem, st>>>(I, mode, succ, slots, obj, counters, batch, batch == 1 ? log : nullptr, log_cap);
    if (launched) *launched = 1;
    return cudaGetLastError();
}

cudaError_t launch_two_opt_batch(const InstDev &I, int mode, int *succ, const int *slots, long long *obj, long long *counters,
                                 int batch, int num_sms, cudaStream_t st, int *launched, MoveRec *log, long long log_cap) {
    const bool att = (I.metric == M_ATT);
    const bool ex = I.exact32 != 0;
    if (!I.fp32_ok) return launch_batch_t<false, false, false>(I, mode, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);
    if (att && ex) return launch_batch_t<true, true, true>(I, mode, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);
    if (att) return launch_batch_t<true, false, true>(I, mode, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);
    if (ex) return launch_batch_t<false, true, true>(I, mode, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);
    return launch_batch_t<false, false, true>(I, mode, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);
}

}  // namespace tspb

// ---- best improvement in POSITION space (the grid kernel's evaluator, one thread block per tour) ----------------------------
// The node-space evaluator above needs two fresh distances per pair; in position space every distance D[p][q] serves the two
// moves (p,q) and (p-1,q-1), a lane owns R consecutive rows and marches along the columns; the distance of the row below them
// is the next lane's: one square root per move (a warp covers 32 R - 1 rows),
// packed FP32x2 arithmetic, one filter test per warp and 4 columns, hits resolved by the whole warp in FP64 — exactly
// bi_scan_kernel, with the tour records {x, y, ds, node} in shared memory instead of L2.  A warp covers 32 R - 1 rows; the
// (row tile, column) space of the upper triangle is cut into equal contiguous shares, one per warp, so a warp loads its
// rows at most twice per pass.  Result = reference src/tabusearch.c:107-178 bit for bit (same (delta, i, j) argmin, same
// forward-path reversal), for GA offspring repair / multi-start / VNS and tabu restarts on EUC_2D / CEIL_2D / ATT instances.
namespace tspb {

constexpr int BPOS_THREADS = 128;
constexpr int BPOS_CB = 4;

template <int R, bool ATT, bool EXACT32>
__device__ __noinline__ MoveKey bpos_cold_warp(const InstDev I, const float4 *rec, int n, int p0, int q0, float thr
                                               TSPB_PROBE_ARG(int own_rows)) {
    const int lane = threadIdx.x & 31;
    MoveKey best = key_none();
#pragma unroll 1
    for (int base = 0; base < R * BPOS_CB; base += 32) {
        const int idx = base + lane;
        const int r = idx / BPOS_CB, c = idx % BPOS_CB;
        const int p = p0 + r, q = q0 + c;
        if (idx < R * BPOS_CB && q >= p + 2 && q <= n - 1 && !(p == 0 && q == n - 1)) {  // reference tabusearch.c:134
            const float4 rp = rec[p], rp1 = rec[p + 1], c0 = rec[q], c1 = rec[q + 1];
            const float qv = (bt_dist32<ATT>(rp.x, rp.y, c0.x, c0.y) - rp.z) + bt_dist32<ATT>(rp1.x, rp1.y, c1.x, c1.y);
            if (qv <= thr + c0.z TSPB_PROBE_OR(I.probe_on)) {
                const int u = node_of(rp), v = node_of(c0);
                long long d1, d2;
                if (EXACT32) {
                    d1 = exact_dist(I.metric, make_double2((double)rp.x, (double)rp.y), make_double2((double)c0.x, (double)c0.y));
                    d2 = exact_dist(I.metric, make_double2((double)rp1.x, (double)rp1.y), make_double2((double)c1.x, (double)c1.y));
                } else {
                    d1 = exact_dist(I.metric, I.pt64[u], I.pt64[v]);
                    d2 = exact_dist(I.metric, I.pt64[node_of(rp1)], I.pt64[node_of(c1)]);
                }
                const long long delta = d1 + d2 - (long long)rp.z - (long long)c0.z;
#if TSPB_FILTER_PROBE
                if (I.probe_on) {  // as bi_cold_warp
                    if (r < own_rows && delta <= I.probe_H) probe_record(I, u, v, delta, qv, thr, qv <= thr + c0.z);
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

// distances from the lane's R rows to one column point (rows in packed pairs); D[R], the distance from the row below them —
// the next lane's first row: a warp owns 32 R - 1 consecutive rows — comes from that lane by one shuffle when NEXT is set
// (R square roots per column instead of R + 1; lane 31's last row, whose lower neighbour lives in another warp's share,
// is masked out by the caller and scanned as the first row of the next row tile)
template <int R, bool ATT, bool NEXT>
__device__ __forceinline__ void bpos_column(const f32x2 (&xr2)[R / 2], const f32x2 (&yr2)[R / 2], float cx, float cy, float (&D)[R + 1]) {
    const f32x2 cxx = f2pack(cx, cx), cyy = f2pack(cy, cy);
#pragma unroll
    for (int k = 0; k < R / 2; ++k) {
        f32x2 dx = f2sub(xr2[k], cxx), dy = f2sub(yr2[k], cyy);
        f32x2 s = f2fma(dy, dy, f2mul(dx, dx));
        if (ATT) s = f2mul(s, f2pack(0.1f, 0.1f));
        D[2 * k] = sqrt_approx(f2lo(s));
        D[2 * k + 1] = sqrt_approx(f2hi(s));
    }
    D[R] = NEXT ? __shfl_down_sync(0xffffffffu, D[0], 1) : 0.f;
}

// One warp scans rows [p0w, p0w + 32 R - 1) x columns [qb, qe) (qb, qe multiples of 4) of the shared-memory tour.
template <int R, bool ATT, bool EXACT32, bool DIAG>
__device__ __forceinline__ void bpos_scan(const InstDev &I, const float4 *rec, int n, int p0w, int qb, int qe, float W,
                                          volatile int *s_hint, MoveKey &best, unsigned long long &colds) {
    const int lane = threadIdx.x & 31;
    const int p0 = p0w + lane * R;
    f32x2 xr2[R / 2], yr2[R / 2], cp2[R / 2];
    const f32x2 zero2 = f2pack(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < R / 2; ++k) {
        const float4 v0 = rec[p0 + 2 * k], v1 = rec[p0 + 2 * k + 1];
        xr2[k] = f2add(f2pack(v0.x, v1.x), zero2);
        yr2[k] = f2add(f2pack(v0.y, v1.y), zero2);
        cp2[k] = f2sub(zero2, f2pack(v0.z, v1.z));  // padding rows: ds = -BIG -> +BIG -> never a candidate
    }
    if (lane == 31) cp2[R / 2 - 1] = f2pack(f2lo(cp2[R / 2 - 1]), TSPB_BIG);  // its lower neighbour is not in this warp: next row tile's first row
    float thr = (float)(*s_hint) + W;
    float4 c0 = rec[qb];
    float4 cnext = rec[qb + 1];
    f32x2 U2[R / 2];
    {
        float D0[R + 1];
        bpos_column<R, ATT, false>(xr2, yr2, c0.x, c0.y, D0);
#pragma unroll
        for (int k = 0; k < R / 2; ++k) U2[k] = f2add(f2pack(D0[2 * k], D0[2 * k + 1]), cp2[k]);
    }
    const int qrel0 = qb - p0;
    for (int q4 = qb; q4 < qe; q4 += BPOS_CB) {
        float M = TSPB_BIG;
#pragma unroll
        for (int c = 0; c < BPOS_CB; ++c) {
            const float4 c1 = cnext;
            cnext = rec[q4 + c + 2];
            float Dn[R + 1];
            bpos_column<R, ATT, true>(xr2, yr2, c1.x, c1.y, Dn);
            float m = TSPB_BIG;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float qv = ((r & 1) ? f2hi(U2[r >> 1]) : f2lo(U2[r >> 1])) + Dn[r + 1];
                if (DIAG) qv = (qrel0 + (q4 - qb) + c >= r + 2) ? qv : TSPB_BIG;
                m = fminf(m, qv);
            }
            M = fminf(M, m - c0.z);
#pragma unroll
            for (int k = 0; k < R / 2; ++k) U2[k] = f2add(f2pack(Dn[2 * k], Dn[2 * k + 1]), cp2[k]);
            c0 = c1;
        }
        unsigned hits = __ballot_sync(0xffffffffu, M <= thr);
        while (hits) {
            const int L = __ffs(hits) - 1;
            const float thrL = __shfl_sync(0xffffffffu, thr, L);
            const MoveKey nb = bpos_cold_warp<R, ATT, EXACT32>(I, rec, n, p0w + L * R, q4, thrL TSPB_PROBE_ARG(L == 31 ? R - 1 : R));
            if (lane == L) {
                colds += 1;
                if (key_less(nb, best)) {
                    best = nb;
                    atomicMin((int *)s_hint, nb.delta);
                }
            }
            if (nb.delta < 0) thr = fminf(thr, (float)nb.delta + W);
            hits &= hits - 1;
            hits &= __ballot_sync(0xffffffffu, M <= thr);
        }
        if (((q4 - qb) & 63) == 64 - BPOS_CB) thr = fminf(thr, (float)(*s_hint) + W);
    }
}

template <int R, bool ATT, bool EXACT32>
__global__ void __launch_bounds__(BPOS_THREADS) two_opt_batch_bi_kernel(const InstDev I, int *succ_all, const int *slots,
                                                                        long long *obj_out, long long *counters, int batch,
                                                                        int alloc, MoveRec *log, long long log_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_hint;
    __shared__ int s_err;
    __shared__ MoveKey s_keys[BPOS_THREADS / 32];
    __shared__ MoveKey s_win;
    __shared__ long long s_cost[BPOS_THREADS / 32];
    constexpr int NW = BPOS_THREADS / 32;
    constexpr int NR = 32 * R - 1;  // rows (moves) per warp tile: the 32nd lane's last row overlaps the next tile's first
    const int n = I.n;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float4 *rec = reinterpret_cast<float4 *>(smem_raw);
    int *pos = reinterpret_cast<int *>(rec + alloc);
    const float W = I.W;
    TourDev T{};  // shared-memory view for apply_swap_range (generic pointers)
    T.n = n;
    T.rec = rec;
    T.pos = pos;

    // the upper triangle as a linear space of column steps: row tile t contributes the columns cb(t) .. n4-1,
    // cb(t) = (t * NR + 2) rounded down to 4 (everything before is masked for all of the tile's rows)
    const int ntr = n >= 4 ? (n - 2 + NR - 1) / NR : 0;
    const int n4 = (n + 3) & ~3;
    long long total_steps = 0;
    for (int t = 0; t < ntr; ++t) total_steps += n4 - ((t * NR + 2) & ~3);
    const long long per = ((total_steps + NW - 1) / NW + 3) & ~3ll;

    for (int b = blockIdx.x; b < batch; b += gridDim.x) {
        int *gsucc = succ_all + (long long)(slots ? slots[b] : b) * n;
        for (int k = tid; k < n; k += BPOS_THREADS) pos[k] = gsucc[k];  // successors, until the order is known
        if (tid == 0) s_err = 0;
        __syncthreads();
        if (tid == 0) {  // visiting order from node 0; also validates the cycle
            int at = 0;
            for (int p = 0; p < n; ++p) {
                if (at < 0 || at >= n || (p > 0 && at == 0)) { s_err = 1; break; }
                rec[p].w = __int_as_float(at);
                at = pos[at];
            }
            if (at != 0) s_err = 1;
        }
        __syncthreads();
        long long moves = 0, passes = 0;
        unsigned long long colds = 0;
        if (!s_err) {
            for (int p = tid; p < alloc; p += BPOS_THREADS) {
                if (p < n) {
                    const int u = node_of(rec[p]);
                    const float2 c = I.pt32[u];
                    rec[p].x = c.x;
                    rec[p].y = c.y;
                } else if (p == n) {
                    const float2 c = I.pt32[0];
                    rec[p] = make_float4(c.x, c.y, -TSPB_BIG, __int_as_float(0));
                } else {
                    rec[p] = make_float4(0.f, 0.f, -TSPB_BIG, __int_as_float(0));
                }
            }
            __syncthreads();
            for (int p = tid; p < n; p += BPOS_THREADS) {
                const int u = node_of(rec[p]), v = node_of(rec[p + 1 == n ? 0 : p + 1]);
                pos[u] = p;
                rec[p].z = (float)dist_nodes(I, u, v);
            }
#if TSPB_FILTER_PROBE
            if (tid == 0) s_hint = I.probe_on ? I.probe_H : 0;  // pinned: bpos_cold_warp returns no key, the pass ends with none
#else
            if (tid == 0) s_hint = 0;
#endif
            __syncthreads();
        }
        if (!s_err && n >= 4) {
            for (;;) {
                MoveKey best = key_none();
                // this warp's share of the column steps: [lo, hi) of the linear space, at most two row tiles
                long long lo = per * warp, hi = lo + per < total_steps ? lo + per : total_steps;
                long long base = 0;
                for (int t = 0; t < ntr && lo < hi; ++t) {
                    const int cb = (t * NR + 2) & ~3;
                    const long long len = n4 - cb;
                    if (lo < base + len) {
                        const int qb = cb + (int)(lo - base);
                        const long long take = (base + len < hi ? base + len : hi) - lo;
                        const int qe = qb + (int)take;
                        if (qb < t * NR + NR + 1) bpos_scan<R, ATT, EXACT32, true>(I, rec, n, t * NR, qb, qe, W, &s_hint, best, colds);
                        else bpos_scan<R, ATT, EXACT32, false>(I, rec, n, t * NR, qb, qe, W, &s_hint, best, colds);
                        lo += take;
                    }
                    base += len;
                }
                best = key_warp_min(best);
                if (lane == 0) s_keys[warp] = best;
                __syncthreads();
                if (tid == 0) {
                    MoveKey k = s_keys[0];
#pragma unroll
                    for (int w = 1; w < NW; ++w)
                        if (key_less(s_keys[w], k)) k = s_keys[w];
                    s_win = k;
                    s_hint = 0;
                }
                __syncthreads();
                const MoveKey win = s_win;
                passes++;
                if (win.delta >= 0) break;  // reference src/tabusearch.c:158
                if (log && tid == 0 && moves < log_cap) {
                    MoveRec mr;
                    mr.i = win.i; mr.j = win.j; mr.delta = win.delta;
                    log[moves] = mr;
                }
                const int wpa = pos[win.i], wpb = pos[win.j];
                __syncthreads();  // everybody has read the two positions before the swap rewrites pos[]
                apply_swap_range<false>(I, T, wpa, wpb, tid, BPOS_THREADS);
                moves++;
                __syncthreads();
                // the runner-up of every warp is most likely still a legal move: its exact delta now seeds the next pass's filter
                if (tid < NW) {
                    const MoveKey c = s_keys[tid];
                    if (c.delta < 0 && !(c.i == win.i && c.j == win.j)) {
                        const int pa = pos[c.i], pb = pos[c.j];
                        int d = pa - pb;
                        if (d < 0) d = -d;
                        if (d > 1 && d != n - 1) {
                            const int pa1 = pa + 1 == n ? 0 : pa + 1, pb1 = pb + 1 == n ? 0 : pb + 1;
                            const long long dl = dist_nodes(I, c.i, c.j) + dist_nodes(I, node_of(rec[pa1]), node_of(rec[pb1])) -
                                                 (long long)rec[pa].z - (long long)rec[pb].z;
                            if (dl < 0) atomicMin(&s_hint, (int)dl);
                        }
                    }
                }
                __syncthreads();
            }
        } else if (!s_err) {
            passes = 1;
        }
        // write back: succ[node(p)] = node(p+1); cost = sum of the exact edge lengths (reference tabusearch.c:168-172)
        long long cost_part = 0;
        if (!s_err) {
            for (int p = tid; p < n; p += BPOS_THREADS) {
                gsucc[node_of(rec[p])] = node_of(rec[p + 1 == n ? 0 : p + 1]);
                cost_part += (long long)rec[p].z;
            }
        }
        for (int m = 16; m > 0; m >>= 1) cost_part += __shfl_xor_sync(0xffffffffu, cost_part, m);
        if (lane == 0) s_cost[warp] = cost_part;
        __syncthreads();
        if (tid == 0) {
            long long c = 0;
            for (int w = 0; w < NW; ++w) c += s_cost[w];
            obj_out[b] = c;
            counters[4 * b + 0] = moves;
            counters[4 * b + 1] = passes;
            counters[4 * b + 2] = passes * ((long long)n * (n - 3) / 2);
            counters[4 * b + 3] = s_err;
        }
        __syncthreads();
    }
}

template <int R, bool ATT, bool EXACT32>
static cudaError_t launch_bpos_t(const InstDev &I, int *succ, const int *slots, long long *obj, long long *counters, int batch,
                                 int num_sms, cudaStream_t st, int *launched, MoveRec *log, long long log_cap) {
    constexpr int NR = 32 * R - 1;
    const int n = I.n;
    const int ntr = n >= 4 ? (n - 2 + NR - 1) / NR : 0;
    int alloc = ntr * NR + R + 1;
    if (alloc < n + 8) alloc = n + 8;
    alloc = (alloc + 3) & ~3;
    const size_t smem = (size_t)alloc * sizeof(float4) + (size_t)n * sizeof(int);
    auto kern = two_opt_batch_bi_kernel<R, ATT, EXACT32>;
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, BPOS_THREADS, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorInvalidValue;
    int grid = num_sms * occ;
    if (grid > batch) grid = batch;
    kern<<<grid, BPOS_THREADS, smem, st>>>(I, succ, slots, obj, counters, batch, alloc, batch == 1 ? log : nullptr, log_cap);
    if (launched) *launched = 1;
    return cudaGetLastError();
}

// best improvement, FP32-filter path only (EUC_2D / CEIL_2D / ATT inside the FP32 window); everything else uses the
// node-space kernel above
cudaError_t launch_two_opt_batch_bi_pos(const InstDev &I, int *succ, const int *slots, long long *obj, long long *counters, int batch,
                                        int num_sms, cudaStream_t st, int *launched, MoveRec *log, long long log_cap) {
    if (!I.fp32_ok || I.dmat) return cudaErrorNotSupported;
    const bool att = (I.metric == M_ATT);
    const bool ex = I.exact32 != 0;
#define BPOS_GO(R_)                                                                                                         \
    do {                                                                                                                    \
        if (att && ex) return launch_bpos_t<R_, true, true>(I, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);   \
        if (att) return launch_bpos_t<R_, true, false>(I, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);        \
        if (ex) return launch_bpos_t<R_, false, true>(I, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);         \
        return launch_bpos_t<R_, false, false>(I, succ, slots, obj, counters, batch, num_sms, st, launched, log, log_cap);                \
    } while (0)
    if (I.n <= 128) BPOS_GO(2);
    BPOS_GO(8);
#undef BPOS_GO
}

}  // namespace tspb
