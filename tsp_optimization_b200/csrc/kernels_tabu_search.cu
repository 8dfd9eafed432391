// kernels_tabu_search.cu — the resident tabu search (reference tabu(), src/tabusearch.c:188-320) on the resident tour, every
// iteration of a call without a host round trip (tspb200_tabu_search, DESIGN.md §4.9).  The host enqueues batches of
//     ts_expire_kernel -> masked scan (kernels_bi_tabu.cu, or bi_scan_exact_search_kernel) -> apply -> ts_step_kernel
// and reads the search's state once per batch.  A scan that finds no improving move sets ctl->done; the step that follows
// ends the iteration (cost, best tour, kick) and starts the next one.  After the last iteration every launch returns at once.
#include "tabu_common.cuh"

namespace tspb {

// reference src/utility.c:17-30 x_udir_pos (n <= 46 340: every index and intermediate fits an int, tm_index in kernels_batch.cu)
__device__ __forceinline__ int ts_index(int x, int y, int n) {
    if (x > y) { const int t = x; x = y; y = t; }
    return x * n + y - ((x + 1) * (x + 2)) / 2;
}
__device__ __forceinline__ int ts_succ(const TourDev &T, int z) { return node_of(T.rec[T.pos[z] + 1]); }  // rec[n] mirrors rec[0]
__device__ __forceinline__ int ts_pred(const TourDev &T, int z) {
    const int p = T.pos[z];
    return node_of(T.rec[p == 0 ? T.n - 1 : p - 1]);
}
// is entry (x, y) in U, the set of blocking entries of this alg_2opt_tabu call (non-zero, iter - v <= tenure)?  Whether
// another thread has meanwhile zeroed an expired entry does not matter: expired entries are not in U either way.
__device__ __forceinline__ bool ts_in_u(const int *list, int x, int y, int n, int iter, int tenure) {
    const int v = *((volatile const int *)&list[ts_index(x, y, n)]);
    return v != 0 && iter - v <= tenure;
}

// Does some pair of one masked pass test the expired entry {x, y}?  The pass (reference src/tabusearch.c:126-156) enumerates
// the non-adjacent pairs a < b (b != succ a, succ b != a) and tests (a,b), (a,a1), (b,b1), (a,b1) with '||': an entry is
// tested in some role when the entries before it in that pair are not in U.
//   T1  {x,y} not a tour edge: the pair (x,y) itself is non-adjacent and tests it first.
//   T2  e = (t, succ t) as (a,a1), a = t: some b > t, non-adjacent to t, with (t,b) not in U.
//   T3  e = (t, succ t) as (b,b1), b = t: some a < t, non-adjacent to t, with (a,t) and (a, succ a) not in U.
//   T4  e as (a,b1): a one end, b1 the other, b = pred b1, a < b, b != succ a, and (a,b), (a,a1), (b,b1) not in U.
// T2 and T3 stop at the first qualifying candidate: U is small, so one is found after a few steps.
__device__ bool ts_reached(const TourDev &T, const int *list, int n, int iter, int tenure, int x, int y) {
    const int sx = ts_succ(T, x), sy = ts_succ(T, y);
    if (sx != y && sy != x) return true;  // T1
    const int t = sx == y ? x : y, u = sx == y ? y : x;
    for (int b = t + 1; b < n; ++b) {     // T2
        if (b == u || ts_succ(T, b) == t) continue;
        if (!ts_in_u(list, t, b, n, iter, tenure)) return true;
    }
    for (int a = 0; a < t; ++a) {         // T3
        if (a == u) continue;
        const int a1 = ts_succ(T, a);
        if (a1 == t) continue;
        if (!ts_in_u(list, a, t, n, iter, tenure) && !ts_in_u(list, a, a1, n, iter, tenure)) return true;
    }
    for (int k = 0; k < 2; ++k) {         // T4
        const int a = k ? y : x, b1 = k ? x : y;
        const int b = ts_pred(T, b1), a1 = ts_succ(T, a);
        if (a < b && b != a1 && !ts_in_u(list, a, b, n, iter, tenure) && !ts_in_u(list, a, a1, n, iter, tenure) &&
            !ts_in_u(list, b, b1, n, iter, tenure))
            return true;
    }
    return false;
}

// zeroes entry (x, y) when it has expired and the coming pass reaches it; true when it stays non-zero
__device__ __forceinline__ bool ts_expire_entry(const TourDev &T, int *list, int n, int iter, int tenure, int x, int y) {
    const int e = ts_index(x, y, n);
    const int v = list[e];
    if (v == 0) return false;
    if (iter - v <= tenure || !ts_reached(T, list, n, iter, tenure, x, y)) return true;
    list[e] = 0;
    return false;
}

// Before every masked pass: the lazy expiry that pass would do, and the table drops the entries that read zero.  The table
// lists a superset of the non-zero entries (only kicks write non-zero values, tc_add lists them), so block 0 alone looks
// at its entries.  An overflowed table (tab_n = -1) is rebuilt: every block walks rows of the whole list, expires what it
// finds and lists the survivors; the last block sets tab_n (-1 again when more than TABU_TAB survive).
__global__ void __launch_bounds__(256) ts_expire_kernel(const TabuSearchArgs A, const TourDev T) {
    __shared__ int s_cnt, s_last;
    TabuSearchDev *S = A.S;
    if (*((volatile int *)&S->finished)) return;
    const int iter = S->cur_iter, tenure = S->cur_tenure;
    if (iter < 0 || tenure < 0) return;  // check_tenure neither blocks nor expires
    const int n = T.n, tid = threadIdx.x;
    int *list = A.list;
    if (S->s.tab_n >= 0) {
        if (blockIdx.x) return;
        const int tab_n = S->s.tab_n;
        const unsigned v = tid < tab_n ? S->s.tab[tid] : 0u;
        const bool keep = tid < tab_n && ts_expire_entry(T, list, n, iter, tenure, (int)(v >> 16), (int)(v & 0xffff));
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        if (keep) S->s.tab[atomicAdd(&s_cnt, 1)] = v;
        __syncthreads();
        if (tid == 0) S->s.tab_n = s_cnt;
        return;
    }
    const int warps = gridDim.x * (blockDim.x >> 5), lane = tid & 31;
    for (int x = blockIdx.x * (blockDim.x >> 5) + (tid >> 5); x < n - 1; x += warps) {
        const int *row = list + ts_index(x, x + 1, n) - (x + 1);  // row[y] = entry (x, y)
        for (int y = x + 1 + lane; y < n; y += 32)
            if (row[y] != 0 && ts_expire_entry(T, list, n, iter, tenure, x, y)) {
                const unsigned k = atomicAdd(&S->scan_cnt, 1u);
                if (k < (unsigned)TABU_TAB) S->s.tab[k] = (unsigned)x << 16 | (unsigned)y;
            }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&S->scan_ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last || tid) return;
    __threadfence();
    const unsigned cnt = *((volatile unsigned *)&S->scan_cnt);
    S->s.tab_n = cnt <= (unsigned)TABU_TAB ? (int)cnt : -1;
    S->scan_cnt = 0;
    S->scan_ticket = 0;
}

// Start of a call: `iters` iterations from the search's next iteration number.
__global__ void ts_init_kernel(const TabuSearchArgs A, Ctl *ctl, int iters, int max_draws) {
    TabuSearchDev *S = A.S;
    S->t = 0;
    S->iters = iters;
    S->max_draws = max_draws;
    S->err = 0;
    S->finished = iters == 0;
    S->cur_iter = S->s.next_iter;
    S->cur_tenure = iters ? A.tenures[0] : 0;
    ctl->done = iters == 0;
    ctl->done_reason = iters == 0 ? DONE_OPTIMUM : DONE_NONE;
    ctl->ap_valid = 0;
}

constexpr int TS_STEP_THREADS = 1024;

// After every pass (and its apply).  When the pass found no improving move, alg_2opt_tabu has returned: the cost is recomputed
// from the exact edge lengths (tabusearch.c:168-172), a strictly cheaper tour is copied to the best tour (:241-243), then
// the kick (:262-309): one thread draws pairs (a, b) = rand_choice(0, n) twice from the search's stream until one passes
// the tests of tabu_kick_select_kernel, at most max_draws pairs, stamps its two removed edges with iter and the block
// applies it.  The next iteration starts with the next tenure; after the last one the search is finished.
__global__ void __launch_bounds__(TS_STEP_THREADS) ts_step_kernel(const TabuSearchArgs A, const InstDev I, const TourDev T) {
    __shared__ long long s_red[TS_STEP_THREADS / 32];
    __shared__ int s_kick[3];  // positions of a and b, pairs drawn (0: max_draws reached)
    TabuSearchDev *S = A.S;
    Ctl *ctl = T.ctl;
    if (*((volatile int *)&S->finished) || !*((volatile int *)&ctl->done)) return;
    const int n = T.n, tid = threadIdx.x;
    const int t = S->t;                // (thread 0 rewrites both after the barriers below)
    const long long best0 = S->best;
    long long part = 0;
    for (int p = tid; p < n; p += TS_STEP_THREADS) part += (long long)T.rec[p].z;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) part += __shfl_xor_sync(0xffffffffu, part, m);
    if ((tid & 31) == 0) s_red[tid >> 5] = part;
    __syncthreads();
    long long cost = 0;
    for (int w = 0; w < TS_STEP_THREADS / 32; ++w) cost += s_red[w];
    const bool better = cost < best0;
    if (better)
        for (int p = tid; p < n; p += TS_STEP_THREADS) A.best_succ[node_of(T.rec[p])] = node_of(T.rec[p + 1]);
    if (tid == 0) {
        A.trace[t] = cost;
        if (better) S->best = cost;
        const int iter = S->cur_iter, tenure = S->cur_tenure;
        int *list = A.list;
        s_kick[2] = 0;
        for (int d = 1; d <= S->max_draws; ++d) {
            const int a = tc_rand_choice(S->s, n), b = tc_rand_choice(S->s, n);
            const int a1 = ts_succ(T, a), b1 = ts_succ(T, b);
            if (a == b || a1 == b || b1 == a) continue;
            const int e1 = ts_index(a, a1, n), e2 = ts_index(b, b1, n);
            if (!tc_check(list, e1, iter, tenure) && !tc_check(list, e2, iter, tenure) &&
                !tc_check(list, ts_index(a, b, n), iter, tenure) && !tc_check(list, ts_index(a1, b1, n), iter, tenure)) {
                list[e1] = iter;
                list[e2] = iter;
                tc_add(S->s, a, a1);
                tc_add(S->s, b, b1);
                s_kick[0] = T.pos[a];
                s_kick[1] = T.pos[b];
                s_kick[2] = d;
                break;
            }
        }
        A.draws[t] = s_kick[2];
        if (s_kick[2] == 0) {  // the reference would keep drawing; ctl->done stays set
            S->err = 2 + t;
            S->finished = 1;
        }
    }
    __syncthreads();
    if (s_kick[2] == 0) return;
    apply_swap_range<false>(I, T, s_kick[0], s_kick[1], tid, TS_STEP_THREADS);
    if (tid == 0) {
        const int next = S->cur_iter + 1;
        S->s.next_iter = next;
        S->t = t + 1;
        if (t + 1 >= S->iters) {
            S->finished = 1;
        } else {
            S->cur_iter = next;
            S->cur_tenure = A.tenures[t + 1];
            ctl->done = 0;
            ctl->done_reason = DONE_NONE;
        }
    }
}

cudaError_t launch_ts_init(const TabuSearchArgs &a, Ctl *ctl, int iters, int max_draws, cudaStream_t st) {
    ts_init_kernel<<<1, 1, 0, st>>>(a, ctl, iters, max_draws);
    return cudaGetLastError();
}

cudaError_t launch_ts_expire(const TabuSearchArgs &a, const TourDev &T, int num_sms, cudaStream_t st) {
    ts_expire_kernel<<<4 * num_sms, 256, 0, st>>>(a, T);
    return cudaGetLastError();
}

cudaError_t launch_ts_step(const TabuSearchArgs &a, const InstDev &I, const TourDev &T, cudaStream_t st) {
    ts_step_kernel<<<1, TS_STEP_THREADS, 0, st>>>(a, I, T);
    return cudaGetLastError();
}

}  // namespace tspb
