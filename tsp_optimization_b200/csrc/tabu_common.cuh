// tabu_common.cuh — what the two device-side tabu searches share (the chains of kernels_batch.cu, one thread block per
// chain, and the resident search of kernels_tabu_search.cu, grid-wide passes): the glibc random() stream the kick draws
// from, check_tenure as the kick tests it, and the table of list entries that may be non-zero.
#pragma once
#include "tsp_state.cuh"

namespace tspb {

// glibc srandom(seed) followed by the 310 discarded outputs (GlibcRandom in instances.py): the last 31 values of the TYPE_3
// recurrence, as tc_rand_choice continues it.  Host side.
inline void glibc_srandom_state(uint32_t seed, TabuChainState &s) {
    if (seed == 0) seed = 1;
    uint32_t x[344];
    x[0] = seed;
    for (int i = 1; i < 31; ++i) {  // 16807 x mod (2^31 - 1) on the signed value (Schrage), as glibc computes it
        const int32_t prev = (int32_t)x[i - 1];
        const int32_t hi = prev / 127773, lo = prev % 127773;
        int32_t word = 16807 * lo - 2836 * hi;
        if (word < 0) word += 2147483647;
        x[i] = (uint32_t)word;
    }
    for (int i = 31; i < 34; ++i) x[i] = x[i - 31];
    for (int i = 34; i < 344; ++i) x[i] = x[i - 31] + x[i - 3];
    for (int i = 344 - 31; i < 344; ++i) s.rng[i % 31] = x[i];
    s.rng_pos = 344 % 31;
}

// glibc random() on a chain's state (x_k = x_{k-31} + x_{k-3}, output x_k >> 1), then rand_choice(0, n) (reference
// src/utility.c:752-754: URAND() = random() / RAND_MAX in FP64, scaled by n and truncated), as GlibcRandom.rand_choice
__device__ __forceinline__ int tc_rand_choice(TabuChainState &st, int n) {
    const int k = st.rng_pos;
    const unsigned v = st.rng[k] + st.rng[k >= 3 ? k - 3 : k + 28];
    st.rng[k] = v;
    st.rng_pos = k == 30 ? 0 : k + 1;
    return (int)(__ddiv_rn((double)(v >> 1), 2147483647.0) * (double)n);
}

// check_tenure (src/tabusearch.c:83-92) on the dense list, as the kick tests it
__device__ __forceinline__ bool tc_check(int *list, int e, int iter, int tenure) {
    if (iter < 0 || tenure < 0) return false;
    const int v = list[e];
    if (v == 0) return false;
    if (iter - v > tenure) {
        list[e] = 0;
        return false;
    }
    return true;
}

// the kick stamped entry (x, y): one thread adds it to the table unless it is listed already (-1 when the table is full)
__device__ __forceinline__ void tc_add(TabuChainState &st, int x, int y) {
    if (st.tab_n < 0) return;
    const unsigned e = (unsigned)min(x, y) << 16 | (unsigned)max(x, y);
    for (int k = 0; k < st.tab_n; ++k)
        if (st.tab[k] == e) return;
    if (st.tab_n == TABU_TAB) st.tab_n = -1;
    else st.tab[st.tab_n++] = e;
}

}  // namespace tspb
