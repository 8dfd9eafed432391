// kernels_bi_tabu.cu — the masked best-improvement pass of the resident tabu search (tspb200_tabu_search, DESIGN.md §4.9):
// the exhaustive FP32-filter scan of kernels_bi_scan.cuh with the tabu test in its cold path (bi_cold_warp_tabu).  One shape,
// 64 threads x 8 rows with the row shuffle and the square-root filter alone, the one the shape model picks for an
// exhaustive single-GPU pass at the tour sizes the list allows (n <= 46 340); the engine makes its own tile plan for it.
// A kernel of its own, so that the unmasked instantiations keep their names and code.
#include "kernels_bi_scan.cuh"

namespace tspb {

constexpr int TS_THREADS = 64, TS_ROWS = 8;

template <bool ATT, bool EXACT32>
__global__ void __launch_bounds__(TS_THREADS, TSPB_BI_MINBLOCKS64) bi_scan_tabu_kernel(const BiArgs A, const int *list,
                                                                                       const TabuSearchDev *S) {
    bi_scan_body<TS_THREADS, TS_ROWS, ATT, EXACT32, false, true, false, true>(A, list, S);
}

int ts_scan_threads() { return TS_THREADS; }
int ts_scan_rows() { return TS_ROWS; }

cudaError_t launch_bi_scan_tabu_fp32(const BiArgs &a, const int *list, const TabuSearchDev *S, int grid, cudaStream_t st) {
    const size_t smem = (size_t)2 * (a.TJ + 2) * sizeof(float4) + (size_t)(2 * a.ntr + 2) * sizeof(int);  // as launch_bi_tr
    auto go = [&](auto kern) -> cudaError_t {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<grid, TS_THREADS, smem, st>>>(a, list, S);
        return cudaGetLastError();
    };
    const bool att = a.inst.metric == M_ATT, ex = a.inst.exact32 != 0;
    if (att && ex) return go(bi_scan_tabu_kernel<true, true>);
    if (att) return go(bi_scan_tabu_kernel<true, false>);
    if (ex) return go(bi_scan_tabu_kernel<false, true>);
    return go(bi_scan_tabu_kernel<false, false>);
}

}  // namespace tspb
