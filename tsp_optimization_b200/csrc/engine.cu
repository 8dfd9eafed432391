// engine.cu — host side of libtspb200.so: context, HBM-resident instance / tour state, launch loops and
// the C ABI declared in include/tspb200.h.  No CPU fallback anywhere: every compute entry point needs a
// CUDA device and fails with TSPB200_E_CUDA otherwise.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/tspb200.h"
#include "tsp_state.cuh"

namespace tspb {

// ---- launchers implemented in the kernel translation units ---------------------------------------------
cudaError_t launch_bi_scan(const BiArgs &a, int threads, int rows_per_thread, int grid, bool pdl, cudaStream_t st);
bool bi_shape_supported(int threads, int rows_per_thread);
int bi_tile_rows(int threads, int rows_per_thread, int row_shuffle);
bool bi_shuffle_supported(int threads, int rows_per_thread);
cudaError_t launch_bi_scan_exact(const InstDev &inst, const TourDev &tour, int rank, int world, int fuse_apply, int grid,
                                 cudaStream_t st);
cudaError_t launch_bi_scan_tabu(const InstDev &inst, const TourDev &tour, int *skip, int iter, int tenure, long long *zl,
                                unsigned long long *zl_count, long long zl_cap, int grid, cudaStream_t st);
cudaError_t launch_bi_decode_packed(const TourDev &tour, cudaStream_t st);
cudaError_t launch_apply_move(const InstDev &inst, const TourDev &tour, int num_sms, int seed, int timing, bool pdl, bool node_space,
                              int fi_late, cudaStream_t st);
cudaError_t launch_tile_prune(const BiArgs &a, int TI, int grid_bi, bool pdl, cudaStream_t st);
cudaError_t launch_rank_align(const XchgDev &x, int rank, int world, Ctl *ctl, cudaStream_t st);
cudaError_t launch_rebuild_node_space(const TourDev &T, cudaStream_t st);
cudaError_t launch_fi_flush(const TourDev &T, cudaStream_t st);
cudaError_t launch_fi_search(const InstDev &I, const TourDev &T, int rank, int world, const XchgDev *xchg, int late, int grid, bool pdl,
                             cudaStream_t st);
cudaError_t launch_fi_finish(const InstDev &I, const TourDev &T, cudaStream_t st);
cudaError_t launch_dist_matrix(const InstDev &I, int *out, long long ld, int row_begin, int row_end, bool fast,
                               unsigned long long *geo_near, cudaStream_t st);
cudaError_t launch_build_state(const InstDev &I, const TourDev &T, const int *order, cudaStream_t st);
cudaError_t launch_succ_to_order(const int *succ, int n, void *work, int *order, int *err, cudaStream_t st);
cudaError_t launch_export_state(const TourDev &T, int *succ, unsigned long long *cost, cudaStream_t st);
cudaError_t launch_tour_cost(const InstDev &I, const int *tours, const int *slots, int as_order, long long *out, int batch,
                             cudaStream_t st);
cudaError_t launch_nn_tour(const NnArgs &a, int grid, cudaStream_t st);
struct NnGridArgs {  // kernels_nn.cu
    InstDev inst;
    int start;
    int GX, GY;
    double xmin, ymin, h, inv_h;
    double scale;
    int *cell_cnt;
    int *cell_fill;
    double2 *spt;
    int *snode;
    int *start_spos;
    int *succ;
    long long *cost;
};
size_t nn_grid_smem_bytes(int n, int ncell);
cudaError_t launch_nn_grid(const NnGridArgs &a, int num_sms, cudaStream_t st);
cudaError_t launch_prep_points(const double2 *raw, double2 *pt64, float2 *pt32, int n, int metric, cudaStream_t st);
int nn_max_grid(int num_sms);
cudaError_t launch_extra_mileage(const InstDev &I, int *succ_out, long long *cost_out, unsigned char *gwork, bool force_global,
                                 cudaStream_t st);
size_t extra_mileage_state_bytes(int n);
cudaError_t launch_nn_batch(const InstDev &I, const int *starts, int batch, int *succ_out, long long *cost_out, float eps,
                            int num_sms, cudaStream_t st);
cudaError_t launch_two_opt_batch(const InstDev &I, int mode, int *succ, const int *slots, long long *obj_delta, long long *counters,
                                 int batch, int num_sms, cudaStream_t st, int *launched, MoveRec *log, long long log_cap);
cudaError_t launch_two_opt_batch_bi_pos(const InstDev &I, int *succ, const int *slots, long long *obj, long long *counters, int batch,
                                        int num_sms, cudaStream_t st, int *launched, MoveRec *log, long long log_cap);
cudaError_t launch_vns_kick(const InstDev &I, const TourDev &T, int idx1, int idx2, int idx3, float4 *scratch, cudaStream_t st);
cudaError_t launch_tabu_kick_select(const TourDev &T, int *skip, const int *pairs, int count, int iter, int tenure, int *accepted,
                                    cudaStream_t st);
cudaError_t launch_population_store(const int *staged, int *pop, const int *slots, int n, int count, int as_order, cudaStream_t st);
cudaError_t launch_population_fetch(const int *pop, const int *slots, int *out, int n, int count, int as_order, cudaStream_t st);

// ---- NCCL, loaded at run time (the torch-bundled or system libnccl.so.2) -------------------------------
typedef struct { char internal[128]; } nccl_unique_id;
typedef void *nccl_comm_t;
struct NcclApi {
    void *handle = nullptr;
    int (*GetUniqueId)(nccl_unique_id *) = nullptr;
    int (*CommInitRank)(nccl_comm_t *, int, nccl_unique_id, int) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load(std::string &err) {
        if (handle) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *nm : names) {
            handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (handle) break;
        }
        if (!handle) { err = std::string("cannot dlopen libnccl.so.2: ") + dlerror(); return false; }
        GetUniqueId = (int (*)(nccl_unique_id *))dlsym(handle, "ncclGetUniqueId");
        CommInitRank = (int (*)(nccl_comm_t *, int, nccl_unique_id, int))dlsym(handle, "ncclCommInitRank");
        CommDestroy = (int (*)(nccl_comm_t))dlsym(handle, "ncclCommDestroy");
        AllReduce = (int (*)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t))dlsym(handle, "ncclAllReduce");
        AllGather = (int (*)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t))dlsym(handle, "ncclAllGather");
        GetErrorString = (const char *(*)(int))dlsym(handle, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllReduce) { err = "libnccl.so.2 lacks required symbols"; return false; }
        return true;
    }
};
static NcclApi g_nccl;
constexpr int NCCL_CHAR = 0;    // ncclInt8
constexpr int NCCL_INT32 = 2;   // ncclInt32
constexpr int NCCL_UINT64 = 5;  // ncclUint64
constexpr int NCCL_MAX = 2;     // ncclMax
constexpr int NCCL_MIN = 3;     // ncclMin

}  // namespace tspb

using namespace tspb;

struct tspb200_ctx {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;

    // instance
    int n = 0, metric = 0;
    InstDev inst{};
    double2 *d_raw = nullptr, *d_pt64 = nullptr;
    float2 *d_pt32 = nullptr;
    int *d_mat = nullptr;
    long long mat_ld = 0;
    double dmax = 0;
    double bb_xmin = 0, bb_xmax = 0, bb_ymin = 0, bb_ymax = 0;  // bounding box of the coordinates (bucket grid of the NN walk)
    bool coords_finite = true;
    int opt_nn_grid = -1;             // nearest neighbour on the bucket grid: -1 auto (planar metrics, n >= 256), 0 off, 1 on
    std::vector<double> h_xy;         // host copy of the coordinates of the resident instance (set_instance short cut)
    float eps32 = 0;                  // bound of |FP32 distance - real distance| for this instance
    float pf_cx = 0, pf_cy = 0;       // translation of the FP32 coordinates for the stage-1 prefilter (BiArgs::pf_cx)
    unsigned long long geo_near = 0;  // GEO matrix entries within 1e-6 of a rounding boundary (last matrix build)

    // tour (device buffers are kept across set_instance / tour_upload calls while they are big enough: cudaMalloc is
    // a synchronising call, and a slow one once peer access is enabled)
    bool has_tour = false;
    int inst_cap = 0;                 // nodes the instance arrays can hold
    int tour_cap_n = 0;               // nodes the per-node tour arrays can hold
    int tour_cap_rec = 0;             // records allocated in tour.rec
    long long tour_cap_log = 0;       // move-log entries allocated
    int tile_cap = 0;                 // ints allocated in each tile table
    int box_cap = 0;                  // entries allocated in each of the pruning box arrays
    long long live_cap = 0;           // entries allocated in the live-tile list
    bool node_dirty = false;          // the tour changed (upload, best-improvement moves, kicks, restore) since the node-space tables were built
    bool fi_cursor_stale = false;     // ... and the first-improvement sweep state refers to a tour that no longer exists
    double dist_bound = 0;            // upper bound of any distance of the instance (edge lengths live in FP32 words)
    // grow-only scratch buffers of the one-shot entry points (batched 2-opt, NN, tour costs, extra mileage)
    void *scratch_ptr[24] = {};
    size_t scratch_cap[24] = {};
    TourDev tour{};
    int *d_order = nullptr, *d_succ = nullptr;
    unsigned long long *d_cost = nullptr;
    Ctl *d_ctl = nullptr, *h_ctl = nullptr;
    long long log_cap = 0;
    double obj_in = 0;

    // BI tiling
    int T = 256, R = 8, TJ = 256, grid_bi = 296, ntr = 0, ntiles = 0;
    long long shape_key[6] = {-1, -1, -1, -1, -1, -1};
    int shape_T = 64, shape_R = 8, shape_TJ = 256;
    int *d_tile_row_start = nullptr, *d_tile_row_j0 = nullptr;

    // options
    int opt_T = 0, opt_R = 0, opt_TJ = 0, opt_grid = 0, opt_force_path = -1, opt_batch = 0, opt_fuse_apply = -1;
    long long opt_time_limit_ms = 0;
    int opt_seed_hint = 1;
    int opt_pdl = 1;
    int opt_prefilter = -1;           // exhaustive best-improvement scan: stage-1 prefilter on squared distances (-1 auto, 0 off, 1 on)
    int opt_single_block = -1;
    int opt_prune = -1;         // exact tile pruning of the best-improvement scan: -1 auto, 0 off (exhaustive scan), 1 on
    int opt_timing = 0;         // accumulate the per-pass breakdown (scan / tail / exchange wait / apply) on the device
    int opt_em_global = 0;      // tests: extra mileage keeps its state in the global work buffer even when it fits shared memory
    int opt_batch_kernel = 0;   // batched best improvement: 0 = position-space kernel when applicable, 1 = always the node-space kernel
    unsigned long long *d_dbg = nullptr;  // per-block time stamps of the last pass ("timing" = 2)
#if TSPB_FILTER_PROBE
    int probe_H = 0;                      // option "probe": 0 = off, H <= -1 = pin the threshold of the coming passes at H + W
    ProbeRec *d_probe = nullptr;          // records of the last probed pass (option "probe_cap" entries)
    unsigned long long *d_probe_count = nullptr;
    long long probe_cap = 0;
#endif
    int opt_debug_shard = 0;    // timing experiments only: (world << 8 | rank) -> scan that rank's share of the tiles on one GPU  // -1 auto, 0 never, 1 whenever the tour fits in shared memory
    // benchmark hygiene: write this many bytes (> L2) before every pass and time each pass with its own event pair
    long long opt_flush_bytes = 0;
    unsigned char *d_flush = nullptr;
    long long flush_cap = 0;
    std::vector<cudaEvent_t> pass_events;

    // tabu list of the running alg_2opt_tabu call (device copy + indices zeroed by lazy expiry)
    bool tabu_on = false;
    int tabu_iter = 0, tabu_tenure = 0;
    int *d_skip = nullptr;
    long long skip_cap = 0;
    long long *d_zl = nullptr;
    unsigned long long *d_zl_count = nullptr;
    long long zl_cap = 0;

    // resident sessions (VNS / tabu / GA): saved tours, the tabu list kept in HBM, a population of successor arrays
    bool tour_changed = false;        // the resident tour was perturbed since the last 2-opt run: `done` no longer holds
    float4 *save_rec[2] = {};
    int *save_pos[2] = {};
    int save_n[2] = {}, save_alloc[2] = {};
    bool tabu_session = false;
    int *d_pop = nullptr;
    long long pop_cap = 0;            // tours the population buffer can hold
    int pop_count = 0, pop_n = 0;

    // comm
    nccl_comm_t comm = nullptr;
    int rank = 0, world = 1;
    // argmin exchange over NVLink peer memory (see XchgDev): own slots + IPC-mapped peer slots
    XchgDev xchg{};
    XchgMem *d_slots = nullptr;
    unsigned *d_epoch = nullptr;      // [0] exchange epoch, [1] alignment epoch
    int *d_stop = nullptr;            // collective time-limit decision
    void *peer_mapped[XCHG_MAX_WORLD] = {};
    std::string xchg_note;
    int opt_exchange = 0;  // 0 = peer memory when available, 1 = NCCL allreduce
    int opt_upload_rank = -1;         // successor array -> visiting order at tour upload: -1 auto (device for n >= 2048), 0 host walk, 1 device
    int opt_row_shuffle = -1;         // best-improvement scan: distance below a lane's rows by shuffle (-1 auto = on where built, 0 off, 1 on)
    int row_shuffle = 0;              // what the current tile plan was made for
    int opt_fi_late = 1;              // first improvement on one GPU: the apply launch selects the winner itself (no search-kernel tail)
    unsigned long long fi_parity = 0; // launches of the late-selection search so far in this run (its hit word alternates)
    long long opt_fi_shard_min_gap = 4000000;  // first improvement on several GPUs: searches longer than this many pairs are followed by a sharded one
};

static int fail(tspb200_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    return code;
}

// grow-only device scratch, one buffer per slot; nullptr on allocation failure (cudaGetLastError holds the reason)
static void *dev_scratch(tspb200_ctx *c, int slot, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (c->scratch_cap[slot] < bytes) {
        cudaFree(c->scratch_ptr[slot]);
        c->scratch_ptr[slot] = nullptr;
        c->scratch_cap[slot] = 0;
        if (cudaMalloc(&c->scratch_ptr[slot], bytes) != cudaSuccess) return nullptr;
        c->scratch_cap[slot] = bytes;
    }
    return c->scratch_ptr[slot];
}
#define SCRATCH(var, type, slot, bytes)                                                                   \
    type var = static_cast<type>(dev_scratch(ctx, slot, bytes));                                          \
    if (!var) return fail(ctx, TSPB200_E_CUDA, "cudaMalloc of %zu bytes failed: %s", (size_t)(bytes), cudaGetErrorString(cudaGetLastError()))

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return fail(ctx, TSPB200_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

static void free_tour(tspb200_ctx *c) {
    cudaFree(c->tour.rec); cudaFree(c->tour.pos); cudaFree(c->tour.nrec); cudaFree(c->tour.nlnk);
    cudaFree(c->tour.npxy); cudaFree(c->tour.block_best); cudaFree(c->tour.log);
    cudaFree(c->tour.rowbox); cudaFree(c->tour.colbox); cudaFree(c->tour.rowmaxds); cudaFree(c->tour.colmaxds);
    cudaFree(c->tour.colbox2); cudaFree(c->tour.colmaxds2);
    cudaFree(c->tour.live);
    cudaFree(c->d_order); cudaFree(c->d_succ); cudaFree(c->d_cost);
    cudaFree(c->d_tile_row_start); cudaFree(c->d_tile_row_j0);
    c->tour = TourDev{};
    c->d_order = c->d_succ = nullptr; c->d_cost = nullptr;
    c->d_tile_row_start = c->d_tile_row_j0 = nullptr;
    c->has_tour = false;
    c->tour_cap_n = c->tour_cap_rec = c->tile_cap = 0;
    c->tour_cap_log = 0;
    c->box_cap = 0;
    c->live_cap = 0;
}

static void free_xchg(tspb200_ctx *c) {
    for (int r = 0; r < XCHG_MAX_WORLD; ++r) {
        if (c->peer_mapped[r]) cudaIpcCloseMemHandle(c->peer_mapped[r]);
        c->peer_mapped[r] = nullptr;
    }
    cudaFree(c->d_slots);
    cudaFree(c->d_epoch);
    cudaFree(c->d_stop);
    c->d_slots = nullptr;
    c->d_epoch = nullptr;
    c->d_stop = nullptr;
    c->xchg = XchgDev{};
}

static void free_instance(tspb200_ctx *c) {
    free_tour(c);
    cudaFree(c->d_flush);
    c->d_flush = nullptr;
    c->flush_cap = 0;
    for (cudaEvent_t e : c->pass_events) cudaEventDestroy(e);
    c->pass_events.clear();
    cudaFree(c->d_skip); cudaFree(c->d_zl); cudaFree(c->d_zl_count);
    c->d_skip = nullptr; c->d_zl = nullptr; c->d_zl_count = nullptr;
    c->skip_cap = c->zl_cap = 0;
    c->tabu_on = false;
    c->tabu_session = false;
    for (int k = 0; k < 2; ++k) {
        cudaFree(c->save_rec[k]); cudaFree(c->save_pos[k]);
        c->save_rec[k] = nullptr; c->save_pos[k] = nullptr;
        c->save_n[k] = c->save_alloc[k] = 0;
    }
    cudaFree(c->d_pop);
    c->d_pop = nullptr;
    c->pop_cap = 0;
    c->pop_count = c->pop_n = 0;
    cudaFree(c->d_raw); cudaFree(c->d_pt64); cudaFree(c->d_pt32); cudaFree(c->d_mat);
    c->d_raw = c->d_pt64 = nullptr; c->d_pt32 = nullptr; c->d_mat = nullptr;
    c->n = 0;
    c->inst_cap = 0;
    c->h_xy.clear();
}

extern "C" {

int tspb200_create(int device, tspb200_ctx **out) {
    if (!out) return TSPB200_E_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    tspb200_ctx *ctx = new tspb200_ctx();
    *out = ctx;  // returned even on failure so that the caller can read the message
    if (e != cudaSuccess || count == 0)
        return fail(ctx, TSPB200_E_CUDA, "no CUDA device: %s (libtspb200 has no CPU fallback)",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= count) return fail(ctx, TSPB200_E_ARG, "device %d out of range (%d devices)", device, count);
    ctx->device = device;
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(ctx, TSPB200_E_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
    ctx->num_sms = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&ctx->ev0));
    CK(cudaEventCreate(&ctx->ev1));
    CK(cudaMalloc(&ctx->d_ctl, sizeof(Ctl)));
    CK(cudaMallocHost(&ctx->h_ctl, sizeof(Ctl)));
    return TSPB200_OK;
}

void tspb200_destroy(tspb200_ctx *ctx) {
    if (!ctx) return;
    if (ctx->stream) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        free_xchg(ctx);
        if (ctx->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->comm);
        free_instance(ctx);
        for (int k = 0; k < 16; ++k) cudaFree(ctx->scratch_ptr[k]);
        cudaFree(ctx->d_dbg);
#if TSPB_FILTER_PROBE
        cudaFree(ctx->d_probe);
        cudaFree(ctx->d_probe_count);
#endif
        cudaFree(ctx->d_ctl);
        cudaFreeHost(ctx->h_ctl);
        cudaEventDestroy(ctx->ev0);
        cudaEventDestroy(ctx->ev1);
        cudaStreamDestroy(ctx->stream);
    }
    delete ctx;
}

const char *tspb200_last_error(const tspb200_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tspb200_set_option(tspb200_ctx *ctx, const char *key, int64_t value) {
    if (!ctx || !key) return TSPB200_E_ARG;
    std::string k(key);
    if (k == "rows_per_thread") {
        if (value != 0 && value != 2 && value != 4 && value != 8 && value != 16) return fail(ctx, TSPB200_E_ARG, "rows_per_thread must be 0 (auto), 2, 4, 8 or 16");
        ctx->opt_R = (int)value;
    } else if (k == "block_threads") {
        if (value != 0 && value != 64 && value != 128 && value != 256) return fail(ctx, TSPB200_E_ARG, "block_threads must be 0 (auto), 64, 128 or 256");
        ctx->opt_T = (int)value;
    } else if (k == "fuse_apply") {
        if (value < -1 || value > 1) return fail(ctx, TSPB200_E_ARG, "fuse_apply must be -1 (auto), 0 or 1");
        ctx->opt_fuse_apply = (int)value;
    } else if (k == "exchange") {
        if (value != 0 && value != 1) return fail(ctx, TSPB200_E_ARG, "exchange must be 0 (peer memory when available) or 1 (NCCL)");
        ctx->opt_exchange = (int)value;
    } else if (k == "l2_flush_bytes") {
        if (value < 0) return fail(ctx, TSPB200_E_ARG, "l2_flush_bytes must be >= 0");
        ctx->opt_flush_bytes = value;
    } else if (k == "debug_shard") {
        ctx->opt_debug_shard = (int)value;
        ctx->has_tour = false;
    } else if (k == "single_block") {
        if (value < -1 || value > 1) return fail(ctx, TSPB200_E_ARG, "single_block must be -1 (auto), 0 or 1");
        ctx->opt_single_block = (int)value;
    } else if (k == "prune") {
        if (value < -1 || value > 1) return fail(ctx, TSPB200_E_ARG, "prune must be -1 (auto), 0 or 1");
        ctx->opt_prune = (int)value;
    } else if (k == "timing") {
        if (value < 0 || value > 2) return fail(ctx, TSPB200_E_ARG, "timing must be 0, 1 or 2");
        ctx->opt_timing = (int)value;
    } else if (k == "upload_rank") {
        if (value < -1 || value > 1) return fail(ctx, TSPB200_E_ARG, "upload_rank must be -1 (auto), 0 or 1");
        ctx->opt_upload_rank = (int)value;
    } else if (k == "row_shuffle") {
        if (value < -1 || value > 1) return fail(ctx, TSPB200_E_ARG, "row_shuffle must be -1 (auto), 0 or 1");
        ctx->opt_row_shuffle = (int)value;
        ctx->has_tour = false;  // the tile plan depends on it
    } else if (k == "fi_late") {
        ctx->opt_fi_late = value ? 1 : 0;
    } else if (k == "fi_shard_min_gap") {
        if (value < 0) return fail(ctx, TSPB200_E_ARG, "fi_shard_min_gap must be >= 0 (0 = every search is sharded)");
        ctx->opt_fi_shard_min_gap = value;
    } else if (k == "nn_grid") {
        if (value < -1 || value > 1) return fail(ctx, TSPB200_E_ARG, "nn_grid must be -1 (auto), 0 or 1");
        ctx->opt_nn_grid = (int)value;
    } else if (k == "em_global") {
        ctx->opt_em_global = value ? 1 : 0;
    } else if (k == "batch_kernel") {
        ctx->opt_batch_kernel = value ? 1 : 0;
    } else if (k == "pdl") {
        ctx->opt_pdl = value ? 1 : 0;
    } else if (k == "prefilter") {
        if (value < -1 || value > 1) return fail(ctx, TSPB200_E_ARG, "prefilter must be -1 (auto), 0 or 1");
        ctx->opt_prefilter = (int)value;
    } else if (k == "seed_hint") {
        ctx->opt_seed_hint = value < 0 ? 0 : (value > 2 ? 2 : (int)value);
    } else if (k == "tile_cols") {
        if (value != 0 && (value < 32 || value > 1024 || (value & 3))) return fail(ctx, TSPB200_E_ARG, "tile_cols must be 0 (auto) or a multiple of 4 in [32,1024]");
        ctx->opt_TJ = (int)value;
    } else if (k == "grid") {
        ctx->opt_grid = (int)value;
    } else if (k == "force_path") {
        if (value < -1 || value > 2) return fail(ctx, TSPB200_E_ARG, "force_path must be -1..2");
        ctx->opt_force_path = (int)value;
    } else if (k == "batch") {
        ctx->opt_batch = (int)value;
    } else if (k == "time_limit_ms") {
        ctx->opt_time_limit_ms = value;
#if TSPB_FILTER_PROBE
    } else if (k == "probe") {
        if (value > -1 && value != 0) return fail(ctx, TSPB200_E_ARG, "probe must be 0 (off) or a threshold H <= -1");
        if (value < INT32_MIN) return fail(ctx, TSPB200_E_ARG, "probe threshold out of range");
        if (value && !ctx->d_probe) return fail(ctx, TSPB200_E_STATE, "set probe_cap first");
        ctx->probe_H = (int)value;
    } else if (k == "probe_cap") {
        if (value < 1) return fail(ctx, TSPB200_E_ARG, "probe_cap must be >= 1");
        CK(cudaSetDevice(ctx->device));
        CK(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_probe);
        ctx->d_probe = nullptr;
        ctx->probe_cap = 0;
        CK(cudaMalloc(&ctx->d_probe, sizeof(ProbeRec) * (size_t)value));
        if (!ctx->d_probe_count) CK(cudaMalloc(&ctx->d_probe_count, sizeof(unsigned long long)));
        CK(cudaMemset(ctx->d_probe_count, 0, sizeof(unsigned long long)));
        ctx->probe_cap = value;
#endif
    } else {
        return fail(ctx, TSPB200_E_ARG, "unknown option %s", key);
    }
    return TSPB200_OK;
}

int64_t tspb200_get_info(const tspb200_ctx *ctx, const char *key) {
    if (!ctx || !key) return -1;
    std::string k(key);
    if (k == "num_sms") return ctx->num_sms;
    if (k == "n") return ctx->n;
    if (k == "rows_per_thread") return ctx->R;
    if (k == "block_threads") return ctx->T;
    if (k == "tile_cols") return ctx->TJ;
    if (k == "row_shuffle") return ctx->row_shuffle;
    if (k == "tile_rows") return bi_tile_rows(ctx->T, ctx->R, ctx->row_shuffle);
    if (k == "grid_bi") return ctx->grid_bi;
    if (k == "ntiles") return ctx->ntiles;
    if (k == "exact32") return ctx->inst.exact32;
    if (k == "fp32_ok") return ctx->inst.fp32_ok;
    if (k == "int_coords") return ctx->inst.int_coords;
    if (k == "window_x1000") return (int64_t)(ctx->inst.W * 1000.0f);
    if (k == "matrix_resident") return ctx->d_mat != nullptr;
    if (k == "matrix_ld") return ctx->mat_ld;
    if (k == "cold_calls") return ctx->h_ctl ? (int64_t)ctx->h_ctl->cold_calls : -1;  // as of the last host sync
    if (k == "pf_hits") return ctx->h_ctl ? (int64_t)ctx->h_ctl->pf_hits : -1;
    if (k == "prefilter") return ctx->opt_prefilter;
    if (k == "tiles_scanned") return ctx->h_ctl ? (int64_t)ctx->h_ctl->tiles_scanned : -1;
    // per-pass breakdown accumulated since the tour was uploaded (option "timing"), ns; tm_count = passes accumulated
    if (k.rfind("tm_", 0) == 0 && ctx->h_ctl) {
        const char *names[] = {"tm_gap", "tm_scan", "tm_spread", "tm_tail", "tm_xwait", "tm_apply_gap", "tm_apply", "tm_count"};
        for (int t = 0; t < 8; ++t)
            if (k == names[t]) return (int64_t)ctx->h_ctl->tm_acc[t];
    }
    if (k == "dist_bound") return (int64_t)ctx->dist_bound;
    if (k == "geo_near_boundary") return (int64_t)ctx->geo_near;
    if (k == "exchange_p2p") return ctx->xchg.enabled && ctx->opt_exchange == 0;
    if (k == "world") return ctx->world;
    if (k == "rank") return ctx->rank;
#if TSPB_FILTER_PROBE
    if (k == "window_bits") {  // W exactly, as the kernels read it
        uint32_t b;
        memcpy(&b, &ctx->inst.W, sizeof b);
        return (int64_t)b;
    }
    if (k == "probe_count") {  // records appended by the last probed pass (more than probe_cap: the buffer overflowed)
        unsigned long long c = 0;
        if (!ctx->d_probe_count || cudaMemcpy(&c, ctx->d_probe_count, sizeof c, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return (int64_t)c;
    }
#endif
    return -1;
}

// ---- instance --------------------------------------------------------------------------------------------

int tspb200_set_instance(tspb200_ctx *ctx, const double *xy, int n, int weight_type) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!xy || n < 1) return fail(ctx, TSPB200_E_ARG, "bad instance (n=%d)", n);
    CK(cudaSetDevice(ctx->device));
    // the very same instance again (callers such as the reference's drivers re-enter with unchanged coordinates): nothing to do,
    // the device tables, a resident matrix and the sessions stay valid
    if (n == ctx->n && weight_type == ctx->metric && ctx->h_xy.size() == (size_t)2 * n &&
        memcmp(ctx->h_xy.data(), xy, sizeof(double) * 2 * (size_t)n) == 0)
        return TSPB200_OK;
    if (n > ctx->inst_cap) {
        free_instance(ctx);
    } else {  // same buffers, new contents: whatever was derived from the old instance is void
        CK(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_mat);
        ctx->d_mat = nullptr;
        ctx->mat_ld = 0;
        ctx->has_tour = false;
        ctx->tabu_session = false;  // sessions belong to the instance they were opened on
        ctx->pop_count = 0;
        ctx->save_n[0] = ctx->save_n[1] = 0;
    }
    ctx->n = n;
    ctx->metric = weight_type;
    // host-side scan: FP32 representability, bounding box -> filter window
    bool exact32 = true, finite = true, int_coords = true;
    double xmin = xy[0], xmax = xy[0], ymin = xy[1], ymax = xy[1], dc = 0;
    for (int k = 0; k < n; ++k) {
        double x = xy[2 * k], y = xy[2 * k + 1];
        if (!std::isfinite(x) || !std::isfinite(y)) finite = false;
        float fx = (float)x, fy = (float)y;
        if ((double)fx != x || (double)fy != y) exact32 = false;
        if (int_coords && (std::fabs(x) >= 9.0e15 || std::fabs(y) >= 9.0e15 || x != (double)(long long)x || y != (double)(long long)y))
            int_coords = false;
        dc = std::fmax(dc, std::fmax(std::fabs((double)fx - x), std::fabs((double)fy - y)));
        xmin = std::fmin(xmin, x); xmax = std::fmax(xmax, x);
        ymin = std::fmin(ymin, y); ymax = std::fmax(ymax, y);
    }
    double dmax = std::hypot(xmax - xmin, ymax - ymin);
    ctx->dmax = dmax;
    ctx->bb_xmin = xmin; ctx->bb_xmax = xmax; ctx->bb_ymin = ymin; ctx->bb_ymax = ymax;
    ctx->coords_finite = finite;
    // upper bound of any distance: the 2-opt state keeps edge lengths as exact integers in FP32 words (< 2^24)
    if (!finite) ctx->dist_bound = INFINITY;
    else if (weight_type == TSPB200_GEO) ctx->dist_bound = 20040.0;                        // pi * 6378.388 + 2
    else if (weight_type == TSPB200_ATT) ctx->dist_bound = dmax / std::sqrt(10.0) + 2.0;
    else if (weight_type == TSPB200_MAN_2D || weight_type == TSPB200_MAX_2D) ctx->dist_bound = (xmax - xmin) + 2.0;  // dy == 0
    else ctx->dist_bound = dmax + 2.0;
    const bool metric_fp32 = (weight_type != TSPB200_GEO && weight_type != TSPB200_MAN_2D && weight_type != TSPB200_MAX_2D);
    // FP32 filter usable when distances stay well inside the FP32 integer range (exact ds as float)
    const bool fp32_ok = finite && metric_fp32 && dmax < 4.0e6;
    // |D_fp32 - r_true| <= eps: MUFU.SQRT + the FP32 dx/dy/s roundings are < 2^-21 relative, coordinate rounding
    // contributes <= 2*sqrt(2)*dc; see DESIGN.md §3 for the derivation of W = 1 + 4*eps (EUC_2D) and 0.125 + 4*eps
    // (CEIL_2D, ATT) below.
    double eps = dmax * std::ldexp(1.0, -20) + 4.0 * dc;
    ctx->inst = InstDev{};
    ctx->inst.n = n;
    ctx->inst.metric = weight_type;
    ctx->inst.exact32 = exact32 ? 1 : 0;
    ctx->inst.fp32_ok = fp32_ok ? 1 : 0;
    ctx->inst.int_coords = (int_coords && exact32 && finite) ? 1 : 0;
    // Filter window W: a pair whose exact delta is <= the best one must pass "Q_fp32 <= best + W".  The two fresh integer
    // distances of a move differ from the real ones by at most 1/2 each for EUC_2D (nint), and are never BELOW the real ones
    // for CEIL_2D and ATT (both round up): delta_exact >= Q_real - 1 resp. Q_real.  The FP32 evaluation of Q adds at most
    // 2 eps (two distances) + three roundings of sums <= 2 dmax (0.4 eps); 4 eps is allowed for.  Every pair inside the
    // window costs a trip through the exact path, so the window is kept as narrow as the arithmetic permits
    // (round 1 used 2 + 2 eps for every metric: ~2x the exact-path calls on EUC_2D).
    const bool rounds_up = weight_type == TSPB200_CEIL_2D || weight_type == TSPB200_ATT;
    ctx->eps32 = (float)eps;
    // The stage-1 prefilter's rounding margins scale with the squared norms of the coordinates it reads (DESIGN.md §3), so
    // it reads them translated to the bounding box's center, rounded to an integer.  The translation must not round any
    // FP32 coordinate (FP32 differences, hence every filter decision, stay what they are): otherwise none is used.
    ctx->pf_cx = ctx->pf_cy = 0;
    if (finite) {
        const double cx = std::nearbyint(0.5 * (xmin + xmax)), cy = std::nearbyint(0.5 * (ymin + ymax));
        bool exact = std::fabs(cx) < 16777216.0 && std::fabs(cy) < 16777216.0;  // the center itself is an FP32 value
        for (int k = 0; k < n && exact; ++k) {
            const double x = (double)(float)xy[2 * k] - cx, y = (double)(float)xy[2 * k + 1] - cy;
            exact = (double)(float)x == x && (double)(float)y == y;
        }
        if (exact) {
            ctx->pf_cx = (float)cx;
            ctx->pf_cy = (float)cy;
        }
    }
    ctx->inst.W = metric_fp32 ? (float)((rounds_up ? 0.125 : 1.0) + 4.0 * eps) : (float)(2.0 + 2.0 * eps);
    ctx->inst.band = (float)std::ldexp(1.0, -20);
    if (n > ctx->inst_cap) {
        CK(cudaMalloc(&ctx->d_raw, sizeof(double2) * (size_t)n));
        CK(cudaMalloc(&ctx->d_pt64, sizeof(double2) * (size_t)n));
        CK(cudaMalloc(&ctx->d_pt32, sizeof(float2) * (size_t)n));
        ctx->inst_cap = n;
    }
    CK(cudaMemcpyAsync(ctx->d_raw, xy, sizeof(double2) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_prep_points(ctx->d_raw, ctx->d_pt64, ctx->d_pt32, n, weight_type, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->inst.pt64 = ctx->d_pt64;
    ctx->inst.pt32 = ctx->d_pt32;
    ctx->inst.dmat = nullptr;
    ctx->inst.dmat_ld = 0;
    ctx->h_xy.assign(xy, xy + 2 * (size_t)n);
    return TSPB200_OK;
}

// ---- distance matrix -------------------------------------------------------------------------------------
int tspb200_dist_matrix_build(tspb200_ctx *ctx, double *gpu_ms) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    const long long ld = ((long long)n + 3) / 4 * 4;
    if (!ctx->d_mat) {
        size_t bytes = (size_t)n * (size_t)ld * sizeof(int);
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        if (bytes + (1ull << 30) > free_b)
            return fail(ctx, TSPB200_E_UNSUPPORTED, "distance matrix of %d nodes needs %.1f GB, %.1f GB free: use the on-the-fly path", n, bytes / 1e9, free_b / 1e9);
        CK(cudaMalloc(&ctx->d_mat, bytes));
        ctx->mat_ld = ld;
    }
    InstDev I = ctx->inst;
    I.dmat = nullptr;  // the kernel computes, never gathers
    const bool fast = I.fp32_ok && I.exact32;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    unsigned long long *d_near = nullptr;
    if (I.metric == TSPB200_GEO) {  // GEO: count entries that sit on a rounding boundary (library cos / acos, see tsp_device.cuh)
        d_near = static_cast<unsigned long long *>(dev_scratch(ctx, 8, sizeof(unsigned long long)));
        if (!d_near) return fail(ctx, TSPB200_E_CUDA, "cudaMalloc failed");
        CK(cudaMemsetAsync(d_near, 0, sizeof(unsigned long long), ctx->stream));
    }
    CK(launch_dist_matrix(I, ctx->d_mat, ld, 0, n, fast, d_near, ctx->stream));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    if (d_near) CK(cudaMemcpyAsync(&ctx->geo_near, d_near, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (gpu_ms) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        *gpu_ms = ms;
    }
    return TSPB200_OK;
}

int tspb200_dist_matrix_get(tspb200_ctx *ctx, int32_t *out) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->d_mat) return fail(ctx, TSPB200_E_STATE, "no resident matrix");
    if (!out) return fail(ctx, TSPB200_E_ARG, "null output");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    CK(cudaMemcpy2DAsync(out, sizeof(int) * (size_t)n, ctx->d_mat, sizeof(int) * (size_t)ctx->mat_ld, sizeof(int) * (size_t)n,
                         (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSPB200_OK;
}

int tspb200_dist_matrix(tspb200_ctx *ctx, int32_t *out) {
    int rc = tspb200_dist_matrix_build(ctx, nullptr);
    if (rc) return rc;
    return tspb200_dist_matrix_get(ctx, out);
}

// One row of the matrix, out[j] = (int32) calc_dist(i, j), computed on the device without building the matrix (instances whose
// n x n matrix is not wanted on the host: the drop-in's scalar calc_dist fetches rows through this).
int tspb200_dist_row(tspb200_ctx *ctx, int i, int32_t *out) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    if (!out || i < 0 || i >= ctx->n) return fail(ctx, TSPB200_E_ARG, "bad row %d", i);
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    const long long ld = ((long long)n + 3) / 4 * 4;
    SCRATCH(d_row, int *, 13, sizeof(int) * (size_t)ld);
    InstDev I = ctx->inst;
    I.dmat = nullptr;
    CK(launch_dist_matrix(I, d_row, ld, i, i + 1, I.fp32_ok && I.exact32, nullptr, ctx->stream));
    CK(cudaMemcpyAsync(out, d_row, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSPB200_OK;
}

int tspb200_dist_matrix_free(tspb200_ctx *ctx) {
    if (!ctx || !ctx->stream) return TSPB200_E_CUDA;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->d_mat);
    ctx->d_mat = nullptr;
    ctx->mat_ld = 0;
    return TSPB200_OK;
}

// ---- tours -----------------------------------------------------------------------------------------------
// which evaluator a 2-opt run uses
static int select_path(const tspb200_ctx *ctx) {
    if (ctx->opt_force_path >= 0) return ctx->opt_force_path;
    if (ctx->inst.fp32_ok) return 0;
    return ctx->d_mat ? 2 : 1;
}

static InstDev inst_for_path(const tspb200_ctx *ctx, int path) {
    InstDev I = ctx->inst;
    if (path == 2) { I.dmat = ctx->d_mat; I.dmat_ld = ctx->mat_ld; }
    else { I.dmat = nullptr; I.dmat_ld = 0; }
    if (path != 0) I.fp32_ok = 0;
#if TSPB_FILTER_PROBE
    I.probe_on = ctx->probe_H != 0;
    I.probe_H = ctx->probe_H;
    I.probe_rec = ctx->d_probe;
    I.probe_count = ctx->d_probe_count;
    I.probe_cap = ctx->probe_cap;
#endif
    return I;
}

// Tile plan of the best-improvement scan (pure host arithmetic, also exported for the CPU-side tests).
// Tile-row I covers positions [I*TI, (I+1)*TI), TI = T*R (threads per block x rows per thread); its tile columns are
// J0(I)..(n-1)/TJ with J0(I) = (I*TI + 2) / TJ, i.e. every column block that can hold a q >= p+2 for some p of the row.
static long long tile_plan(int n, int TI, int TJ, std::vector<int> *row_start, std::vector<int> *row_j0) {
    const int ntr = n >= 4 ? (n - 2 + TI - 1) / TI : 0;
    long long total = 0;
    if (row_start) { row_start->clear(); row_j0->clear(); }
    for (int I = 0; I < ntr; ++I) {
        int j0 = (int)(((long long)I * TI + 2) / TJ);
        int jl = (n - 1) / TJ;
        if (row_start) { row_start->push_back((int)total); row_j0->push_back(j0); }
        total += (jl - j0 + 1);
    }
    if (row_start) row_start->push_back((int)total);
    return total;
}

// Picks (T, R, TJ) by a small cost model.  One round of tiles keeps an SM busy with (resident blocks per SM) x T threads,
// each doing (TJ + OV) column steps of R+1 square roots (OV ~ the row loads, first column and end-of-tile barrier), and the
// SFU is what those threads share.  A pass whose tiles fit the resident blocks is one such round; a deeper pass draws its
// tiles dynamically and ends within about one tile of the ideal, so
//   time ~ rounds x threads per SM x (TJ + OV) x (R + 1),   rounds = 1  or  tiles per rank / resident blocks + 1.
// The per-shape factors are measured on B200 at n = 100 000 (tools/shardshape.py): 64-thread blocks (8 per SM, 16 warps)
// hide latency best; R = 16 (1.0625 sqrt per move) pays with 150 registers, i.e. 12 warps per SM; R = 4 and 2 spend more
// instructions per move than their sqrt count alone says.
static int bi_blocks_per_sm(int t, int r, bool pruned = false) {  // 64 threads, exhaustive scan: TSPB_BI_MINBLOCKS64 (kernels_bi_scan.cuh)
    return r >= 16 ? (t == 256 ? 1 : 384 / t) : (t == 64 && !pruned ? 10 : 512 / t);
}

// With the row shuffle (64-thread shapes) a thread issues R instead of R + 1 square roots per column and a tile has
// (T/32)(32R - 1) rows; the factors of those shapes are the measured ones of the shuffle variant (64 x 4: 1435 vs 1288 us).
static void choose_tile_shape(int n, int num_sms, int world, int opt_T, int opt_R, int opt_TJ, bool shuffle, int *T, int *R, int *TJ) {
    struct Shape { int t, r; double penalty, penalty_shuffle; };
    const Shape cand[] = {{64, 8, 1.0, 1.0}, {128, 16, 1.04, 0}, {128, 8, 1.015, 0}, {256, 8, 1.05, 0}, {64, 4, 1.15, 1.11}, {64, 2, 1.3, 1.25}};
    const double OV = 16.0;
    double best = 1e300;
    int bt = 64, br = 2, btj = 32;
    for (const Shape &c : cand) {
        const int t = opt_T ? opt_T : c.t, r = opt_R ? opt_R : c.r;
        if (!bi_shape_supported(t, r)) continue;
        const int bps = bi_blocks_per_sm(t, r);
        const long long slots = (long long)num_sms * bps;
        for (int tj = 32; tj <= 256; tj += 8) {
            const int tjj = opt_TJ ? opt_TJ : tj;
            const bool sh = shuffle && bi_shuffle_supported(t, r);
            const long long nt = tile_plan(n, bi_tile_rows(t, r, sh ? 1 : 0), tjj, nullptr, nullptr);
            const long long per_rank = (nt + world - 1) / world;
            const double rounds = per_rank <= slots ? 1.0 : (double)per_rank / (double)slots + 1.0;
            if (r >= 16 && rounds < 4.0 && !opt_R) continue;  // 12 warps per SM hide the per-tile prologue only over several rounds
            const double cost = rounds * (bps * t) * (tjj + OV) * (sh ? r * (c.penalty_shuffle > 0 ? c.penalty_shuffle : c.penalty) : (r + 1) * c.penalty);
            if (cost < best) { best = cost; bt = t; br = r; btj = tjj; }
            if (opt_TJ) break;
        }
    }
    *T = bt; *R = br; *TJ = btj;
}

// exact tile pruning pays once a pass is deep enough that skipping tiles outweighs the two extra (tiny) launches
constexpr int PRUNE_AUTO_MIN_N = 3000;
constexpr int BI_PREFILTER_MIN_N = 30000;  // exhaustive scans with at least this tour size's pairs per rank use the stage-1 prefilter (see tspb200_bi_run)
static bool prune_wanted(const tspb200_ctx *ctx) {
    return ctx->opt_prune >= 0 ? ctx->opt_prune == 1 : ctx->n >= PRUNE_AUTO_MIN_N;
}

static void plan_tiles(tspb200_ctx *ctx, std::vector<int> &row_start, std::vector<int> &row_j0) {
    const int world_eff = ctx->opt_debug_shard ? (ctx->opt_debug_shard >> 8) : ctx->world;
    // the shape search costs ~0.2 ms of host time: remembered per (n, ranks, options)
    const long long key[6] = {ctx->n, world_eff * 4 + (ctx->opt_row_shuffle + 1), ctx->opt_T, ctx->opt_R, ctx->opt_TJ, ctx->num_sms};
    if (memcmp(key, ctx->shape_key, sizeof key) != 0) {
        choose_tile_shape(ctx->n, ctx->num_sms, world_eff, ctx->opt_T, ctx->opt_R, ctx->opt_TJ, ctx->opt_row_shuffle != 0, &ctx->shape_T, &ctx->shape_R, &ctx->shape_TJ);
        memcpy(ctx->shape_key, key, sizeof key);
    }
    ctx->T = ctx->shape_T; ctx->R = ctx->shape_R; ctx->TJ = ctx->shape_TJ;
    // A pruned pass scans a few per cent of the tiles: small tiles (256 positions x 64 columns) hug the live region much
    // more tightly than the throughput shape (measured on uni100000: 64 x 4 x 64 -> 76 us per pass, 64 x 8 x 256 -> 130 us).
    // Mid-size tours have so few live tiles that a pass is one tile per block, i.e. as long as its slowest tile: smaller
    // tiles still (n = 10 000: 64 x 2 x 32 -> 25.7 us per pass, 64 x 4 x 64 -> 28.1; n = 20 000: 64 x 4 x 32 -> 31.5, 64 x 4 x 64 -> 32.2;
    // profiles/r2_prune_probe_small_tiles.jsonl).
    if (prune_wanted(ctx) && ctx->inst.fp32_ok && ctx->opt_force_path <= 0 && ctx->n >= PRUNE_AUTO_MIN_N) {
        if (!ctx->opt_T) ctx->T = 64;
        if (!ctx->opt_R) ctx->R = ctx->n < 15000 ? 2 : 4;
        if (!ctx->opt_TJ) ctx->TJ = ctx->n < 40000 ? 32 : 64;
        if (!bi_shape_supported(ctx->T, ctx->R)) { ctx->T = 64; ctx->R = 4; }
    }
    const bool pruned_plan = prune_wanted(ctx) && ctx->inst.fp32_ok && ctx->opt_force_path <= 0 && ctx->n >= PRUNE_AUTO_MIN_N;
    const int slots = ctx->num_sms * bi_blocks_per_sm(ctx->T, ctx->R, pruned_plan);
    ctx->row_shuffle = (ctx->opt_row_shuffle != 0 && bi_shuffle_supported(ctx->T, ctx->R)) ? 1 : 0;
    ctx->ntiles = (int)tile_plan(ctx->n, bi_tile_rows(ctx->T, ctx->R, ctx->row_shuffle), ctx->TJ, &row_start, &row_j0);
    ctx->ntr = (int)row_j0.size();
    long long per_rank = (ctx->ntiles + world_eff - 1) / world_eff;
    int grid = ctx->opt_grid > 0 ? ctx->opt_grid : slots;
    if (grid > per_rank) grid = (int)(per_rank > 0 ? per_rank : 1);
    if (grid > 4096) grid = 4096;  // block_best[] capacity
    ctx->grid_bi = grid;
}

// Timing experiments: copies a device-side debug buffer to the host ("block_times": [grid][2] %globaltimer stamps of the
// last best-improvement pass run with option "timing" = 2).
int tspb200_debug_fetch(tspb200_ctx *ctx, const char *what, void *out, int64_t bytes) {
    if (!ctx || !ctx->stream || !what || !out) return TSPB200_E_ARG;
#if TSPB_FILTER_PROBE
    if (std::string(what) == "probe") {  // the records of the last probed pass, at most probe_cap of them
        if (!ctx->d_probe) return fail(ctx, TSPB200_E_STATE, "nothing recorded for probe");
        CK(cudaSetDevice(ctx->device));
        CK(cudaStreamSynchronize(ctx->stream));
        const int64_t have = (int64_t)sizeof(ProbeRec) * ctx->probe_cap;
        CK(cudaMemcpy(out, ctx->d_probe, (size_t)(bytes < have ? bytes : have), cudaMemcpyDeviceToHost));
        return TSPB200_OK;
    }
#endif
    const bool phases = std::string(what) == "block_phases";  // [grid][8]: start, drawn, loaded, scanned, folded, tiles, ticket, -
    if ((std::string(what) != "block_times" && !phases) || !ctx->d_dbg) return fail(ctx, TSPB200_E_STATE, "nothing recorded for %s", what);
    const int64_t have = (int64_t)sizeof(unsigned long long) * (phases ? 8 : 2) * 4096;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(out, ctx->d_dbg + (phases ? 8192 : 0), (size_t)(bytes < have ? bytes : have), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSPB200_OK;
}

// Host-only helper (no device needed): the tile plan for (n, T, R, TJ); T, R or TJ == 0 -> automatic choice for
// `num_sms` SMs and `world` ranks. row_start gets ntr+1 entries, row_j0 ntr entries.
int tspb200_debug_tile_plan_ex(int n, int T, int R, int TJ, int num_sms, int world, int row_shuffle, int *out_T, int *out_R,
                               int *out_TJ, int *out_tile_rows, int *row_start, int *row_j0, int cap, int *ntr) {
    if (n < 1 || num_sms < 1 || world < 1) return TSPB200_E_ARG;
    int t = T, r = R, tj = TJ;
    if (t == 0 || r == 0 || tj == 0) choose_tile_shape(n, num_sms, world, T, R, TJ, row_shuffle != 0, &t, &r, &tj);
    if (!bi_shape_supported(t, r)) return TSPB200_E_ARG;
    const int sh = (row_shuffle && bi_shuffle_supported(t, r)) ? 1 : 0;  // what plan_tiles() does with the option
    const int TI = bi_tile_rows(t, r, sh);
    std::vector<int> rs, rj;
    tile_plan(n, TI, tj, &rs, &rj);
    if ((int)rs.size() > cap) return TSPB200_E_ARG;
    for (size_t k = 0; k < rs.size(); ++k) row_start[k] = rs[k];
    for (size_t k = 0; k < rj.size(); ++k) row_j0[k] = rj[k];
    if (ntr) *ntr = (int)rj.size();
    if (out_T) *out_T = t;
    if (out_R) *out_R = r;
    if (out_TJ) *out_TJ = tj;
    if (out_tile_rows) *out_tile_rows = TI;
    return TSPB200_OK;
}

int tspb200_debug_tile_plan(int n, int T, int R, int TJ, int num_sms, int world, int *out_T, int *out_R, int *out_TJ,
                            int *row_start, int *row_j0, int cap, int *ntr) {
    return tspb200_debug_tile_plan_ex(n, T, R, TJ, num_sms, world, 0, out_T, out_R, out_TJ, nullptr, row_start, row_j0, cap, ntr);
}

int tspb200_tour_upload(tspb200_ctx *ctx, const int32_t *succ, int64_t log_cap) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    if (!succ) return fail(ctx, TSPB200_E_ARG, "null succ");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    if (!(ctx->dist_bound < 16777216.0))
        return fail(ctx, TSPB200_E_UNSUPPORTED, "2-opt keeps edge lengths as exact integers in FP32 words: distances up to %.0f "
                    "(>= 2^24) are not supported", ctx->dist_bound);
    // successor array -> visiting order from node 0 (also validates that succ is one Hamiltonian cycle): by pointer jumping
    // on the device for big tours (kernels_misc.cu launch_succ_to_order), by a walk on the host for small ones
    const bool rank_on_device = ctx->opt_upload_rank >= 0 ? ctx->opt_upload_rank == 1 : n >= 2048;
    std::vector<int> order(rank_on_device ? 0 : (size_t)n);
    if (!rank_on_device) {
        std::vector<unsigned char> seen((size_t)n, 0);
        int at = 0;
        for (int p = 0; p < n; ++p) {
            if (at < 0 || at >= n || seen[at]) return fail(ctx, TSPB200_E_ARG, "succ[] is not a single cycle over %d nodes", n);
            seen[at] = 1;
            order[p] = at;
            at = succ[at];
        }
        if (at != 0) return fail(ctx, TSPB200_E_ARG, "succ[] does not close the cycle at node 0");
    }
    std::vector<int> row_start, row_j0;
    plan_tiles(ctx, row_start, row_j0);
    const int TI = ctx->T * ctx->R;  // (an upper bound of the tile height when the shuffle variant is planned)
    const int alloc = ((n + TI - 1) / TI) * TI + 2 * TI + 1024 + 16;
    if (n > ctx->tour_cap_n || alloc > ctx->tour_cap_rec || log_cap > ctx->tour_cap_log) {
        free_tour(ctx);
        CK(cudaMalloc(&ctx->tour.rec, sizeof(float4) * (size_t)alloc));
        CK(cudaMalloc(&ctx->tour.pos, sizeof(int) * (size_t)n));
        CK(cudaMalloc(&ctx->tour.nrec, sizeof(float4) * (size_t)n));
        CK(cudaMalloc(&ctx->tour.nlnk, sizeof(float4) * (size_t)n));
        CK(cudaMalloc(&ctx->tour.npxy, sizeof(float2) * (size_t)n));
        CK(cudaMalloc(&ctx->tour.block_best, sizeof(MoveKey) * 4096));
        if (log_cap > 0) CK(cudaMalloc(&ctx->tour.log, sizeof(MoveRec) * (size_t)log_cap));
        CK(cudaMalloc(&ctx->d_order, sizeof(int) * (size_t)n));
        CK(cudaMalloc(&ctx->d_succ, sizeof(int) * (size_t)n));
        CK(cudaMalloc(&ctx->d_cost, sizeof(unsigned long long)));
        ctx->tour_cap_n = n;
        ctx->tour_cap_rec = alloc;
        ctx->tour_cap_log = log_cap;
    }
    ctx->tour.n = n;
    ctx->tour.alloc = alloc;
    ctx->tour.ctl = ctx->d_ctl;
    ctx->tour.log_cap = log_cap;  // entries the kernels may write (<= allocated); 0 with a null pointer = no log
    if (log_cap == 0 && ctx->tour_cap_log == 0) ctx->tour.log = nullptr;
    ctx->log_cap = log_cap;
    const int tile_need = (int)row_start.size() + 1;
    if (tile_need > ctx->tile_cap) {
        cudaFree(ctx->d_tile_row_start); cudaFree(ctx->d_tile_row_j0);
        ctx->d_tile_row_start = ctx->d_tile_row_j0 = nullptr;
        ctx->tile_cap = 0;
        CK(cudaMalloc(&ctx->d_tile_row_start, sizeof(int) * (size_t)tile_need));
        CK(cudaMalloc(&ctx->d_tile_row_j0, sizeof(int) * (size_t)tile_need));
        ctx->tile_cap = tile_need;
    }
    // exact tile pruning: boxes per tile-row / tile-column and the live-tile list of this rank
    {
        const int box_need = n / 32 + 8;  // >= tile-columns at the smallest tile width and >= tile-rows
        if (box_need > ctx->box_cap) {
            cudaFree(ctx->tour.rowbox); cudaFree(ctx->tour.colbox); cudaFree(ctx->tour.rowmaxds); cudaFree(ctx->tour.colmaxds);
            cudaFree(ctx->tour.colbox2); cudaFree(ctx->tour.colmaxds2);
            ctx->tour.rowbox = ctx->tour.colbox = ctx->tour.colbox2 = nullptr;
            ctx->tour.rowmaxds = ctx->tour.colmaxds = ctx->tour.colmaxds2 = nullptr;
            ctx->box_cap = 0;
            CK(cudaMalloc(&ctx->tour.rowbox, sizeof(float4) * (size_t)box_need));
            CK(cudaMalloc(&ctx->tour.colbox, sizeof(float4) * (size_t)box_need));
            CK(cudaMalloc(&ctx->tour.rowmaxds, sizeof(float) * (size_t)box_need));
            CK(cudaMalloc(&ctx->tour.colmaxds, sizeof(float) * (size_t)box_need));
            CK(cudaMalloc(&ctx->tour.colbox2, sizeof(float4) * (size_t)box_need));
            CK(cudaMalloc(&ctx->tour.colmaxds2, sizeof(float) * (size_t)box_need));
            ctx->box_cap = box_need;
        }
        // at least one entry per block of the scan grid: a block reads entry blockIdx.x before it knows how many are live
        const long long live_need = (long long)(ctx->ntiles > 4096 ? ctx->ntiles : 4096) + 32;
        if (live_need > ctx->live_cap) {
            cudaFree(ctx->tour.live);
            ctx->tour.live = nullptr;
            ctx->live_cap = 0;
            CK(cudaMalloc(&ctx->tour.live, sizeof(int2) * (size_t)live_need));
            CK(cudaMemsetAsync(ctx->tour.live, 0, sizeof(int2) * (size_t)live_need, ctx->stream));
            ctx->live_cap = live_need;
        }
    }
    CK(cudaMemcpyAsync(ctx->d_tile_row_start, row_start.data(), sizeof(int) * row_start.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (!row_j0.empty())
        CK(cudaMemcpyAsync(ctx->d_tile_row_j0, row_j0.data(), sizeof(int) * row_j0.size(), cudaMemcpyHostToDevice, ctx->stream));
    int *d_rank_err = nullptr;
    if (rank_on_device) {
        SCRATCH(d_work, unsigned char *, 19, sizeof(int2) * 2 * (size_t)n + sizeof(int) * ((size_t)n + 4));
        d_rank_err = reinterpret_cast<int *>(d_work + sizeof(int2) * 2 * (size_t)n + sizeof(int) * (size_t)n);
        CK(cudaMemcpyAsync(ctx->d_succ, succ, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemsetAsync(ctx->d_order, 0, sizeof(int) * (size_t)n, ctx->stream));  // a rejected succ[] leaves holes: keep them valid node ids
        CK(launch_succ_to_order(ctx->d_succ, n, d_work, ctx->d_order, d_rank_err, ctx->stream));
    } else {
        CK(cudaMemcpyAsync(ctx->d_order, order.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    }
    Ctl c0;
    memset(&c0, 0, sizeof c0);
    c0.cur_i = 0; c0.cur_j = 1;
    c0.fi_found = FI_NONE;
    c0.max_moves = -1;
    c0.last.i = c0.last.j = 0x7fffffff;
    c0.pass_min = KEY_PACK_NONE;
    c0.tm_scan_first = c0.tm_blk_end_min = c0.tm_apply_first = ~0ull;
    *ctx->h_ctl = c0;
    ctx->node_dirty = true;  // the node-space tables are built by the first first-improvement run that needs them
    ctx->fi_cursor_stale = false;
    ctx->tour_changed = false;
    CK(cudaMemcpyAsync(ctx->d_ctl, ctx->h_ctl, sizeof(Ctl), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->tour.block_best, 0, sizeof(MoveKey) * 4096, ctx->stream));  // delta 0 = "no previous winner"
    InstDev I = inst_for_path(ctx, select_path(ctx));
    CK(launch_build_state(I, ctx->tour, ctx->d_order, ctx->stream));
    int rank_err = 0;
    if (rank_on_device) CK(cudaMemcpyAsync(&rank_err, d_rank_err, sizeof rank_err, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (rank_err) {  // (the state built from a bogus order is never used: has_tour stays false)
        ctx->has_tour = false;
        return fail(ctx, TSPB200_E_ARG, "succ[] is not a single cycle over %d nodes", n);
    }
    ctx->has_tour = true;
    return TSPB200_OK;
}

int tspb200_tour_download(tspb200_ctx *ctx, int32_t *succ, double *cost) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(ctx->d_cost, 0, sizeof(unsigned long long), ctx->stream));
    CK(launch_export_state(ctx->tour, ctx->d_succ, ctx->d_cost, ctx->stream));
    unsigned long long c = 0;
    if (succ) CK(cudaMemcpyAsync(succ, ctx->d_succ, sizeof(int) * (size_t)ctx->n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&c, ctx->d_cost, sizeof c, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (cost) *cost = (double)(long long)c;
    return TSPB200_OK;
}

int tspb200_tour_log(tspb200_ctx *ctx, tspb200_move *log, int64_t cap, int64_t *count) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(ctx->h_ctl, ctx->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    long long have = ctx->h_ctl->log_count;
    if (have > ctx->log_cap) have = ctx->log_cap;
    if (have > cap) have = cap;
    if (count) *count = ctx->h_ctl->log_count;
    if (log && have > 0) {
        static_assert(sizeof(tspb200_move) == sizeof(MoveRec), "log record layout");
        CK(cudaMemcpyAsync(log, ctx->tour.log, sizeof(MoveRec) * (size_t)have, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return TSPB200_OK;
}

static int run_batch(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int batch, tspb200_stats *st, tspb200_move *log,
                     int64_t log_cap, int64_t *log_count);

static int run_batch_sequential(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int batch, tspb200_stats *st,
                                tspb200_move *log, int64_t log_cap, int64_t *log_count);

static int sync_ctl(tspb200_ctx *ctx) {
    CK(cudaMemcpyAsync(ctx->h_ctl, ctx->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_ctl->error == 2) return fail(ctx, TSPB200_E_NCCL, "multi-GPU exchange timed out: a peer rank never delivered its key");
    if (ctx->h_ctl->error) return fail(ctx, TSPB200_E_DEVICE_CHECK, "device-side consistency check failed (code %d)", ctx->h_ctl->error);
    return TSPB200_OK;
}

// A run that stopped at a cap leaves done = 1 behind with done_reason = DONE_CAP; the next run — whichever mode — clears
// it (include/tspb200.h: repeated calls continue where the previous one stopped).  A real local optimum stays final.
// `reset_fi_cursor`: the first-improvement sweep state refers to a tour that best-improvement moves have changed since;
// the next fi_run starts a fresh sweep.  The host owns the state here: the stream was just synchronised by sync_ctl().
static int prepare_run(tspb200_ctx *ctx, bool reset_fi_cursor, long long max_moves_abs) {
    Ctl *h = ctx->h_ctl;
    if (h->done && (h->done_reason == DONE_CAP || ctx->tour_changed)) {
        h->done = 0;
        h->done_reason = DONE_NONE;
    }
    ctx->tour_changed = false;
    if (reset_fi_cursor) {
        h->cur_i = 0;
        h->cur_j = 1;
        h->sweep_moves = 0;
        h->fi_found = FI_NONE;
        h->fi_seg = 0;
    }
    h->max_moves = max_moves_abs;
    h->fi_shard_min_gap = ctx->opt_fi_shard_min_gap;
    h->fi_pend_node = -1;
    h->fi_mode[0] = h->fi_mode[1] = 0;
    h->fi_sel[0] = h->fi_sel[1] = FI_NONE;  // both hit words of the late-selection search start clean, parity 0 first
    ctx->fi_parity = 0;
    if (reset_fi_cursor || ctx->opt_fi_shard_min_gap == 0) h->fi_shard = ctx->opt_fi_shard_min_gap == 0 ? 1 : 0;
    CK(cudaMemcpyAsync(ctx->d_ctl, h, sizeof(Ctl), cudaMemcpyHostToDevice, ctx->stream));
    return TSPB200_OK;
}

int tspb200_bi_run(tspb200_ctx *ctx, int64_t max_passes, tspb200_stats *st) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    int path = select_path(ctx);
    if (ctx->tabu_on) {  // the masked scan is the literal (exact) evaluator: matrix gather when resident, else FP64
        if (ctx->world > 1) return fail(ctx, TSPB200_E_UNSUPPORTED, "the tabu-masked scan is single-GPU");
        path = ctx->d_mat ? 2 : 1;
    }
    if (path == 2 && !ctx->d_mat) return fail(ctx, TSPB200_E_STATE, "matrix path selected but no resident matrix");
    if (path == 0 && !ctx->inst.fp32_ok) return fail(ctx, TSPB200_E_UNSUPPORTED, "FP32 filter path is not valid for this instance");
    const bool packable = n <= KEY_PACK_MAX_N && 2.0 * ctx->dist_bound < (double)KEY_PACK_MAX_DELTA;
    if (ctx->world > 1 && !packable)
        return fail(ctx, TSPB200_E_UNSUPPORTED, "multi-GPU key packing supports n <= 131072 and |delta| < 2^27");
    InstDev I = inst_for_path(ctx, path);
    BiArgs a;
    a.inst = I;
    a.tour = ctx->tour;
    a.tile_row_start = ctx->d_tile_row_start;
    a.tile_row_j0 = ctx->d_tile_row_j0;
    a.ntr = ctx->ntr;
    a.ntiles = ctx->ntiles;
    a.TJ = ctx->TJ;
    a.rank = ctx->rank;
    a.world = ctx->world;
    if (ctx->opt_debug_shard && ctx->world == 1) {  // timing experiment: a rank's share of the tiles, everything else single-GPU
        a.world = ctx->opt_debug_shard >> 8;
        a.rank = ctx->opt_debug_shard & 0xff;
    }
    // 2 = the scan kernel's last block also applies the move (mid-size tours: a launch costs more than the swap)
    const bool fuse_in_kernel = ctx->world == 1 && path == 0 && !ctx->tabu_on &&
                                (ctx->opt_fuse_apply >= 0 ? ctx->opt_fuse_apply == 1 : false);
    a.fuse_apply = ctx->world == 1 ? (fuse_in_kernel ? 2 : 1) : 0;
    a.seed_hint = ctx->opt_seed_hint;
    a.packed_tail = (path == 0 && packable && ctx->opt_seed_hint < 2) ? 1 : 0;
    // E: the square-root filter's own FP32 error (< 1.75 eps: two distances, three sums) plus the roundings of the
    // prefilter's a = ds_p + h, b = ds_q + h and h (< 0.75 eps), DESIGN.md §3
    a.pf_slack = 4.0f * ctx->eps32;
    a.pf_cx = ctx->pf_cx;
    a.pf_cy = ctx->pf_cy;
    a.timing = ctx->opt_timing;
    if (a.timing == 2 && !ctx->d_dbg) CK(cudaMalloc(&ctx->d_dbg, sizeof(unsigned long long) * (2 + 8) * 4096));  // {start, end} + 8 phase stamps per block
    a.dbg = ctx->d_dbg;
    // exact tile pruning: same moves, fewer evaluated pairs (the throughput benchmarks switch it off: "prune" = 0)
    const bool prune = path == 0 && !ctx->tabu_on && ctx->ntr > 0 && prune_wanted(ctx);
    a.pruned = prune ? 1 : 0;
    // stage-1 prefilter (kernels_bi_scan.cuh): exhaustive scans with a large share of pairs per rank.  Measured on B200
    // (profiles/r4_prefilter_by_n_w1.jsonl): a pass at n = 100 000 is 25 % faster, one at n = 10 000 slower — a pass of one or a
    // few waves is latency-bound, and its stage-1 hits (an L2 round trip each) sit on the critical path.  What counts is the
    // work of this rank, n^2 / (2 world) pairs, so the rule compares that with a single-GPU pass at BI_PREFILTER_MIN_N.
    // Pruned passes scan only the tiles that hold improving moves, where stage 1 hits too often to pay (DESIGN.md §4.1).
    const bool pf_auto = (double)n * (double)n >= (double)BI_PREFILTER_MIN_N * BI_PREFILTER_MIN_N * a.world;
    a.prefilter = (!prune || TSPB_BI_PREFILTER_PRUNED) && (ctx->opt_prefilter == 1 || (ctx->opt_prefilter == -1 && pf_auto)) ? 1 : 0;
    a.row_shuffle = ctx->row_shuffle;
    // multi-GPU: keys travel as NVLink peer stores from the scan kernel (path 0) unless NCCL was asked for
    const bool use_xchg = ctx->world > 1 && path == 0 && ctx->xchg.enabled && ctx->opt_exchange == 0;
    a.xchg = ctx->xchg;
    a.xchg.enabled = use_xchg ? 1 : 0;
    // programmatic dependent launch along the (prune ->) scan -> apply chain; not across a NCCL collective
    const bool pdl = path == 0 && !ctx->tabu_on && ctx->opt_pdl && (ctx->world == 1 || use_xchg);
    // "seed_hint" = 2: the apply launch's last block re-evaluates every block winner of the pass and seeds the next pass's
    // filter with the best one that is still legal.  It halves the exact-path calls of a one-wave pass (n = 10 000: 356 k ->
    // 188 k per run) but lengthens the serial section by ~5 us, a net loss (36.4 vs 32.3 us per pass): off by default.
    bool seed_all = path == 0 && !prune && ctx->opt_seed_hint >= 2;
    int grid_seed = ctx->grid_bi;  // block winners of the previous pass the pruned mode's tile_boxes_kernel re-evaluates
    int rc = sync_ctl(ctx);
    if (rc) return rc;
#if TSPB_FILTER_PROBE
    if (I.probe_on) {  // the threshold starts at H and no seed may lower it (the cold paths return no key)
        a.seed_hint = 0;
        seed_all = false;
        grid_seed = 0;
        ctx->h_ctl->hint = ctx->probe_H;  // copied to the device by prepare_run
        CK(cudaMemsetAsync(ctx->d_probe_count, 0, sizeof(unsigned long long), ctx->stream));
    }
#endif
    rc = prepare_run(ctx, false, -1);
    if (rc) return rc;
    const long long passes0 = ctx->h_ctl->passes, moves0 = ctx->h_ctl->moves, delta0 = ctx->h_ctl->obj_delta;
    const unsigned long long scanned0 = ctx->h_ctl->tiles_scanned;
    int exact_grid = ctx->opt_grid > 0 ? ctx->opt_grid : 4 * ctx->num_sms;
    if (exact_grid > n) exact_grid = n > 0 ? n : 1;
    // passes per host round trip: large instances run for milliseconds per pass, small ones for microseconds
    // (a pass that finds the tour already optimal returns at once, so over-launching by a batch costs microseconds, while
    // every host round trip idles the GPU — and, on several GPUs, every rank that waits for this one's next key)
    const long long batch_cap = ctx->opt_batch > 0 ? ctx->opt_batch : (n >= 5000 && !prune ? 64 : 256);
    long long batch = ctx->opt_batch > 0 ? ctx->opt_batch : 8;  // grows: short runs (TSPLIB-size tours) stop after a few passes
    long long host_launches = 0;
    int status = TSPB200_LOCAL_OPTIMUM;
    // "l2_flush_bytes": every pass starts with a cold L2 and is timed by its own event pair (the flush is outside the
    // timed intervals); nothing else changes, and there is still no host round trip between the passes of a batch.
    // On several GPUs the ranks' flushes do not take the same time; an alignment barrier over the peer slots between the
    // flush and the start event keeps that skew — an artefact of the benchmark — out of the peers' timed intervals.
    const bool flush = ctx->opt_flush_bytes > 0;
    double flush_ms = 0;
    if (flush) {
        if (ctx->flush_cap < ctx->opt_flush_bytes) {
            cudaFree(ctx->d_flush);
            ctx->d_flush = nullptr;
            ctx->flush_cap = 0;
            CK(cudaMalloc(&ctx->d_flush, (size_t)ctx->opt_flush_bytes));
            ctx->flush_cap = ctx->opt_flush_bytes;
        }
        while ((long long)ctx->pass_events.size() < 2 * batch_cap) {
            cudaEvent_t e;
            CK(cudaEventCreate(&e));
            ctx->pass_events.push_back(e);
        }
    }
    auto t_start = std::chrono::steady_clock::now();
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    long long remaining = max_passes;
    bool done = ctx->h_ctl->done != 0;
    while (!done) {
        long long k = batch;
        if (max_passes >= 0) {
            if (remaining <= 0) { status = TSPB200_STOPPED_BY_CAP; break; }
            if (k > remaining) k = remaining;
        }
        for (long long q = 0; q < k; ++q) {
            if (flush) {
                CK(cudaMemsetAsync(ctx->d_flush, (int)(q & 0xff), (size_t)ctx->opt_flush_bytes, ctx->stream));
                if (use_xchg) CK(launch_rank_align(ctx->xchg, ctx->rank, ctx->world, ctx->d_ctl, ctx->stream));
                CK(cudaEventRecord(ctx->pass_events[2 * q], ctx->stream));
            }
            if (prune) {
                CK(launch_tile_prune(a, bi_tile_rows(ctx->T, ctx->R, ctx->row_shuffle), grid_seed, pdl, ctx->stream));
                host_launches += 2;
            }
            if (ctx->tabu_on)
                CK(launch_bi_scan_tabu(I, ctx->tour, ctx->d_skip, ctx->tabu_iter, ctx->tabu_tenure, ctx->d_zl, ctx->d_zl_count,
                                       ctx->zl_cap, exact_grid, ctx->stream));
            else if (path == 0) CK(launch_bi_scan(a, ctx->T, ctx->R, ctx->grid_bi, pdl, ctx->stream));
            else CK(launch_bi_scan_exact(I, ctx->tour, ctx->rank, ctx->world, a.fuse_apply, exact_grid, ctx->stream));
            host_launches++;
            if (ctx->world > 1 && !use_xchg) {  // NCCL variant; with peer memory the scan kernel's tail did the exchange
                unsigned long long *p = &ctx->d_ctl->packed;
                int nr = g_nccl.AllReduce(p, p, 1, NCCL_UINT64, NCCL_MIN, ctx->comm, ctx->stream);
                if (nr != 0) return fail(ctx, TSPB200_E_NCCL, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(nr) : "?");
                CK(launch_bi_decode_packed(ctx->tour, ctx->stream));
                host_launches++;
            }
            if (!fuse_in_kernel) {
                // exhaustive scan: the apply launch's last block seeds the next pass's filter from all block winners (the
                // pruned mode's tile_boxes_kernel does the same before its filter)
                CK(launch_apply_move(I, ctx->tour, ctx->num_sms, seed_all ? ctx->grid_bi : 0, ctx->opt_timing, pdl, false, 0, ctx->stream));
                host_launches++;
            }
            if (flush) CK(cudaEventRecord(ctx->pass_events[2 * q + 1], ctx->stream));
        }
        if (max_passes >= 0) remaining -= k;
        if (batch < batch_cap) batch = batch * 2 < batch_cap ? batch * 2 : batch_cap;
        rc = sync_ctl(ctx);
        if (rc) return rc;
        if (flush) {
            for (long long q = 0; q < k; ++q) {
                float ms = 0;
                CK(cudaEventElapsedTime(&ms, ctx->pass_events[2 * q], ctx->pass_events[2 * q + 1]));
                flush_ms += ms;
            }
        }
        done = ctx->h_ctl->done != 0;
        if (!done && ctx->opt_time_limit_ms > 0) {
            auto el = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t_start).count();
            int stop = el > ctx->opt_time_limit_ms ? 1 : 0;
            if (ctx->world > 1) {
                // the stop decision must be collective: a rank that left alone would leave its peers waiting for its keys
                CK(cudaMemcpyAsync(ctx->d_stop, &stop, sizeof stop, cudaMemcpyHostToDevice, ctx->stream));
                int nr = g_nccl.AllReduce(ctx->d_stop, ctx->d_stop, 1, NCCL_INT32, NCCL_MAX, ctx->comm, ctx->stream);
                if (nr != 0) return fail(ctx, TSPB200_E_NCCL, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(nr) : "?");
                CK(cudaMemcpyAsync(&stop, ctx->d_stop, sizeof stop, cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
            }
            if (stop) { status = TSPB200_TIME_LIMIT_EXCEEDED; break; }
        }
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_ctl->moves != moves0) {
        ctx->node_dirty = true;       // the node-space tables of the first-improvement search are rebuilt on demand
        ctx->fi_cursor_stale = true;
    }
    if (st) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        memset(st, 0, sizeof *st);
        st->passes = ctx->h_ctl->passes - passes0;
        st->moves = ctx->h_ctl->moves - moves0;
        const long long pairs = (long long)n * (n - 3) / 2;
        st->evals = st->passes * pairs;
        if (prune) {
            // pairs really evaluated (estimate: scanned tiles / this rank's tiles); the skipped ones were excluded by the bound
            const long long own = ((long long)ctx->ntiles - a.rank + a.world - 1) / a.world;
            st->tiles_scanned = (long long)(ctx->h_ctl->tiles_scanned - scanned0);
            st->tiles_total = st->passes * own;
            if (st->tiles_total > 0) st->evals = (long long)((double)st->evals * (double)st->tiles_scanned / (double)st->tiles_total);
        }
        st->launches = host_launches;
        st->obj_delta = ctx->h_ctl->obj_delta - delta0;
        st->gpu_ms = flush ? flush_ms : ms;
        st->status = done ? TSPB200_LOCAL_OPTIMUM : status;
        st->path = path;
        st->cost = 0;
    }
    return TSPB200_OK;
}

int tspb200_fi_run(tspb200_ctx *ctx, int64_t max_moves, tspb200_stats *st) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    const int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) return fail(ctx, TSPB200_E_STATE, "matrix path selected but no resident matrix");
    InstDev I = inst_for_path(ctx, path);
    int rc = sync_ctl(ctx);
    if (rc) return rc;
    const long long passes0 = ctx->h_ctl->passes, moves0 = ctx->h_ctl->moves, delta0 = ctx->h_ctl->obj_delta,
                    swept0 = ctx->h_ctl->pairs_swept;
    // max_moves is an absolute cap on the device counter
    long long cap = max_moves >= 0 ? moves0 + max_moves : -1;
    rc = prepare_run(ctx, ctx->fi_cursor_stale, cap);
    if (rc) return rc;
    ctx->fi_cursor_stale = false;
    if (n < 4) {  // no non-adjacent pair exists: one empty sweep
        if (st) { memset(st, 0, sizeof *st); st->passes = 1; st->path = path; }
        return TSPB200_OK;
    }
    if (ctx->node_dirty) {  // only the first-improvement apply launches keep the node-space tables current
        CK(launch_rebuild_node_space(ctx->tour, ctx->stream));
        ctx->node_dirty = false;
    }
    int grid = ctx->opt_grid > 0 ? ctx->opt_grid : 2 * ctx->num_sms;
    if (grid > n - 1) grid = n - 1;
    long long batch = ctx->opt_batch > 0 ? ctx->opt_batch : 128;
    long long host_launches = 0;
    int status = TSPB200_LOCAL_OPTIMUM;
    auto t_start = std::chrono::steady_clock::now();
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    bool done = false;
    if (max_moves == 0) { done = false; status = TSPB200_STOPPED_BY_CAP; }
    else {
        // several GPUs: the segments of the pair order are dealt over the ranks; the first improving pair of every rank is
        // min-exchanged through the NVLink peer slots inside the search kernel (or by NCCL + fi_finish_kernel)
        const bool use_xchg = ctx->world > 1 && ctx->xchg.enabled && ctx->opt_exchange == 0;
        const bool pdl = ctx->opt_pdl != 0 && (ctx->world == 1 || use_xchg);
        XchgDev xd = ctx->xchg;
        while (!done) {
            for (long long q = 0; q < batch; ++q) {
                // one GPU: the search only folds its hits into ctl->fi_sel[parity]; the apply launch takes the winner from there
                const bool late_ok = ctx->opt_fi_late && (ctx->world == 1 || use_xchg);  // (the NCCL exchange keeps the published-move path)
                const int late = late_ok ? 1 + (int)(ctx->fi_parity++ & 1) : 0;
                CK(launch_fi_search(I, ctx->tour, ctx->rank, ctx->world, use_xchg ? &xd : nullptr, late, grid, pdl, ctx->stream));
                host_launches++;
                if (ctx->world > 1 && !use_xchg) {
                    unsigned long long *p = &ctx->d_ctl->fi_found;
                    int nr = g_nccl.AllReduce(p, p, 1, NCCL_UINT64, NCCL_MIN, ctx->comm, ctx->stream);
                    if (nr != 0) return fail(ctx, TSPB200_E_NCCL, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(nr) : "?");
                    CK(launch_fi_finish(I, ctx->tour, ctx->stream));
                    host_launches++;
                }
                CK(launch_apply_move(I, ctx->tour, ctx->num_sms, 0, 0, pdl, true, late, ctx->stream));
                host_launches += 1;
            }
            rc = sync_ctl(ctx);
            if (rc) return rc;
            done = ctx->h_ctl->done != 0;
            if (!done && ctx->opt_time_limit_ms > 0) {
                auto el = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t_start).count();
                int stop = el > ctx->opt_time_limit_ms ? 1 : 0;
                if (ctx->world > 1) {  // collective decision, see tspb200_bi_run
                    CK(cudaMemcpyAsync(ctx->d_stop, &stop, sizeof stop, cudaMemcpyHostToDevice, ctx->stream));
                    int nr = g_nccl.AllReduce(ctx->d_stop, ctx->d_stop, 1, NCCL_INT32, NCCL_MAX, ctx->comm, ctx->stream);
                    if (nr != 0) return fail(ctx, TSPB200_E_NCCL, "ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(nr) : "?");
                    CK(cudaMemcpyAsync(&stop, ctx->d_stop, sizeof stop, cudaMemcpyDeviceToHost, ctx->stream));
                    CK(cudaStreamSynchronize(ctx->stream));
                }
                if (stop) { status = TSPB200_TIME_LIMIT_EXCEEDED; break; }
            }
        }
        if (done && cap >= 0 && ctx->h_ctl->moves >= cap) status = TSPB200_STOPPED_BY_CAP;
        if (ctx->opt_fi_late && (ctx->world == 1 || use_xchg)) CK(launch_fi_flush(ctx->tour, ctx->stream));  // the last apply's parked pos[] entry
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (st) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        memset(st, 0, sizeof *st);
        st->passes = ctx->h_ctl->passes - passes0;
        st->moves = ctx->h_ctl->moves - moves0;
        st->evals = ctx->h_ctl->pairs_swept - swept0;
        st->launches = host_launches;
        st->obj_delta = ctx->h_ctl->obj_delta - delta0;
        st->gpu_ms = ms;
        st->status = status;
        st->path = path;
    }
    return TSPB200_OK;
}

int tspb200_two_opt(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int64_t max_iters, tspb200_stats *st,
                    tspb200_move *log, int64_t log_cap, int64_t *log_count) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (mode != TSPB200_FI && mode != TSPB200_BI) return fail(ctx, TSPB200_E_ARG, "mode must be TSPB200_FI or TSPB200_BI");
    // TSPLIB-size tours run to their local optimum inside ONE thread block with the tour in shared memory: no launch per
    // move, which is what a ~1000-node tour is bound by on the grid path (FI: ~30 us per move; BI: ~16 us per pass).
    // Crossover measured on B200 (tools/firoute.py): FI up to ~1500 nodes (n = 1000: 4.7 vs 5.4 ms, n = 2000: 15.4 vs 13.2 ms),
    // BI up to ~160 (n = 128: 0.28 vs 0.39 ms, n = 200: 0.92 vs 0.78 ms).
    {
        const int n = ctx->n;
        const int lim = mode == TSPB200_FI ? 1536 : 160;
        const bool want = ctx->opt_single_block < 0 ? (n >= 1 && n <= lim) : (ctx->opt_single_block == 1 && (long long)n * 28 + 16 <= 200 * 1024);
        // (the block kernel cannot poll the clock; a tour this small is done within milliseconds, so any limit of a second
        // or more — the reference's CLI default is 900 s — is honoured trivially)
        const bool time_ok = ctx->opt_time_limit_ms <= 0 || ctx->opt_time_limit_ms >= 1000;
        if (want && max_iters < 0 && ctx->world == 1 && !ctx->tabu_on && time_ok && succ) {
            double o = obj ? *obj : 0.0;
            tspb200_stats local;
            int rc = run_batch(ctx, mode, succ, &o, 1, &local, log, log ? log_cap : 0, log_count);
            if (rc) return rc;
            if (obj) *obj = o;
            local.cost = o;
            if (st) *st = local;
            ctx->has_tour = false;  // the resident-tour state was not touched; make a stale one unusable
            return TSPB200_OK;
        }
    }
    int rc = tspb200_tour_upload(ctx, succ, log ? log_cap : 0);
    if (rc) return rc;
    tspb200_stats local;
    memset(&local, 0, sizeof local);
    rc = (mode == TSPB200_BI) ? tspb200_bi_run(ctx, max_iters, &local) : tspb200_fi_run(ctx, max_iters, &local);
    if (rc) return rc;
    double cost = 0;
    rc = tspb200_tour_download(ctx, succ, &cost);
    if (rc) return rc;
    if (mode == TSPB200_BI) {
        local.cost = cost;  // reference tabusearch.c:168-172: recomputed from scratch
        if (obj) *obj = cost;
    } else {
        double o = (obj ? *obj : 0.0) + (double)local.obj_delta;  // reference heuristics.c:486
        local.cost = o;
        if (obj) *obj = o;
    }
    if (log || log_count) {
        rc = tspb200_tour_log(ctx, log, log_cap, log_count);
        if (rc) return rc;
    }
    if (st) *st = local;
    return TSPB200_OK;
}

// alg_2opt_tabu with a tabu list (reference src/tabusearch.c:107-178): best improvement over the pairs that pass the
// four check_tenure() tests, with the reference's lazy-expiry side effects replayed on the caller's array.
int tspb200_two_opt_tabu(tspb200_ctx *ctx, int32_t *succ, double *obj, int32_t *skip_edge, int iter, int tenure,
                         int64_t max_passes, tspb200_stats *st, tspb200_move *log, int64_t log_cap, int64_t *log_count) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!skip_edge) return tspb200_two_opt(ctx, TSPB200_BI, succ, obj, max_passes, st, log, log_cap, log_count);
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    const int n = ctx->n;
    // the reference indexes the list with an int x_udir_pos (src/utility.c:17-30): n*(n-1)/2 must fit
    if (n > 46340) return fail(ctx, TSPB200_E_UNSUPPORTED, "tabu list index overflows int for n=%d (reference limit)", n);
    CK(cudaSetDevice(ctx->device));
    const long long len = (long long)n * (n - 1) / 2;
    if (ctx->skip_cap < len) {
        cudaFree(ctx->d_skip); cudaFree(ctx->d_zl); cudaFree(ctx->d_zl_count);
        ctx->d_skip = nullptr; ctx->d_zl = nullptr; ctx->d_zl_count = nullptr;
        ctx->skip_cap = 0;
        ctx->zl_cap = len < (1ll << 22) ? len : (1ll << 22);
        CK(cudaMalloc(&ctx->d_skip, sizeof(int) * (size_t)(len > 0 ? len : 1)));
        CK(cudaMalloc(&ctx->d_zl, sizeof(long long) * (size_t)(ctx->zl_cap > 0 ? ctx->zl_cap : 1)));
        CK(cudaMalloc(&ctx->d_zl_count, sizeof(unsigned long long)));
        ctx->skip_cap = len;
    }
    CK(cudaMemcpyAsync(ctx->d_skip, skip_edge, sizeof(int) * (size_t)len, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_zl_count, 0, sizeof(unsigned long long), ctx->stream));
    ctx->tabu_on = true;
    ctx->tabu_iter = iter;
    ctx->tabu_tenure = tenure;
    int rc = tspb200_two_opt(ctx, TSPB200_BI, succ, obj, max_passes, st, log, log_cap, log_count);
    ctx->tabu_on = false;
    if (rc) return rc;
    // replay the lazy expiry (check_tenure zeroes the entry, src/tabusearch.c:86-88) on the caller's list
    unsigned long long cnt = 0;
    CK(cudaMemcpyAsync(&cnt, ctx->d_zl_count, sizeof cnt, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if ((long long)cnt > ctx->zl_cap) {
        CK(cudaMemcpyAsync(skip_edge, ctx->d_skip, sizeof(int) * (size_t)len, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    } else if (cnt > 0) {
        std::vector<long long> zl((size_t)cnt);
        CK(cudaMemcpyAsync(zl.data(), ctx->d_zl, sizeof(long long) * (size_t)cnt, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (long long e : zl) skip_edge[e] = 0;
    }
    return TSPB200_OK;
}

// One thread block per tour, whole tour state in shared memory (csrc/kernels_batch.cu).  log / log_count: only for
// batch == 1 (the single-tour route of tspb200_two_opt for TSPLIB-size instances).
static int run_batch(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int batch, tspb200_stats *st, tspb200_move *log,
                     int64_t log_cap, int64_t *log_count) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    if (mode != TSPB200_FI && mode != TSPB200_BI) return fail(ctx, TSPB200_E_ARG, "mode must be TSPB200_FI or TSPB200_BI");
    if (!succ || batch < 1) return fail(ctx, TSPB200_E_ARG, "bad batch");
    if (!(ctx->dist_bound < 16777216.0))
        return fail(ctx, TSPB200_E_UNSUPPORTED, "2-opt keeps edge lengths as exact integers in FP32 words: distances up to %.0f "
                    "(>= 2^24) are not supported", ctx->dist_bound);
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    const int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) return fail(ctx, TSPB200_E_STATE, "matrix path selected but no resident matrix");
    InstDev I = inst_for_path(ctx, path);
    const long long lcap = (log && batch == 1 && log_cap > 0) ? log_cap : 0;
    SCRATCH(d_succ, int *, 0, sizeof(int) * (size_t)n * batch);
    SCRATCH(d_delta, long long *, 1, sizeof(long long) * (size_t)batch);
    SCRATCH(d_cnt, long long *, 2, sizeof(long long) * 4 * (size_t)batch);
    MoveRec *d_log = nullptr;
    if (lcap) {
        SCRATCH(d_log_, MoveRec *, 3, sizeof(MoveRec) * (size_t)lcap);
        d_log = d_log_;
    }
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    CK(cudaMemcpyAsync(d_succ, succ, sizeof(int) * (size_t)n * batch, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_delta, 0, sizeof(long long) * (size_t)batch, ctx->stream));
    CK(cudaMemsetAsync(d_cnt, 0, sizeof(long long) * 4 * (size_t)batch, ctx->stream));
#if TSPB_FILTER_PROBE
    if (I.probe_on) CK(cudaMemsetAsync(ctx->d_probe_count, 0, sizeof(unsigned long long), ctx->stream));
#endif
    int launched = 0;
    // best improvement on the FP32-filter path: the position-space block kernel; everything else: the node-space one
    cudaError_t le = cudaErrorNotSupported;
    if (mode == TSPB200_BI && path == 0 && ctx->opt_batch_kernel != 1)
        le = launch_two_opt_batch_bi_pos(I, d_succ, nullptr, d_delta, d_cnt, batch, ctx->num_sms, ctx->stream, &launched, d_log, lcap);
    if (le == cudaErrorNotSupported)
        le = launch_two_opt_batch(I, mode, d_succ, nullptr, d_delta, d_cnt, batch, ctx->num_sms, ctx->stream, &launched, d_log, lcap);
    if (le == cudaErrorInvalidValue) {
        // a tour that does not fit one block's shared memory: the tours go through the grid kernels one after the other
        // (still the CUDA path; the reference has no size limit either)
        cudaGetLastError();
        return run_batch_sequential(ctx, mode, succ, obj, batch, st, log, log_cap, log_count);
    }
    if (le != cudaSuccess) return fail(ctx, TSPB200_E_CUDA, "batched 2-opt launch failed: %s", cudaGetErrorString(le));
    std::vector<long long> h_delta((size_t)batch), h_cnt((size_t)batch * 4);
    CK(cudaMemcpyAsync(succ, d_succ, sizeof(int) * (size_t)n * batch, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(h_delta.data(), d_delta, sizeof(long long) * (size_t)batch, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(h_cnt.data(), d_cnt, sizeof(long long) * 4 * (size_t)batch, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (lcap) {
        long long have = h_cnt[0] < lcap ? h_cnt[0] : lcap;
        static_assert(sizeof(tspb200_move) == sizeof(MoveRec), "log record layout");
        if (have > 0) CK(cudaMemcpy(log, d_log, sizeof(MoveRec) * (size_t)have, cudaMemcpyDeviceToHost));
    }
    if (log_count) *log_count = batch == 1 ? h_cnt[0] : 0;
    tspb200_stats local;
    memset(&local, 0, sizeof local);
    for (int b = 0; b < batch; ++b) {
        local.moves += h_cnt[4 * b + 0];
        local.passes += h_cnt[4 * b + 1];
        local.evals += h_cnt[4 * b + 2];
        if (h_cnt[4 * b + 3]) return fail(ctx, mode >= 0 && batch == 1 ? TSPB200_E_ARG : TSPB200_E_DEVICE_CHECK,
                                          "2-opt: succ[] of tour %d is not a single cycle over %d nodes", b, n);
        if (mode == TSPB200_FI) local.obj_delta += h_delta[b];
        if (obj) {
            if (mode == TSPB200_BI) obj[b] = (double)h_delta[b];  // kernel stores the recomputed cost for BI
            else obj[b] += (double)h_delta[b];
        }
    }
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    local.gpu_ms = ms;
    local.launches = launched;
    local.path = path;
    local.status = TSPB200_LOCAL_OPTIMUM;
    if (batch == 1) local.cost = obj ? obj[0] : 0.0;
    if (st) *st = local;
    return TSPB200_OK;
}

// Tours too large for the one-block kernels: each tour runs through the resident-tour grid path (upload, run to the local
// optimum, download).  The context's resident tour is replaced.
static int run_batch_sequential(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int batch, tspb200_stats *st,
                                tspb200_move *log, int64_t log_cap, int64_t *log_count) {
    const int n = ctx->n;
    tspb200_stats total;
    memset(&total, 0, sizeof total);
    for (int b = 0; b < batch; ++b) {
        int32_t *s = succ + (size_t)b * n;
        const bool want_log = log && batch == 1 && log_cap > 0;
        int rc = tspb200_tour_upload(ctx, s, want_log ? log_cap : 0);
        if (rc) return rc;
        tspb200_stats one;
        memset(&one, 0, sizeof one);
        rc = mode == TSPB200_BI ? tspb200_bi_run(ctx, -1, &one) : tspb200_fi_run(ctx, -1, &one);
        if (rc) return rc;
        double cost = 0;
        rc = tspb200_tour_download(ctx, s, &cost);
        if (rc) return rc;
        if (obj) obj[b] = mode == TSPB200_BI ? cost : obj[b] + (double)one.obj_delta;
        if (want_log || (log_count && batch == 1)) {
            rc = tspb200_tour_log(ctx, log, log_cap, log_count);
            if (rc) return rc;
        }
        total.passes += one.passes; total.moves += one.moves; total.evals += one.evals; total.launches += one.launches;
        total.obj_delta += one.obj_delta; total.gpu_ms += one.gpu_ms; total.path = one.path;
        total.tiles_scanned += one.tiles_scanned; total.tiles_total += one.tiles_total;
    }
    total.status = TSPB200_LOCAL_OPTIMUM;
    if (batch == 1) total.cost = obj ? obj[0] : 0.0;
    if (st) *st = total;
    if (log_count && batch != 1) *log_count = 0;
    ctx->has_tour = false;
    return TSPB200_OK;
}

int tspb200_two_opt_batch(tspb200_ctx *ctx, int mode, int32_t *succ, double *obj, int batch, tspb200_stats *st) {
    return run_batch(ctx, mode, succ, obj, batch, st, nullptr, 0, nullptr);
}

int tspb200_nn_tour(tspb200_ctx *ctx, int start, int32_t *succ, double *cost) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    const int n = ctx->n;
    if (start < 0 || start >= n) return fail(ctx, TSPB200_E_ARG, "start node %d out of range", start);  // WRONG_STARTING_NODE
    CK(cudaSetDevice(ctx->device));
    int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) path = 1;
    InstDev I = inst_for_path(ctx, path == 2 ? 2 : 1);
    SCRATCH(d_succ, int *, 4, sizeof(int) * (size_t)n);
    // Planar metrics: the walk over a bucket grid (kernels_nn.cu) — same tour, ~10x fewer microseconds per step.
    const bool planar = ctx->metric == TSPB200_EUC_2D || ctx->metric == TSPB200_CEIL_2D || ctx->metric == TSPB200_ATT;
    const bool grid_wanted = ctx->opt_nn_grid >= 0 ? ctx->opt_nn_grid == 1 : n >= 256;
    if (planar && path != 2 && ctx->coords_finite && grid_wanted && n >= 2) {
        const double W = ctx->bb_xmax - ctx->bb_xmin, H = ctx->bb_ymax - ctx->bb_ymin;
        const long long nwords = ((long long)n + 31) / 32;
        const long long cap = (200ll * 1024 - 4 * nwords) / 4 - 2;  // cells whose table fits one block's shared memory next to the bitmask
        if (cap >= 16) {
            double cells = std::fmin(std::fmax((double)n / 2.5, 1.0), (double)(cap < 40000 ? cap : 40000));
            double h = (W > 0 && H > 0) ? std::sqrt(W * H / cells) : std::fmax(W, H) / cells;
            if (!(h > 0)) h = 1.0;
            long long gx, gy;
            for (;;) {
                gx = (long long)std::floor(W / h) + 1;
                gy = (long long)std::floor(H / h) + 1;
                if (gx * gy <= cap) break;
                h *= 1.1;
            }
            NnGridArgs g;
            g.inst = I; g.start = start; g.GX = (int)gx; g.GY = (int)gy;
            g.xmin = ctx->bb_xmin; g.ymin = ctx->bb_ymin;
            g.inv_h = 1.0 / h; g.h = 1.0 / g.inv_h;
            g.scale = ctx->metric == TSPB200_ATT ? 3.1622776601683795 * (1.0 + 1e-12) : 1.0;
            const size_t ncell = (size_t)(gx * gy);
            SCRATCH(d_cells, int *, 16, sizeof(int) * (2 * ncell + 2));
            SCRATCH(d_spt, double2 *, 17, sizeof(double2) * (size_t)n);
            SCRATCH(d_snode, int *, 18, sizeof(int) * ((size_t)n + 1));
            SCRATCH(d_gcost, long long *, 8, sizeof(long long));
            g.cell_cnt = d_cells; g.cell_fill = d_cells + ncell + 1;
            g.spt = d_spt; g.snode = d_snode; g.start_spos = d_snode + n;
            g.succ = d_succ; g.cost = d_gcost;
            cudaError_t ge = launch_nn_grid(g, ctx->num_sms, ctx->stream);
            long long gc = 0;
            if (ge == cudaSuccess) ge = cudaMemcpyAsync(succ, d_succ, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
            if (ge == cudaSuccess) ge = cudaMemcpyAsync(&gc, d_gcost, sizeof gc, cudaMemcpyDeviceToHost, ctx->stream);
            if (ge == cudaSuccess) ge = cudaStreamSynchronize(ctx->stream);
            if (ge != cudaSuccess) return fail(ctx, TSPB200_E_CUDA, "nearest-neighbour grid kernels failed: %s", cudaGetErrorString(ge));
            if (cost) *cost = (double)gc;
            return TSPB200_OK;
        }
    }
    SCRATCH(d_vis, unsigned char *, 5, (size_t)n);
    SCRATCH(d_slots, unsigned long long *, 6, sizeof(unsigned long long) * 3);
    SCRATCH(d_bar, unsigned *, 7, sizeof(unsigned));
    SCRATCH(d_cost, long long *, 8, sizeof(long long));
    CK(cudaMemsetAsync(d_vis, 0, (size_t)n, ctx->stream));
    CK(cudaMemsetAsync(d_slots, 0xff, sizeof(unsigned long long) * 3, ctx->stream));
    CK(cudaMemsetAsync(d_bar, 0, sizeof(unsigned), ctx->stream));
    NnArgs a;
    a.inst = I; a.start = start; a.succ = d_succ; a.visited = d_vis; a.slots = d_slots; a.barrier = d_bar; a.cost = d_cost;
    int grid = nn_max_grid(ctx->num_sms);
    int want = (n + 255) / 256;
    if (grid > want) grid = want;
    if (grid < 1) grid = 1;
    cudaError_t le = launch_nn_tour(a, grid, ctx->stream);
    long long c = 0;
    if (le == cudaSuccess) le = cudaMemcpyAsync(succ, d_succ, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    if (le == cudaSuccess) le = cudaMemcpyAsync(&c, d_cost, sizeof c, cudaMemcpyDeviceToHost, ctx->stream);
    if (le == cudaSuccess) le = cudaStreamSynchronize(ctx->stream);
    if (le != cudaSuccess) return fail(ctx, TSPB200_E_CUDA, "nearest-neighbour kernel failed: %s", cudaGetErrorString(le));
    if (cost) *cost = (double)c;
    return TSPB200_OK;
}

// Batched nearest neighbour: `batch` independent greedy() runs, one thread block each (reference HEU_Greedy_iter,
// src/heuristics.c:168-205, is this with starts = 0..n-1 followed by "keep the first strictly better tour").
int tspb200_nn_tour_batch(tspb200_ctx *ctx, const int32_t *starts, int batch, int32_t *succ, double *costs) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    if (!starts || !costs || batch < 1) return fail(ctx, TSPB200_E_ARG, "bad arguments");
    const int n = ctx->n;
    for (int b = 0; b < batch; ++b)
        if (starts[b] < 0 || starts[b] >= n) return fail(ctx, TSPB200_E_ARG, "start node %d out of range", starts[b]);  // WRONG_STARTING_NODE
    CK(cudaSetDevice(ctx->device));
    int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) path = 1;
    InstDev I = inst_for_path(ctx, path == 2 ? 2 : 1);
    I.fp32_ok = ctx->inst.fp32_ok;  // the FP32 filter of the batched kernel is valid whenever the 2-opt filter is
    const float eps = ctx->eps32;
    SCRATCH(d_starts, int *, 9, sizeof(int) * (size_t)batch);
    SCRATCH(d_cost, long long *, 10, sizeof(long long) * (size_t)batch);
    int *d_succ = nullptr;
    if (succ) {
        SCRATCH(d_succ_, int *, 11, sizeof(int) * (size_t)batch * n);
        d_succ = d_succ_;
    }
    CK(cudaMemcpyAsync(d_starts, starts, sizeof(int) * (size_t)batch, cudaMemcpyHostToDevice, ctx->stream));
    cudaError_t le = launch_nn_batch(I, d_starts, batch, d_succ, d_cost, eps, ctx->num_sms, ctx->stream);
    if (le == cudaErrorInvalidValue) {
        // the coordinates do not fit one block's shared memory (n > ~22 000): one grid-wide nearest-neighbour run per start
        cudaGetLastError();
        std::vector<int32_t> tmp(succ ? 0 : (size_t)n);
        for (int b = 0; b < batch; ++b) {
            int rc = tspb200_nn_tour(ctx, starts[b], succ ? succ + (size_t)b * n : tmp.data(), &costs[b]);
            if (rc) return rc;
        }
        return TSPB200_OK;
    }
    std::vector<long long> h((size_t)batch);
    if (le == cudaSuccess && succ) le = cudaMemcpyAsync(succ, d_succ, sizeof(int) * (size_t)batch * n, cudaMemcpyDeviceToHost, ctx->stream);
    if (le == cudaSuccess) le = cudaMemcpyAsync(h.data(), d_cost, sizeof(long long) * (size_t)batch, cudaMemcpyDeviceToHost, ctx->stream);
    if (le == cudaSuccess) le = cudaStreamSynchronize(ctx->stream);
    if (le != cudaSuccess) return fail(ctx, TSPB200_E_CUDA, "batched nearest-neighbour kernel failed: %s", cudaGetErrorString(le));
    for (int b = 0; b < batch; ++b) costs[b] = (double)h[(size_t)b];
    return TSPB200_OK;
}

// Extra-mileage construction (reference HEU_extramileage, src/heuristics.c:208-314).
int tspb200_extra_mileage(tspb200_ctx *ctx, int32_t *succ, double *cost) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 2) return fail(ctx, TSPB200_E_ARG, "extra mileage needs at least 2 nodes");
    if (!succ) return fail(ctx, TSPB200_E_ARG, "null succ");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) path = 1;
    InstDev I = inst_for_path(ctx, path == 2 ? 2 : 1);
    SCRATCH(d_succ, int *, 12, sizeof(int) * (size_t)n);
    SCRATCH(d_cost, long long *, 13, sizeof(long long));
    // instances whose insertion state (21 bytes per node) exceeds one block's shared memory keep it in a global work buffer
    SCRATCH(d_work, unsigned char *, 14, extra_mileage_state_bytes(n));
    cudaError_t le = launch_extra_mileage(I, d_succ, d_cost, d_work, ctx->opt_em_global != 0, ctx->stream);
    long long c = 0;
    if (le == cudaSuccess) le = cudaMemcpyAsync(succ, d_succ, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    if (le == cudaSuccess) le = cudaMemcpyAsync(&c, d_cost, sizeof c, cudaMemcpyDeviceToHost, ctx->stream);
    if (le == cudaSuccess) le = cudaStreamSynchronize(ctx->stream);
    if (le != cudaSuccess) return fail(ctx, TSPB200_E_CUDA, "extra-mileage kernel failed: %s", cudaGetErrorString(le));
    if (cost) *cost = (double)c;
    return TSPB200_OK;
}

int tspb200_tour_costs(tspb200_ctx *ctx, const int32_t *tours, int batch, int as_order, double *out) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    if (!tours || !out || batch < 1) return fail(ctx, TSPB200_E_ARG, "bad arguments");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) path = 1;
    InstDev I = inst_for_path(ctx, path == 2 ? 2 : 1);
    SCRATCH(d_t, int *, 14, sizeof(int) * (size_t)n * batch);
    SCRATCH(d_o, long long *, 15, sizeof(long long) * (size_t)batch);
    CK(cudaMemcpyAsync(d_t, tours, sizeof(int) * (size_t)n * batch, cudaMemcpyHostToDevice, ctx->stream));
    cudaError_t le = launch_tour_cost(I, d_t, nullptr, as_order, d_o, batch, ctx->stream);
    std::vector<long long> h((size_t)batch);
    if (le == cudaSuccess) le = cudaMemcpyAsync(h.data(), d_o, sizeof(long long) * (size_t)batch, cudaMemcpyDeviceToHost, ctx->stream);
    if (le == cudaSuccess) le = cudaStreamSynchronize(ctx->stream);
    if (le != cudaSuccess) return fail(ctx, TSPB200_E_CUDA, "tour cost kernel failed: %s", cudaGetErrorString(le));
    for (int b = 0; b < batch; ++b) out[b] = (double)h[b];
    return TSPB200_OK;
}

// ---- resident sessions -----------------------------------------------------------------------------------------
// The callers of the 2-opt path (reference HEU_VNS src/vns.c:103-183, tabu() src/tabusearch.c:188-320, HEU_Genetic
// src/genetic.c:445-560) alternate a small perturbation with a 2-opt run.  These entry points keep the tour / the tabu
// list / the population in HBM across those steps; the caller keeps the random number generator and the control flow.

int tspb200_tour_cost(tspb200_ctx *ctx, double *cost) { return tspb200_tour_download(ctx, nullptr, cost); }

// Saves / restores the resident tour (position-space records + positions) in one of two device slots: the "best solution so
// far" copies of reference vns.c:121-122,171-173 and tabusearch.c:241-243,313-314 without leaving the device.
int tspb200_tour_save(tspb200_ctx *ctx, int slot) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    if (slot < 0 || slot > 1) return fail(ctx, TSPB200_E_ARG, "slot must be 0 or 1");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n, alloc = ctx->tour.alloc;
    if (ctx->save_alloc[slot] < alloc) {
        cudaFree(ctx->save_rec[slot]); cudaFree(ctx->save_pos[slot]);
        ctx->save_rec[slot] = nullptr; ctx->save_pos[slot] = nullptr;
        ctx->save_alloc[slot] = 0;
        CK(cudaMalloc(&ctx->save_rec[slot], sizeof(float4) * (size_t)alloc));
        CK(cudaMalloc(&ctx->save_pos[slot], sizeof(int) * (size_t)alloc));
        ctx->save_alloc[slot] = alloc;
    }
    CK(cudaMemcpyAsync(ctx->save_rec[slot], ctx->tour.rec, sizeof(float4) * (size_t)alloc, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->save_pos[slot], ctx->tour.pos, sizeof(int) * (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->save_n[slot] = n;
    return TSPB200_OK;
}

int tspb200_tour_restore(tspb200_ctx *ctx, int slot) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    if (slot < 0 || slot > 1 || ctx->save_n[slot] != ctx->n || ctx->save_alloc[slot] < ctx->tour.alloc)
        return fail(ctx, TSPB200_E_STATE, "nothing saved in slot %d for this tour", slot);
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(ctx->tour.rec, ctx->save_rec[slot], sizeof(float4) * (size_t)ctx->tour.alloc, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->tour.pos, ctx->save_pos[slot], sizeof(int) * (size_t)ctx->n, cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->node_dirty = true;  // node-space tables are rebuilt from the records on the next first-improvement run
    ctx->fi_cursor_stale = true;
    ctx->tour_changed = true;
    return TSPB200_OK;
}

// reference src/vns.c:11-100 kick(): idx1, idx2, idx3 are the three tour indices the reference draws with rand_choice
// (in any order; they are sorted here like vns.c:34-50).  *cost (may be NULL) = the recomputed tour cost (vns.c:78-86).
int tspb200_vns_kick(tspb200_ctx *ctx, int idx1, int idx2, int idx3, double *cost) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    const int n = ctx->n;
    if (idx1 > idx2) std::swap(idx1, idx2);
    if (idx1 > idx3) std::swap(idx1, idx3);
    if (idx2 > idx3) std::swap(idx2, idx3);
    if (idx1 < 0 || idx3 >= n || idx2 - idx1 < 2 || idx3 - idx2 < 2)
        return fail(ctx, TSPB200_E_ARG, "kick indices must be distinct, non-adjacent tour indices in [0, n) (reference vns.c:25-31)");
    CK(cudaSetDevice(ctx->device));
    int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) path = 1;
    InstDev I = inst_for_path(ctx, path);
    SCRATCH(d_scr, float4 *, 3, sizeof(float4) * (size_t)n);
    CK(launch_vns_kick(I, ctx->tour, idx1, idx2, idx3, d_scr, ctx->stream));
    ctx->fi_cursor_stale = true;  // the next alg_2opt starts a fresh sweep on the kicked tour
    ctx->node_dirty = true;       // ... and rebuilds its node-space tables from the kicked records
    ctx->tour_changed = true;
    if (cost) return tspb200_tour_cost(ctx, cost);
    return TSPB200_OK;
}

// reference tabu() src/tabusearch.c:188-320 with the tabu list resident in HBM.
int tspb200_tabu_begin(tspb200_ctx *ctx) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    const int n = ctx->n;
    if (n > 46340) return fail(ctx, TSPB200_E_UNSUPPORTED, "tabu list index overflows int for n=%d (reference limit)", n);
    CK(cudaSetDevice(ctx->device));
    const long long len = (long long)n * (n - 1) / 2;
    if (ctx->skip_cap < len || !ctx->d_zl_count) {
        cudaFree(ctx->d_skip); cudaFree(ctx->d_zl); cudaFree(ctx->d_zl_count);
        ctx->d_skip = nullptr; ctx->d_zl = nullptr; ctx->d_zl_count = nullptr;
        ctx->skip_cap = 0;
        ctx->zl_cap = len < (1ll << 22) ? len : (1ll << 22);
        CK(cudaMalloc(&ctx->d_skip, sizeof(int) * (size_t)(len > 0 ? len : 1)));
        CK(cudaMalloc(&ctx->d_zl, sizeof(long long) * (size_t)(ctx->zl_cap > 0 ? ctx->zl_cap : 1)));
        CK(cudaMalloc(&ctx->d_zl_count, sizeof(unsigned long long)));
        ctx->skip_cap = len;
    }
    CK(cudaMemsetAsync(ctx->d_skip, 0, sizeof(int) * (size_t)(len > 0 ? len : 1), ctx->stream));  // CALLOC, tabusearch.c:196
    CK(cudaMemsetAsync(ctx->d_zl_count, 0, sizeof(unsigned long long), ctx->stream));
    ctx->tabu_session = true;
    return TSPB200_OK;
}

// alg_2opt_tabu(inst, tabu_edge, prev, iter, tenure) on the resident tour and the resident list (tabusearch.c:238)
int tspb200_tabu_run(tspb200_ctx *ctx, int iter, int tenure, int64_t max_passes, tspb200_stats *st) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->tabu_session) return fail(ctx, TSPB200_E_STATE, "no tabu session (tspb200_tabu_begin)");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    const long long keep = ctx->zl_cap;
    ctx->zl_cap = 0;  // the list never leaves the device: nothing to replay on a host copy
    ctx->tabu_on = true;
    ctx->tabu_iter = iter;
    ctx->tabu_tenure = tenure;
    ctx->tour_changed = true;  // a new call is a new search: whatever ended the previous one does not hold for this iter/tenure
    int rc = tspb200_bi_run(ctx, max_passes, st);
    ctx->tabu_on = false;
    ctx->zl_cap = keep;
    if (rc) return rc;
    if (st) {
        double cost = 0;
        rc = tspb200_tour_cost(ctx, &cost);  // tabusearch.c:168-172
        if (rc) return rc;
        st->cost = cost;
    }
    return TSPB200_OK;
}

// The random kick of tabusearch.c:262-309: `pairs` = count candidate (a, b) node pairs in the order the caller drew them;
// the first one that passes the reference's tests is applied as a 2-opt move and its two removed edges become tabu.
// *accepted = its index, or -1 when every candidate was rejected (draw more and call again).
int tspb200_tabu_kick(tspb200_ctx *ctx, const int32_t *pairs, int count, int iter, int tenure, int *accepted) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->tabu_session) return fail(ctx, TSPB200_E_STATE, "no tabu session (tspb200_tabu_begin)");
    if (!ctx->has_tour) return fail(ctx, TSPB200_E_STATE, "no tour uploaded");
    if (!pairs || count < 1 || !accepted) return fail(ctx, TSPB200_E_ARG, "bad arguments");
    CK(cudaSetDevice(ctx->device));
    int path = ctx->d_mat ? 2 : 1;
    InstDev I = inst_for_path(ctx, path);
    SCRATCH(d_pairs, int *, 9, sizeof(int) * 2 * (size_t)count + sizeof(int));
    int *d_acc = d_pairs + 2 * (size_t)count;
    CK(cudaMemcpyAsync(d_pairs, pairs, sizeof(int) * 2 * (size_t)count, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_tabu_kick_select(ctx->tour, ctx->d_skip, d_pairs, count, iter, tenure, d_acc, ctx->stream));
    CK(launch_apply_move(I, ctx->tour, ctx->num_sms, 0, 0, false, false, 0, ctx->stream));
    int acc = -1;
    CK(cudaMemcpyAsync(&acc, d_acc, sizeof acc, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (acc == -2) return fail(ctx, TSPB200_E_ARG, "kick candidate out of range");
    *accepted = acc;
    if (acc >= 0) {
        ctx->node_dirty = true;
        ctx->fi_cursor_stale = true;
        ctx->tour_changed = true;
    }
    return TSPB200_OK;
}

int tspb200_tabu_end(tspb200_ctx *ctx, int32_t *skip_out) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!ctx->tabu_session) return fail(ctx, TSPB200_E_STATE, "no tabu session");
    CK(cudaSetDevice(ctx->device));
    if (skip_out) {
        const long long len = (long long)ctx->n * (ctx->n - 1) / 2;
        CK(cudaMemcpyAsync(skip_out, ctx->d_skip, sizeof(int) * (size_t)len, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    ctx->tabu_session = false;
    return TSPB200_OK;
}

// ---- resident population (reference HEU_Genetic, src/genetic.c): tours stay in HBM as successor arrays --------------
static int pop_slots_to_device(tspb200_ctx *ctx, const int32_t *slots, int count, int **d_slots) {
    *d_slots = nullptr;
    if (!slots) return TSPB200_OK;
    for (int k = 0; k < count; ++k)
        if (slots[k] < 0 || slots[k] >= ctx->pop_count) return fail(ctx, TSPB200_E_ARG, "population slot %d out of range", slots[k]);
    SCRATCH(d, int *, 10, sizeof(int) * (size_t)count);
    CK(cudaMemcpyAsync(d, slots, sizeof(int) * (size_t)count, cudaMemcpyHostToDevice, ctx->stream));
    *d_slots = d;
    return TSPB200_OK;
}

// Creates (count tours, slots == NULL) or updates (the listed slots) the resident population.  as_order != 0: tours are
// chromosomes (visiting orders, genetic.c:22-26), converted on the device (from_chromosome_to_edges, genetic.c:34-44).
int tspb200_population_upload(tspb200_ctx *ctx, const int32_t *tours, const int32_t *slots, int count, int as_order) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->n < 1) return fail(ctx, TSPB200_E_STATE, "no instance");
    if (!tours || count < 1) return fail(ctx, TSPB200_E_ARG, "bad arguments");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    if (!slots) {
        if (count > ctx->pop_cap || ctx->pop_n != n) {
            CK(cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->d_pop);
            ctx->d_pop = nullptr;
            ctx->pop_cap = 0;
            CK(cudaMalloc(&ctx->d_pop, sizeof(int) * (size_t)n * (size_t)count));
            ctx->pop_cap = count;
            ctx->pop_n = n;
        }
        ctx->pop_count = count;
    } else if (ctx->pop_count < 1 || ctx->pop_n != n) {
        return fail(ctx, TSPB200_E_STATE, "no resident population");
    }
    int *d_slots = nullptr;
    int rc = pop_slots_to_device(ctx, slots, count, &d_slots);
    if (rc) return rc;
    SCRATCH(d_stage, int *, 0, sizeof(int) * (size_t)n * (size_t)count);
    CK(cudaMemcpyAsync(d_stage, tours, sizeof(int) * (size_t)n * (size_t)count, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_population_store(d_stage, ctx->d_pop, d_slots, n, count, as_order, ctx->stream));
    return TSPB200_OK;
}

int tspb200_population_download(tspb200_ctx *ctx, int32_t *tours, const int32_t *slots, int count, int as_order) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->pop_count < 1 || ctx->pop_n != ctx->n) return fail(ctx, TSPB200_E_STATE, "no resident population");
    if (!tours || count < 1 || (!slots && count > ctx->pop_count)) return fail(ctx, TSPB200_E_ARG, "bad arguments");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n;
    int *d_slots = nullptr;
    int rc = pop_slots_to_device(ctx, slots, count, &d_slots);
    if (rc) return rc;
    SCRATCH(d_stage, int *, 0, sizeof(int) * (size_t)n * (size_t)count);
    CK(launch_population_fetch(ctx->d_pop, d_slots, d_stage, n, count, as_order, ctx->stream));
    CK(cudaMemcpyAsync(tours, d_stage, sizeof(int) * (size_t)n * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSPB200_OK;
}

// fitness() (genetic.c:51-60) of the listed slots (all when slots == NULL): only `count` doubles cross the bus
int tspb200_population_costs(tspb200_ctx *ctx, const int32_t *slots, int count, double *out) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->pop_count < 1 || ctx->pop_n != ctx->n) return fail(ctx, TSPB200_E_STATE, "no resident population");
    if (!out || count < 1 || (!slots && count > ctx->pop_count)) return fail(ctx, TSPB200_E_ARG, "bad arguments");
    CK(cudaSetDevice(ctx->device));
    int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) path = 1;
    InstDev I = inst_for_path(ctx, path == 2 ? 2 : 1);
    int *d_slots = nullptr;
    int rc = pop_slots_to_device(ctx, slots, count, &d_slots);
    if (rc) return rc;
    SCRATCH(d_o, long long *, 15, sizeof(long long) * (size_t)count);
    CK(launch_tour_cost(I, ctx->d_pop, d_slots, 0, d_o, count, ctx->stream));
    std::vector<long long> h((size_t)count);
    CK(cudaMemcpyAsync(h.data(), d_o, sizeof(long long) * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < count; ++b) out[b] = (double)h[(size_t)b];
    return TSPB200_OK;
}

// alg_2opt (mode FI, genetic.c:435) / best improvement on the listed slots in place.  obj (count doubles, may be NULL):
// FI adds the applied deltas to the incoming values, BI overwrites them with the recomputed costs.
int tspb200_population_two_opt(tspb200_ctx *ctx, int mode, const int32_t *slots, int count, double *obj, tspb200_stats *st) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (ctx->pop_count < 1 || ctx->pop_n != ctx->n) return fail(ctx, TSPB200_E_STATE, "no resident population");
    if (mode != TSPB200_FI && mode != TSPB200_BI) return fail(ctx, TSPB200_E_ARG, "mode must be TSPB200_FI or TSPB200_BI");
    if (count < 1 || (!slots && count > ctx->pop_count)) return fail(ctx, TSPB200_E_ARG, "bad arguments");
    if (!(ctx->dist_bound < 16777216.0)) return fail(ctx, TSPB200_E_UNSUPPORTED, "distances >= 2^24 are not supported by the 2-opt kernels");
    CK(cudaSetDevice(ctx->device));
    const int path = select_path(ctx);
    if (path == 2 && !ctx->d_mat) return fail(ctx, TSPB200_E_STATE, "matrix path selected but no resident matrix");
    InstDev I = inst_for_path(ctx, path);
    int *d_slots = nullptr;
    int rc = pop_slots_to_device(ctx, slots, count, &d_slots);
    if (rc) return rc;
    SCRATCH(d_delta, long long *, 1, sizeof(long long) * (size_t)count);
    SCRATCH(d_cnt, long long *, 2, sizeof(long long) * 4 * (size_t)count);
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    CK(cudaMemsetAsync(d_delta, 0, sizeof(long long) * (size_t)count, ctx->stream));
    CK(cudaMemsetAsync(d_cnt, 0, sizeof(long long) * 4 * (size_t)count, ctx->stream));
    int launched = 0;
    cudaError_t le = cudaErrorNotSupported;
    if (mode == TSPB200_BI && path == 0 && ctx->opt_batch_kernel != 1)
        le = launch_two_opt_batch_bi_pos(I, ctx->d_pop, d_slots, d_delta, d_cnt, count, ctx->num_sms, ctx->stream, &launched, nullptr, 0);
    if (le == cudaErrorNotSupported)
        le = launch_two_opt_batch(I, mode, ctx->d_pop, d_slots, d_delta, d_cnt, count, ctx->num_sms, ctx->stream, &launched, nullptr, 0);
    if (le == cudaErrorInvalidValue)
        return fail(ctx, TSPB200_E_UNSUPPORTED, "resident populations use the one-block kernels: n=%d does not fit (use tspb200_two_opt_batch)", ctx->n);
    if (le != cudaSuccess) return fail(ctx, TSPB200_E_CUDA, "batched 2-opt launch failed: %s", cudaGetErrorString(le));
    std::vector<long long> h_delta((size_t)count), h_cnt((size_t)count * 4);
    CK(cudaMemcpyAsync(h_delta.data(), d_delta, sizeof(long long) * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(h_cnt.data(), d_cnt, sizeof(long long) * 4 * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    tspb200_stats local;
    memset(&local, 0, sizeof local);
    for (int b = 0; b < count; ++b) {
        if (h_cnt[4 * (size_t)b + 3]) return fail(ctx, TSPB200_E_DEVICE_CHECK, "population slot %d does not hold a single cycle", slots ? slots[b] : b);
        local.moves += h_cnt[4 * (size_t)b + 0];
        local.passes += h_cnt[4 * (size_t)b + 1];
        local.evals += h_cnt[4 * (size_t)b + 2];
        if (mode == TSPB200_FI) local.obj_delta += h_delta[(size_t)b];
        if (obj) {
            if (mode == TSPB200_BI) obj[b] = (double)h_delta[(size_t)b];
            else obj[b] += (double)h_delta[(size_t)b];
        }
    }
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    local.gpu_ms = ms;
    local.launches = launched;
    local.path = path;
    local.status = TSPB200_LOCAL_OPTIMUM;
    if (st) *st = local;
    return TSPB200_OK;
}

// ---- multi-GPU -------------------------------------------------------------------------------------------
int tspb200_comm_unique_id(void *id128) {
    std::string err;
    if (!id128) return TSPB200_E_ARG;
    if (!g_nccl.load(err)) { fprintf(stderr, "tspb200: %s\n", err.c_str()); return TSPB200_E_NCCL; }
    nccl_unique_id id;
    if (g_nccl.GetUniqueId(&id) != 0) return TSPB200_E_NCCL;
    memcpy(id128, &id, sizeof id);
    return TSPB200_OK;
}

int tspb200_comm_init(tspb200_ctx *ctx, const void *id128, int rank, int world) {
    if (!ctx || !ctx->stream) return fail(ctx, TSPB200_E_CUDA, "context has no CUDA device");
    if (!id128 || world < 1 || rank < 0 || rank >= world) return fail(ctx, TSPB200_E_ARG, "bad communicator arguments");
    std::string err;
    if (!g_nccl.load(err)) return fail(ctx, TSPB200_E_NCCL, "%s", err.c_str());
    CK(cudaSetDevice(ctx->device));
    nccl_unique_id id;
    memcpy(&id, id128, sizeof id);
    if (ctx->comm) { g_nccl.CommDestroy(ctx->comm); ctx->comm = nullptr; }
    free_xchg(ctx);
    ctx->xchg_note.clear();
    ctx->rank = 0;
    ctx->world = 1;
    ctx->has_tour = false;  // tile plan depends on the world size

    // ---- everything local is allocated BEFORE the first collective: a rank must never leave a collective half-way
    // because of a local failure (its peers would block in it); local failures are folded into the agreed `ok` flag ----
    int ok = (world <= XCHG_MAX_WORLD && g_nccl.AllGather) ? 1 : 0;
    if (!ok) ctx->xchg_note = "peer exchange needs world <= 16 and ncclAllGather";
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof mine);
    char *d_h = nullptr;
    std::vector<cudaIpcMemHandle_t> all((size_t)world);
    bool local_ok = cudaMalloc(&d_h, sizeof(cudaIpcMemHandle_t) * (size_t)(world + 1)) == cudaSuccess &&
                    cudaMalloc(&ctx->d_stop, sizeof(int)) == cudaSuccess &&
                    cudaMalloc(&ctx->d_slots, sizeof(XchgMem)) == cudaSuccess &&
                    cudaMalloc(&ctx->d_epoch, 2 * sizeof(unsigned)) == cudaSuccess &&
                    cudaMemsetAsync(ctx->d_slots, 0, sizeof(XchgMem), ctx->stream) == cudaSuccess &&
                    cudaMemsetAsync(ctx->d_epoch, 0, 2 * sizeof(unsigned), ctx->stream) == cudaSuccess;
    if (!local_ok) {
        cudaGetLastError();
        cudaFree(d_h);
        free_xchg(ctx);
        return fail(ctx, TSPB200_E_CUDA, "cannot allocate the communicator's device buffers");
    }
    if (ok && cudaIpcGetMemHandle(&mine, ctx->d_slots) != cudaSuccess) {
        cudaGetLastError();
        ok = 0;
        ctx->xchg_note = "cudaIpcGetMemHandle failed";
    }
    auto bail = [&](int code, const char *what, int nr) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(d_h);
        free_xchg(ctx);
        if (ctx->comm) { g_nccl.CommDestroy(ctx->comm); ctx->comm = nullptr; }
        return fail(ctx, code, "%s failed: %s", what, nr >= 0 && g_nccl.GetErrorString ? g_nccl.GetErrorString(nr) : "CUDA error");
    };
    int nr = g_nccl.CommInitRank(&ctx->comm, world, id, rank);
    if (nr != 0) return bail(TSPB200_E_NCCL, "ncclCommInitRank", nr);

    // ---- peer-memory exchange: every rank maps every other rank's slot array (CUDA IPC -> NVLink P2P).  The handles
    // travel through the communicator; the all-gather also orders every rank's memset of its slots before any peer can
    // write to them ----
    if (cudaMemcpyAsync(d_h, &mine, sizeof mine, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) ok = 0;
    if (g_nccl.AllGather) {
        nr = g_nccl.AllGather(d_h, d_h + sizeof(cudaIpcMemHandle_t), sizeof(cudaIpcMemHandle_t), NCCL_CHAR, ctx->comm, ctx->stream);
        if (nr != 0) return bail(TSPB200_E_NCCL, "ncclAllGather", nr);
        if (cudaMemcpyAsync(all.data(), d_h + sizeof(cudaIpcMemHandle_t), sizeof(cudaIpcMemHandle_t) * (size_t)world,
                            cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) ok = 0;
    }
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) ok = 0;
    if (ok) {
        for (int r = 0; r < world && ok; ++r) {
            if (r == rank) { ctx->xchg.peer[r] = ctx->d_slots; continue; }
            void *p = nullptr;
            if (cudaIpcOpenMemHandle(&p, all[(size_t)r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                ok = 0;
                ctx->xchg_note = "cudaIpcOpenMemHandle failed (no peer access between the ranks' devices?)";
                break;
            }
            ctx->peer_mapped[r] = p;
            ctx->xchg.peer[r] = reinterpret_cast<XchgMem *>(p);
        }
    }
    // all ranks must agree: one failure anywhere -> everybody uses the NCCL allreduce
    int *d_ok = reinterpret_cast<int *>(d_h);
    int all_ok = 0;
    cudaMemcpyAsync(d_ok, &ok, sizeof ok, cudaMemcpyHostToDevice, ctx->stream);
    nr = g_nccl.AllReduce(d_ok, d_ok, 1, NCCL_INT32, NCCL_MIN, ctx->comm, ctx->stream);
    if (nr != 0) return bail(TSPB200_E_NCCL, "ncclAllReduce", nr);
    cudaMemcpyAsync(&all_ok, d_ok, sizeof all_ok, cudaMemcpyDeviceToHost, ctx->stream);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return bail(TSPB200_E_CUDA, "cudaStreamSynchronize", -1);
    cudaFree(d_h);
    ctx->xchg.epoch = ctx->d_epoch;
    ctx->xchg.align_epoch = ctx->d_epoch + 1;
    ctx->xchg.enabled = all_ok ? 1 : 0;
    if (!all_ok && ctx->xchg_note.empty()) ctx->xchg_note = "a peer rank could not map the exchange slots";
    ctx->rank = rank;   // only now: a failed init leaves the context single-GPU
    ctx->world = world;
    return TSPB200_OK;
}

int tspb200_comm_destroy(tspb200_ctx *ctx) {
    if (!ctx) return TSPB200_E_ARG;
    if (ctx->stream) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); }
    free_xchg(ctx);
    if (ctx->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->comm);
    ctx->comm = nullptr;
    ctx->rank = 0;
    ctx->world = 1;
    ctx->has_tour = false;
    return TSPB200_OK;
}

}  // extern "C"
