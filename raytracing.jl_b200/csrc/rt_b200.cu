// rt_b200.cu -- the C ABI of include/rt_b200.h on top of the sm_100a kernels (mesh_dev.cuh, trace.cuh,
// walk.cuh, scan.cuh).  Build (see __graft_entry__.build):
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -shared -Xcompiler -fPIC
// -fmad=false is REQUIRED for bit-parity with the reference's IEEE arithmetic (Julia never fuses a*b+c).
#include "../../include/rt_b200.h"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "scan.cuh"
#include "sweep.cuh"
#include "eval3.cuh"
#include "march.cuh"
#include "trace.cuh"
#include "locate.cuh"

using namespace rt;

// ---- minimal NCCL surface, resolved with dlopen so the library has no link-time dependency ------------
typedef struct ncclComm *ncclComm_t;
typedef struct {
    char internal[128];
} ncclUniqueId;
typedef int ncclResult_t;
enum { ncclFloat64 = 8, ncclSum = 0 };
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
};

struct rt_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    cudaEvent_t pev[6][2] = {};   // per phase: start/stop events; elapsed times are read lazily (rt_phase_ms, rt_stats)
    bool pev_dirty[6] = {false, false, false, false, false, false};
    cudaEvent_t tev[2] = {nullptr, nullptr};

    // mesh
    bool has_mesh = false;
    bool mixed = false;  // 3- and 4-node cells (SURVEY 8f-4): literal walk only
    DevMesh m{};
    DevBuf b_cell_ptrs;
    DevBuf b_xy, b_cell_nodes, b_nc_ptrs, b_nc_data, b_nbr, b_cells, b_edges, b_qual, b_bdist, b_sc, b_grid_ptrs,
        b_grid_nodes, b_twin, b_he, b_node_reach;
    double clear_tiny = -1.0;
    double smax = 0.0, lmax = 0.0;

    // per-angle tables
    int n2 = 0;
    DevBuf b_ang_d, b_ang_i;  // doubles: phi,sin,cos,tan,dxe,dye,delta ; int64: nx,ny,base(n2+1)
    std::vector<long long> h_base;
    std::vector<double> h_phi;
    bool has_delta = false;

    // tracks of the shard
    bool traced = false;
    long long uid_begin = 1, n_shard = 0;
    TrackSoA t{};
    DevBuf b_trk_d, b_trk_i, b_trk_l, b_trk_c;
    DevBuf b_err;

    // segmentation
    bool segmented = false;
    DevBuf b_count, b_status, b_offsets, b_tile, b_vol, b_voln;
    // control words of one rt_segmentize in ONE 64-byte block: reset with one copy, read back with one copy (every separate
    // memset / memcpy is a few microseconds of an otherwise idle GPU at the start and at the end of a call)
    //   [0..3] counters (fast transitions, literal iterations, nn / knn queries)  [4] first bad track  [5] verify flag | guard flag << 32
    DevBuf b_ctrl;
    std::vector<double> h_delta;       // delta_eff as last uploaded (the upload is skipped when the caller passes the same values)
    DevBuf b_layout;  // per-track chunk layout (walk.cuh ChunkLayout)
    DevBuf b_nch, b_blk_chunks, b_unit_base, b_unit_block, b_ch_i, b_ch_d;  // chunk plan (walk.cuh ChunkPlan)
    DevBuf b_order, b_okeys, b_ohist;  // spatial execution order of the units
    DevBuf b_omega, b_sigma, b_tau;  // sweep-facing exports (sweep.cuh)
    DevBuf b_area, b_factor;         // exact element volumes, volume-correction factors (sweep.cuh)
    DevBuf b_exc;                    // compact download: exception list (sweep.cuh k_p_exceptions)
    cudaStream_t aux_stream = nullptr;  // ... built on a side stream while the columns cross the bus
    cudaEvent_t ev_aux = nullptr;
    bool area_valid = false;
    long long *h_pin = nullptr;  // page-locked scratch for the small device->host read-backs of rt_segmentize (16 words)
    DevBuf b_cell_bin;
    DevBuf b_scratch, b_gcounts, b_gcursor;  // rt_mesh_upload staging (kept between uploads)
    DevBuf b_tsum;    // self-verifying pipelines: per-track length sums
    DevBuf b_pool, b_pool_next, b_pool_cursor;  // single-walk pipeline: record blocks (walk.cuh kRecBlock), chain, cursor
    int count_batches = 0;             // single-walk pipeline: how many uid batches the count walk needed (info)
    // The chunk plan (k_plan_chunks .. k_unit_scatter) depends on the tracks, the mesh density and the chunk options only: it is
    // kept between calls and rebuilt when one of them changes (plan_key), so the steady-state segmentize! needs neither its
    // kernels nor the host round trip that sizes its arrays.
    unsigned long long trace_gen = 0;  // bumped by rt_trace / rt_mesh_upload
    struct PlanKey {
        unsigned long long gen = ~0ULL;
        double chunk_len = -1.0;
        int band = -1, order_grid = -1;
        double band_min = -1.0, band_div = -1.0;
        long long n = -1;
        bool operator==(const PlanKey &o) const { return gen == o.gen && chunk_len == o.chunk_len && band == o.band && order_grid == o.order_grid && n == o.n &&
                   band_min == o.band_min && band_div == o.band_div; }
    } plan_key;
    bool plan_has_order = false;
    int opt_debug_clear_pool = 0;      // test hook (initcheck): zero the record pool before every walk, so that the evaluation's speculative
                                       // load of a chunk's first records (issued before its count is known) never reads unwritten words
    double opt_band_cost = 28.0;       // shard planning: cost of one boundary-band cell in fast transitions (measured: cfg4 on 8 GPUs)
    int opt_plan_cache = 1;            // 0: rebuild the chunk plan in every call (test knob)
    // Optimistic evaluation: when the previous call's Segment columns are still allocated, the evaluation is launched right behind
    // the walk WITHOUT reading the segment total back first; the thread of the scan that writes the total compares it (and the
    // record pool's cursor) with the capacities on the device (scan.cuh ScanGuard) and cancels the evaluation if they do not fit --
    // the host learns it with the final read-back of the call and repeats the call on the careful path.
    int opt_optimistic = 1;
    bool skip_optimistic_once = false;
    int optimistic_cancels = 0;        // calls whose optimistic evaluation the device-side guard cancelled (info)
    unsigned long long fit_gen = ~0ULL;  // trace generation whose previous call fitted the Segment columns and the pool in ONE batch

    int opt_band_chunks = 1;           // shorter chunks for tracks that run along the bounding box (walk.cuh k_plan_chunks)
    // ... when that stretch is longer than opt_band_min regular chunks, into chunks opt_band_div times shorter.  Both are relative to
    // the regular chunk: where tracks are plentiful (cfg4, cfg5: a chunk is a whole track) fine chunks would only multiply the
    // chunk slots.  0.0625 x 208 = 13 crossings: on cfg3 the two angles next to each axis qualify; with the 0.25 of round 1 the
    // second one did not below 128-segment chunks and its band stretches were the walk's longest serial chains
    // (profiles/r2_chunk_band.txt: walk phase 0.70 -> 0.62 ms)
    double opt_band_min = 0.0625;
    double opt_band_div = 8.0;
    long long opt_pool_slots = 0;      // test hook: at most this many chunk slots per count batch (0: as many as fit)
    double opt_pool_extra = 1.25;      // spare pool blocks, as a multiple of (expected segments / kRecBlock)
    int opt_pipeline = 3;              // 3: single walk (k_march counts AND records, k_eval3 evaluates) [default]; 0: hybrid (k_march without records
                                       // counts, geometric fill walk), 1: sequential (walk.cuh only); 3 falls back to 0 (pool exhausted) or 1, 0 falls back to 1
    int verify_fallbacks = 0;
    int opt_debug_verify_fail = 0;     // test hook: make the verification of the two-stage pipeline fail
    double tau_ms = 0.0;
    cudaEvent_t ev2[2] = {nullptr, nullptr};  // kernel stopwatch of the synchronous exports (rt_optical_lengths, rt_find_elements)
    DevBuf b_loc_xy, b_loc_elem, b_loc_knn;   // rt_find_elements: points, element ids, k-nearest branch counter
    double locate_knn = 0.0, locate_ms = 0.0;
    int opt_order_grid = 32;           // G x G tiles (0: identity order)
    const int *order_eval = nullptr;   // execution order of the evaluation (plain Morton order)
    int opt_order_classes = 3;         // duration bins of the walk's launch order, longest units first (walk.cuh k_unit_keys); 0: spatial order
                                       // only.  Three bins: finer ones cost more in locality than they gain in balance (profiles/r2_walk_order.txt)
    int n_sm = 148;
    long long n_units = 0;
    double opt_chunk_segments = 208.0;              // minimum expected segments per chunk (profiles/r2_chunk_band.txt)
    double opt_target_walkers = 148.0 * 2048.0 * 4.0;  // chunks are sized so that about this many walkers exist
    double sum_len = 0.0;              // total track length of the shard
    double edge_sum = 0.0, area = 0.0;  // mesh density scalars (chunk sizing)
    long long total_segments = 0;
    long long cap_cfg = 0;  // user limit on resident segments (0 = as many as fit)
    long long cap = 0;      // allocated
    DevBuf b_seg_d, b_seg_e;
    double *s_px = nullptr, *s_py = nullptr, *s_qx = nullptr, *s_qy = nullptr, *s_len = nullptr;
    int *s_elem = nullptr;
    long long res_trk_begin = 0, res_trk_end = 0, res_off_base = 0, res_nseg = 0;  // resident batch (shard-local)
    bool vol_valid = false;
    // Inside the batch callback of rt_segmentize the resident batch is valid although the call has not finished (`segmented` is
    // false until it returns); the volume correction then uses the normalised volumes of the PREVIOUS call, which the current one
    // overwrites only after its last callback (k_normalise, rt_volumes).
    bool in_batch_cb = false;
    bool prev_vol_valid = false;  // the call before the current rt_segmentize left volumes in b_voln

    double phase_ms[6] = {0, 0, 0, 0, 0, 0};
    double stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};

    // NCCL
    NcclApi nccl;
    ncclComm_t comm = nullptr;
    int n_ranks = 1, rank = 0;
    // The all-reduce of the volumes runs on its own stream, so that the next segmentize! of the caller overlaps with it: the
    // per-element sums are accumulated alternately in b_vol / b_vol_alt, the collective reads the one just filled.
    cudaStream_t coll_stream = nullptr;
    DevBuf b_vol_alt;
    int vol_cur = 0;
    double *vol_acc = nullptr;                              // accumulation buffer of the current / last rt_segmentize
    cudaEvent_t ev_fill_done = nullptr;                     // ctx->stream: the sums are complete
    cudaEvent_t ev_vol_free[2] = {nullptr, nullptr};        // coll_stream: the collective has consumed buffer i (and b_voln is ready)
    bool ev_vol_used[2] = {false, false};
    bool voln_done = false;                                 // b_voln already holds the normalised volumes of the last rt_segmentize (no communicator)
    int voln_ready = -1;                                    // index of the event that marks b_voln complete (-1: main stream)
    long long collectives = 0;                              // ncclAllReduce calls issued by rt_volumes, failed-rank joins included (info)
};

static inline unsigned long long *d_counters(rt_ctx *c) { return (unsigned long long *)c->b_ctrl.p; }
static inline unsigned long long *d_bad(rt_ctx *c) { return (unsigned long long *)c->b_ctrl.p + 4; }
static inline int *d_verify(rt_ctx *c) { return (int *)((unsigned long long *)c->b_ctrl.p + 5); }
static inline int *d_guard(rt_ctx *c) { return (int *)((unsigned long long *)c->b_ctrl.p + 5) + 1; }
constexpr int kPinWords = 32, kPinCtrlInit = 16, kPinCtrl = 24;  // page-locked scratch: template and read-back of the control block

static int fail(rt_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    return code;
}

#define CK(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess)                                                                                \
            return fail(ctx, RT_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,              \
                        cudaGetErrorString(e_));                                                              \
    } while (0)

static cudaError_t ensure(DevBuf &b, size_t bytes) {
    if (bytes <= b.bytes && b.p) return cudaSuccess;
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
    cudaError_t e = cudaMalloc(&b.p, bytes ? bytes : 1);
    if (e == cudaSuccess) b.bytes = bytes;
    return e;
}
static void release(DevBuf &b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
}

static inline unsigned blocks_for(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

template <typename Tin, typename Tout>
static cudaError_t exclusive_scan(rt_ctx *ctx, const Tin *in, Tout *out, long long n, Tout carry = Tout(0), ScanGuard guard = ScanGuard{}) {
    long long n_tiles = (n + kScanTile - 1) / kScanTile;
    cudaError_t e = ensure(ctx->b_tile, sizeof(Tout) * (size_t)n_tiles);
    if (e != cudaSuccess) return e;
    Tout *tiles = (Tout *)ctx->b_tile.p;
    k_scan_tile_sums<Tin, Tout><<<(unsigned)n_tiles, kScanThreads, 0, ctx->stream>>>(in, tiles, n);
    k_scan_tile_offsets<Tout><<<1, kScanThreads, 0, ctx->stream>>>(tiles, n_tiles);
    k_scan_apply<Tin, Tout><<<(unsigned)n_tiles, kScanThreads, 0, ctx->stream>>>(in, out, tiles, n, carry, guard);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------
extern "C" const char *rt_version(void) { return "rt_b200 0.1 (sm_100a, fp64, fmad=false)"; }

extern "C" int rt_create(rt_ctx **out, int device) {
    if (!out) return RT_ERR_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) return RT_ERR_CUDA;  // no CPU fallback
    rt_ctx *ctx = new rt_ctx();
    ctx->device = device;
    cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, device);
    if (ctx->n_sm <= 0) ctx->n_sm = 148;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->tev[0]) != cudaSuccess || cudaEventCreate(&ctx->tev[1]) != cudaSuccess ||
        cudaEventCreate(&ctx->ev2[0]) != cudaSuccess || cudaEventCreate(&ctx->ev2[1]) != cudaSuccess) {
        delete ctx;
        return RT_ERR_CUDA;
    }
    if (cudaHostAlloc((void **)&ctx->h_pin, kPinWords * sizeof(long long), cudaHostAllocDefault) != cudaSuccess) {
        delete ctx;
        return RT_ERR_NOMEM;
    }
    for (int ph = 0; ph < 6; ++ph)
        for (int q = 0; q < 2; ++q)
            if (cudaEventCreate(&ctx->pev[ph][q]) != cudaSuccess) {
                delete ctx;
                return RT_ERR_CUDA;
            }
    *out = ctx;
    return RT_OK;
}

extern "C" void rt_destroy(rt_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->coll_stream) cudaStreamSynchronize(ctx->coll_stream);  // a collective may still be in flight
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->comm && ctx->nccl.CommDestroy) ctx->nccl.CommDestroy(ctx->comm);
    DevBuf *all[] = {&ctx->b_cell_ptrs, &ctx->b_xy,      &ctx->b_cell_nodes, &ctx->b_nc_ptrs,  &ctx->b_nc_data, &ctx->b_nbr,     &ctx->b_cells,
                     &ctx->b_edges,   &ctx->b_qual,       &ctx->b_bdist,    &ctx->b_sc,      &ctx->b_grid_ptrs, &ctx->b_grid_nodes,
                     &ctx->b_ang_d,   &ctx->b_ang_i,      &ctx->b_trk_d,    &ctx->b_trk_i,   &ctx->b_trk_l,   &ctx->b_trk_c,
                     &ctx->b_err,     &ctx->b_count,      &ctx->b_status,   &ctx->b_offsets, &ctx->b_tile,    &ctx->b_vol,
                     &ctx->b_voln,    &ctx->b_ctrl,       &ctx->b_seg_d,   &ctx->b_seg_e,
                     &ctx->b_twin,    &ctx->b_he,         &ctx->b_node_reach,
                     &ctx->b_nch,     &ctx->b_blk_chunks, &ctx->b_unit_base, &ctx->b_unit_block, &ctx->b_ch_i, &ctx->b_ch_d,
                     &ctx->b_order,   &ctx->b_okeys,      &ctx->b_ohist,     &ctx->b_tsum,
                     &ctx->b_scratch, &ctx->b_gcounts,   &ctx->b_gcursor,   &ctx->b_cell_bin,
                     &ctx->b_omega,   &ctx->b_sigma,     &ctx->b_tau,
                     &ctx->b_pool,    &ctx->b_pool_next, &ctx->b_pool_cursor,
                     &ctx->b_area,    &ctx->b_factor,    &ctx->b_layout,    &ctx->b_vol_alt,  &ctx->b_exc,
                     &ctx->b_loc_xy,  &ctx->b_loc_elem,  &ctx->b_loc_knn};
    for (DevBuf *b : all) release(*b);
    for (int ph = 0; ph < 6; ++ph)
        for (int q = 0; q < 2; ++q)
            if (ctx->pev[ph][q]) cudaEventDestroy(ctx->pev[ph][q]);
    if (ctx->coll_stream) {
        cudaStreamSynchronize(ctx->coll_stream);
        cudaStreamDestroy(ctx->coll_stream);
    }
    for (cudaEvent_t e : {ctx->ev_fill_done, ctx->ev_vol_free[0], ctx->ev_vol_free[1]})
        if (e) cudaEventDestroy(e);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->ev_aux) cudaEventDestroy(ctx->ev_aux);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    delete ctx;
}

extern "C" const char *rt_last_error(const rt_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int rt_host_alloc(void **ptr, size_t bytes) {
    return cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault) == cudaSuccess ? RT_OK : RT_ERR_NOMEM;
}
extern "C" int rt_host_free(void *ptr) { return cudaFreeHost(ptr) == cudaSuccess ? RT_OK : RT_ERR_CUDA; }

// phase stopwatches: events only, no host synchronisation on the hot path
static void tic(rt_ctx *ctx, int ph) { cudaEventRecord(ctx->pev[ph][0], ctx->stream); }
static void toc(rt_ctx *ctx, int ph) {
    cudaEventRecord(ctx->pev[ph][1], ctx->stream);
    ctx->pev_dirty[ph] = true;
}
static void collect_phase_ms(rt_ctx *ctx) {
    for (int ph = 0; ph < 6; ++ph) {
        if (!ctx->pev_dirty[ph]) continue;
        float ms = 0.f;
        if (cudaEventSynchronize(ctx->pev[ph][1]) == cudaSuccess && cudaEventElapsedTime(&ms, ctx->pev[ph][0], ctx->pev[ph][1]) == cudaSuccess)
            ctx->phase_ms[ph] = (double)ms;
        ctx->pev_dirty[ph] = false;
    }
}

// ------------------------------------------------------------------------------------------------------
// mesh
// ------------------------------------------------------------------------------------------------------
extern "C" int rt_mesh_upload(rt_ctx *ctx, int32_t n_nodes, const double *xy, int32_t n_cells, const int32_t *cell_ptrs,
                              const int32_t *cell_data, const int32_t *node_cell_ptrs, const int32_t *node_cell_data,
                              const double bb_min[2], const double bb_max[2]) {
    if (!ctx) return RT_ERR_ARG;
    if (n_nodes < 3 || n_cells < 1 || !xy || !cell_ptrs || !cell_data || (!node_cell_ptrs != !node_cell_data) || (!bb_min != !bb_max))
        return fail(ctx, RT_ERR_ARG, "rt_mesh_upload: null or empty mesh arrays");
    const bool dev_nc = node_cell_ptrs == nullptr;  // build the vertex -> cells table on the device
    const bool dev_bb = bb_min == nullptr;          // reduce the bounding box on the device
    bool mixed = false;
    for (int32_t c = 0; c < n_cells; ++c) {
        const int nn = cell_ptrs[c + 1] - cell_ptrs[c];
        if (nn == 4)
            mixed = true;
        else if (nn != 3)
            return fail(ctx, RT_ERR_ARG, "rt_mesh_upload: cell %d has %d nodes (triangles and quadrilaterals only)", c + 1, nn);
    }
    if (mixed && dev_nc) return fail(ctx, RT_ERR_ARG, "rt_mesh_upload: a mesh with quadrilaterals needs the vertex -> cells table from the caller");
    const size_t n_cd = (size_t)(cell_ptrs[n_cells] - 1);  // entries of the cell -> nodes table
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    tic(ctx, 0);
    size_t n_nc = dev_nc ? (size_t)3 * n_cells : (size_t)(node_cell_ptrs[n_nodes] - 1);
    CK(ensure(ctx->b_xy, sizeof(double2) * (size_t)n_nodes));
    CK(ensure(ctx->b_cell_nodes, sizeof(int) * n_cd));
    CK(ensure(ctx->b_nc_ptrs, sizeof(int) * ((size_t)n_nodes + 1)));
    CK(ensure(ctx->b_nc_data, sizeof(int) * n_nc));
    CK(ensure(ctx->b_nbr, sizeof(int) * 3 * (size_t)n_cells));
    CK(ensure(ctx->b_cells, sizeof(CellRec) * (size_t)n_cells));
    CK(ensure(ctx->b_edges, sizeof(EdgeRec) * 3 * (size_t)n_cells));
    CK(ensure(ctx->b_qual, sizeof(float) * (size_t)n_cells));
    CK(ensure(ctx->b_bdist, sizeof(float) * (size_t)n_cells));
    CK(ensure(ctx->b_sc, sizeof(MeshScalars)));
    // stage the 1-based tables through a (persistent) scratch buffer and convert on the device; no host synchronisation here:
    // the three tables use disjoint scratch regions
    const size_t tab_n[3] = {n_cd, dev_nc ? 0 : (size_t)n_nodes + 1, dev_nc ? 0 : n_nc};
    CK(ensure(ctx->b_scratch, sizeof(int32_t) * (tab_n[0] + tab_n[1] + tab_n[2])));
    CK(cudaMemcpyAsync(ctx->b_xy.p, xy, sizeof(double) * 2 * (size_t)n_nodes, cudaMemcpyHostToDevice, st));
    const int32_t *tab_src[3] = {cell_data, node_cell_ptrs, node_cell_data};
    void *tab_dst[3] = {ctx->b_cell_nodes.p, ctx->b_nc_ptrs.p, ctx->b_nc_data.p};
    size_t tab_off = 0;
    for (int q = 0; q < 3; ++q) {
        if (tab_n[q] == 0) continue;
        int32_t *stage = (int32_t *)ctx->b_scratch.p + tab_off;
        CK(cudaMemcpyAsync(stage, tab_src[q], sizeof(int32_t) * tab_n[q], cudaMemcpyHostToDevice, st));
        k_to_zero_based<<<blocks_for((long long)tab_n[q], 256), 256, 0, st>>>(stage, (int *)tab_dst[q], (long long)tab_n[q]);
        tab_off += tab_n[q];
    }

    if (mixed) {  // the CSR offsets of the cell -> nodes table (triangle meshes do not need them: 3 * cell)
        DevBuf stage;
        CK(ensure(stage, sizeof(int32_t) * ((size_t)n_cells + 1)));
        CK(ensure(ctx->b_cell_ptrs, sizeof(int) * ((size_t)n_cells + 1)));
        CK(cudaMemcpyAsync(stage.p, cell_ptrs, sizeof(int32_t) * ((size_t)n_cells + 1), cudaMemcpyHostToDevice, st));
        k_to_zero_based<<<blocks_for((long long)n_cells + 1, 256), 256, 0, st>>>((const int32_t *)stage.p, (int *)ctx->b_cell_ptrs.p, (long long)n_cells + 1);
        CK(cudaStreamSynchronize(st));
        release(stage);
    }
    if (dev_nc) {  // count -> scan -> fill -> sort (ascending cell id around every node, src/mesh.jl:27)
        DevBuf deg, cur;
        CK(ensure(deg, sizeof(int) * (size_t)n_nodes));
        CK(ensure(cur, sizeof(int) * (size_t)n_nodes));
        CK(cudaMemsetAsync(deg.p, 0, sizeof(int) * (size_t)n_nodes, st));
        CK(cudaMemsetAsync(cur.p, 0, sizeof(int) * (size_t)n_nodes, st));
        k_nc_count<<<blocks_for(3LL * n_cells, 256), 256, 0, st>>>(n_cells, (const int *)ctx->b_cell_nodes.p, (int *)deg.p);
        CK((exclusive_scan<int, int>(ctx, (const int *)deg.p, (int *)ctx->b_nc_ptrs.p, (long long)n_nodes)));
        k_nc_fill<<<blocks_for(3LL * n_cells, 256), 256, 0, st>>>(n_cells, (const int *)ctx->b_cell_nodes.p, (const int *)ctx->b_nc_ptrs.p,
                                                                   (int *)cur.p, (int *)ctx->b_nc_data.p);
        k_nc_sort<<<blocks_for(n_nodes, 256), 256, 0, st>>>(n_nodes, (const int *)ctx->b_nc_ptrs.p, (int *)ctx->b_nc_data.p);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(st));
        release(deg);
        release(cur);
    }
    double bbv[4];
    if (dev_bb) {
        DevBuf dbb;
        CK(ensure(dbb, sizeof(double) * 4));
        const double init[4] = {INFINITY, INFINITY, -INFINITY, -INFINITY};
        CK(cudaMemcpyAsync(dbb.p, init, sizeof(init), cudaMemcpyHostToDevice, st));
        k_bbox<<<std::min(1024u, blocks_for(n_nodes, 256)), 256, 0, st>>>((const double2 *)ctx->b_xy.p, n_nodes, (double *)dbb.p);
        CK(cudaMemcpyAsync(bbv, dbb.p, sizeof(bbv), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        release(dbb);
        bb_min = bbv;
        bb_max = bbv + 2;
    }
    DevMesh &m = ctx->m;
    m.n_nodes = n_nodes;
    m.n_cells = n_cells;
    m.xy = (const double2 *)ctx->b_xy.p;
    m.cell_nodes = (const int *)ctx->b_cell_nodes.p;
    m.cell_ptrs = mixed ? (const int *)ctx->b_cell_ptrs.p : nullptr;
    m.nc_ptrs = (const int *)ctx->b_nc_ptrs.p;
    m.nc_data = (const int *)ctx->b_nc_data.p;
    m.cells = (const CellRec *)ctx->b_cells.p;
    m.edges = (const EdgeRec *)ctx->b_edges.p;
    m.bbmin[0] = bb_min[0];
    m.bbmin[1] = bb_min[1];
    m.bbmax[0] = bb_max[0];
    m.bbmax[1] = bb_max[1];
    // node grid: ~2 nodes per bin
    double w = bb_max[0] - bb_min[0], h = bb_max[1] - bb_min[1];
    if (!(w > 0 && h > 0)) return fail(ctx, RT_ERR_ARG, "rt_mesh_upload: empty bounding box");
    double gh = sqrt(w * h / ((double)n_nodes / 2.0));
    m.gx = std::max(1, (int)ceil(w / gh));
    m.gy = std::max(1, (int)ceil(h / gh));
    m.g0x = bb_min[0];
    m.g0y = bb_min[1];
    m.gh = gh;
    m.ginv = 1.0 / gh;
    size_t n_bins = (size_t)m.gx * m.gy;
    CK(ensure(ctx->b_grid_ptrs, sizeof(int) * (n_bins + 1)));
    CK(ensure(ctx->b_grid_nodes, sizeof(int) * (size_t)n_nodes));
    m.grid_ptrs = (const int *)ctx->b_grid_ptrs.p;
    m.grid_nodes = (const int *)ctx->b_grid_nodes.p;

    CK(cudaMemsetAsync(ctx->b_sc.p, 0, sizeof(MeshScalars), st));
    if (mixed) {
        // only the literal walk runs on a mixed mesh: no neighbour table, no cell / edge / half-edge records -- just the density
        // scalars that size the buffers
        k_mesh_scalars_generic<<<blocks_for(n_cells, 128), 128, 0, st>>>(n_cells, m.cell_ptrs, m.cell_nodes, m.xy, (MeshScalars *)ctx->b_sc.p);
        m.cells = nullptr;
        m.edges = nullptr;
        m.twin = nullptr;
        m.he = nullptr;
    } else {
    k_neighbours<<<blocks_for(3LL * n_cells, 256), 256, 0, st>>>(n_cells, m.cell_nodes, m.nc_ptrs, m.nc_data, (int *)ctx->b_nbr.p);
    k_cell_records<<<blocks_for(n_cells, 128), 128, 0, st>>>(m, (const int *)ctx->b_nbr.p, (CellRec *)ctx->b_cells.p,
                                                             (EdgeRec *)ctx->b_edges.p, (float *)ctx->b_qual.p,
                                                             (float *)ctx->b_bdist.p, (MeshScalars *)ctx->b_sc.p);
    CK(ensure(ctx->b_twin, sizeof(int) * 3 * (size_t)n_cells));
    CK(ensure(ctx->b_he, sizeof(HalfEdge) * 3 * (size_t)n_cells));
    CK(ensure(ctx->b_node_reach, sizeof(float) * (size_t)n_nodes));
    m.twin = (const int *)ctx->b_twin.p;
    m.he = (const HalfEdge *)ctx->b_he.p;
    k_twins<<<blocks_for(3LL * n_cells, 256), 256, 0, st>>>(n_cells, m.cell_nodes, (const int *)ctx->b_nbr.p, (int *)ctx->b_twin.p);
    k_half_edges<<<blocks_for(3LL * n_cells, 128), 128, 0, st>>>(m, (const CellRec *)ctx->b_cells.p, m.twin, (HalfEdge *)ctx->b_he.p);
    CK(cudaMemsetAsync(ctx->b_node_reach.p, 0, sizeof(float) * (size_t)n_nodes, st));
    k_node_reach<<<blocks_for(n_cells, 128), 128, 0, st>>>(m, (const CellRec *)ctx->b_cells.p, (const MeshScalars *)ctx->b_sc.p,
                                                           (float *)ctx->b_node_reach.p);
    }
    // grid: count -> scan -> fill
    DevBuf &counts = ctx->b_gcounts, &cursor = ctx->b_gcursor;
    CK(ensure(counts, sizeof(int) * n_bins));
    CK(ensure(cursor, sizeof(int) * n_bins));
    CK(cudaMemsetAsync(counts.p, 0, sizeof(int) * n_bins, st));
    CK(cudaMemsetAsync(cursor.p, 0, sizeof(int) * n_bins, st));
    k_grid_count<<<blocks_for(n_nodes, 256), 256, 0, st>>>(m, (int *)counts.p);
    CK((exclusive_scan<int, int>(ctx, (const int *)counts.p, (int *)ctx->b_grid_ptrs.p, (long long)n_bins)));
    k_grid_fill<<<blocks_for(n_nodes, 256), 256, 0, st>>>(m, m.grid_ptrs, (int *)cursor.p, (int *)ctx->b_grid_nodes.p);
    m.cell_bin = nullptr;
    if (!mixed) {  // entry points of the seed location walk (k_seed)
        CK(ensure(ctx->b_cell_bin, sizeof(int) * n_bins));
        CK(cudaMemsetAsync(ctx->b_cell_bin.p, 0xff, sizeof(int) * n_bins, st));
        k_cell_bins<<<blocks_for(n_cells, 256), 256, 0, st>>>(m, (const CellRec *)ctx->b_cells.p, (int *)ctx->b_cell_bin.p);
        m.cell_bin = (const int *)ctx->b_cell_bin.p;
    }
    CK(cudaGetLastError());
    MeshScalars sc;
    CK(cudaMemcpyAsync(&sc, ctx->b_sc.p, sizeof(sc), cudaMemcpyDeviceToHost, st));
    toc(ctx, 0);
    CK(cudaStreamSynchronize(st));
    ctx->smax = sc.smax;
    ctx->lmax = sc.lmax;
    ctx->edge_sum = sc.edge_sum;
    ctx->area = sc.area;
    ctx->clear_tiny = -1.0;
    ctx->trace_gen++;
    ctx->mixed = mixed;
    ctx->has_mesh = true;
    ctx->area_valid = false;
    ctx->traced = false;
    ctx->segmented = false;
    return RT_OK;
}

extern "C" int rt_mesh_bbox(rt_ctx *ctx, double bb_min[2], double bb_max[2]) {
    if (!ctx || !ctx->has_mesh || !bb_min || !bb_max) return fail(ctx, RT_ERR_ARG, "rt_mesh_bbox: no mesh");
    for (int q = 0; q < 2; ++q) {
        bb_min[q] = ctx->m.bbmin[q];
        bb_max[q] = ctx->m.bbmax[q];
    }
    return RT_OK;
}

extern "C" int rt_mesh_node_cells(rt_ctx *ctx, int32_t *node_cell_ptrs, int32_t *node_cell_data) {
    if (!ctx || !ctx->has_mesh) return fail(ctx, RT_ERR_ARG, "rt_mesh_node_cells: no mesh");
    CK(cudaSetDevice(ctx->device));
    const size_t nn = (size_t)ctx->m.n_nodes;
    std::vector<int> ptrs(nn + 1);
    CK(cudaMemcpy(ptrs.data(), ctx->b_nc_ptrs.p, sizeof(int) * (nn + 1), cudaMemcpyDeviceToHost));
    if (node_cell_ptrs)
        for (size_t i = 0; i <= nn; ++i) node_cell_ptrs[i] = ptrs[i] + 1;  // 1-based like Gridap's Table
    if (node_cell_data) {
        const size_t n = (size_t)ptrs[nn];
        CK(cudaMemcpy(node_cell_data, ctx->b_nc_data.p, sizeof(int) * n, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < n; ++i) node_cell_data[i] += 1;
    }
    return RT_OK;
}

extern "C" int rt_mesh_neighbours(rt_ctx *ctx, int32_t *cell_nbr) {
    if (!ctx || !ctx->has_mesh || !cell_nbr) return fail(ctx, RT_ERR_ARG, "rt_mesh_neighbours: no mesh");
    if (ctx->mixed) return fail(ctx, RT_ERR_ARG, "rt_mesh_neighbours: triangle meshes only");
    CK(cudaSetDevice(ctx->device));
    size_t n = 3 * (size_t)ctx->m.n_cells;
    CK(cudaMemcpy(cell_nbr, ctx->b_nbr.p, sizeof(int) * n, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; ++i) cell_nbr[i] += 1;  // 1-based, 0 = boundary
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------------
// trace!
// ------------------------------------------------------------------------------------------------------
static int upload_angle_tables(rt_ctx *ctx, int32_t n2, const int64_t *nx, const int64_t *ny, const double *phi,
                               const double *sin_phi, const double *cos_phi, const double *tan_phi, const double *dxe,
                               const double *dye) {
    if (n2 < 2 || (n2 % 2) != 0) return fail(ctx, RT_ERR_ARG, "n_azim_2 must be a positive even number");
    std::vector<double> hd(7 * (size_t)n2, 0.0);
    const double *cols[6] = {phi, sin_phi, cos_phi, tan_phi, dxe, dye};
    for (int q = 0; q < 6; ++q)
        if (cols[q]) memcpy(&hd[(size_t)q * n2], cols[q], sizeof(double) * n2);
    std::vector<long long> hi(3 * (size_t)n2 + 1, 0);
    ctx->h_base.assign((size_t)n2 + 1, 0);
    for (int i = 0; i < n2; ++i) {
        if (nx[i] < 1 || ny[i] < 1) return fail(ctx, RT_ERR_ARG, "n_tracks_x/y must be >= 1");
        hi[i] = nx[i];
        hi[n2 + i] = ny[i];
        ctx->h_base[i + 1] = ctx->h_base[i] + nx[i] + ny[i];
    }
    for (int i = 0; i <= n2; ++i) hi[2 * (size_t)n2 + i] = ctx->h_base[i];
    CK(ensure(ctx->b_ang_d, sizeof(double) * hd.size()));
    CK(ensure(ctx->b_ang_i, sizeof(long long) * hi.size()));
    CK(cudaMemcpyAsync(ctx->b_ang_d.p, hd.data(), sizeof(double) * hd.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->b_ang_i.p, hi.data(), sizeof(long long) * hi.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->n2 = n2;
    ctx->h_phi.assign(phi, phi + n2);
    ctx->has_delta = false;
    return RT_OK;
}

static void fill_trace_params(rt_ctx *ctx, TraceParams &P, const int32_t bcs[4]) {
    int n2 = ctx->n2;
    const double *d = (const double *)ctx->b_ang_d.p;
    const long long *li = (const long long *)ctx->b_ang_i.p;
    P.n2 = n2;
    P.n4 = n2 / 2;
    P.nx = li;
    P.ny = li + n2;
    P.base = li + 2 * n2;
    P.phi = d;
    P.tanp = d + 3 * n2;
    P.dxe = d + 4 * n2;
    P.dye = d + 5 * n2;
    for (int q = 0; q < 4; ++q) P.bcs[q] = bcs ? bcs[q] : 0;
    for (int q = 0; q < 2; ++q) {
        P.bbmin[q] = ctx->m.bbmin[q];
        P.bbmax[q] = ctx->m.bbmax[q];
    }
    P.len_only = nullptr;
    P.cost_w = 0.0;
    P.err = (unsigned long long *)ctx->b_err.p;
}

extern "C" int rt_trace(rt_ctx *ctx, int32_t n_azim_2, const int64_t *n_tracks_x, const int64_t *n_tracks_y, const double *phi,
                        const double *sin_phi, const double *cos_phi, const double *tan_phi, const double *dx_eff,
                        const double *dy_eff, const int32_t bcs[4], int64_t uid_begin, int64_t uid_end) {
    if (!ctx || !ctx->has_mesh) return fail(ctx, RT_ERR_ARG, "rt_trace: upload a mesh first");
    if (!n_tracks_x || !n_tracks_y || !phi || !sin_phi || !cos_phi || !tan_phi || !dx_eff || !dy_eff || !bcs)
        return fail(ctx, RT_ERR_ARG, "rt_trace: null table");
    for (int q = 0; q < 4; ++q)
        if (bcs[q] < 0 || bcs[q] > 2) return fail(ctx, RT_ERR_ARG, "rt_trace: bad boundary condition code");
    CK(cudaSetDevice(ctx->device));
    int rc = upload_angle_tables(ctx, n_azim_2, n_tracks_x, n_tracks_y, phi, sin_phi, cos_phi, tan_phi, dx_eff, dy_eff);
    if (rc) return rc;
    long long n_total = ctx->h_base[n_azim_2];
    if (uid_begin < 1 || uid_end > n_total + 1 || uid_end < uid_begin)
        return fail(ctx, RT_ERR_ARG, "rt_trace: uid range [%lld,%lld) outside [1,%lld]", (long long)uid_begin, (long long)uid_end,
                    n_total + 1);
    long long n = uid_end - uid_begin;
    ctx->uid_begin = uid_begin;
    ctx->n_shard = n;
    ctx->traced = false;
    ctx->segmented = false;
    size_t nn = (size_t)std::max<long long>(n, 1);
    CK(ensure(ctx->b_trk_d, sizeof(double) * 8 * nn));
    CK(ensure(ctx->b_trk_i, sizeof(int) * nn));
    CK(ensure(ctx->b_trk_l, sizeof(long long) * 3 * nn));
    CK(ensure(ctx->b_trk_c, 4 * nn));
    CK(ensure(ctx->b_err, sizeof(unsigned long long)));
    double *d = (double *)ctx->b_trk_d.p;
    TrackSoA &t = ctx->t;
    t.px = d;
    t.py = d + nn;
    t.qx = d + 2 * nn;
    t.qy = d + 3 * nn;
    t.len = d + 4 * nn;
    t.a = d + 5 * nn;
    t.b = d + 6 * nn;
    t.c = d + 7 * nn;
    t.azim = (int *)ctx->b_trk_i.p;
    long long *l = (long long *)ctx->b_trk_l.p;
    t.track_idx = l;
    t.next_fwd = l + nn;
    t.next_bwd = l + 2 * nn;
    signed char *c = (signed char *)ctx->b_trk_c.p;
    t.bc_fwd = c;
    t.bc_bwd = c + nn;
    t.dir_fwd = c + 2 * nn;
    t.dir_bwd = c + 3 * nn;
    CK(cudaMemsetAsync(ctx->b_err.p, 0xff, sizeof(unsigned long long), ctx->stream));
    TraceParams P;
    fill_trace_params(ctx, P, bcs);
    P.uid_begin = uid_begin;
    P.n = n;
    P.t = t;
    tic(ctx, 1);
    DevBuf dsum;
    CK(ensure(dsum, sizeof(double)));
    CK(cudaMemsetAsync(dsum.p, 0, sizeof(double), ctx->stream));
    if (n > 0) {
        k_trace<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(P);
        k_sum_double<<<std::min(1024u, blocks_for(n, 256)), 256, 0, ctx->stream>>>(t.len, n, (double *)dsum.p);
    }
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&ctx->sum_len, dsum.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    unsigned long long err = 0;
    CK(cudaMemcpyAsync(&err, ctx->b_err.p, sizeof(err), cudaMemcpyDeviceToHost, ctx->stream));
    toc(ctx, 1);
    CK(cudaStreamSynchronize(ctx->stream));
    release(dsum);
    if (err != ~0ULL) {
        long long uid = (long long)(err >> 4);
        int code = (int)(err & 15);
        if (code == TRACE_E_NO_EXIT) return fail(ctx, RT_ERR_NO_EXIT, "DomainError: could not found track exit point. (uid %lld)", uid);
        if (code == TRACE_E_NOT_ON_BOUNDARY) return fail(ctx, RT_ERR_NOT_ON_BOUNDARY, "Point do not lie in the boundary. (uid %lld)", uid);
        return fail(ctx, RT_ERR_BC_MISMATCH, "Boundaries do not match! (uid %lld)", uid);
    }
    ctx->traced = true;
    ctx->trace_gen++;
    return RT_OK;
}

template <typename T>
static int fetch_col(rt_ctx *ctx, const T *dev, std::vector<T> &host, size_t n) {
    host.resize(n);
    CK(cudaMemcpy(host.data(), dev, sizeof(T) * n, cudaMemcpyDeviceToHost));
    return RT_OK;
}

extern "C" int rt_tracks_download(rt_ctx *ctx, int64_t *azim_idx, int64_t *track_idx, double *p, double *q, double *phi,
                                  double *len, double *abc, int8_t *bc_fwd, int8_t *bc_bwd, int8_t *dir_fwd, int8_t *dir_bwd,
                                  int64_t *next_fwd_uid, int64_t *next_bwd_uid) {
    if (!ctx || !ctx->traced) return fail(ctx, RT_ERR_NOT_TRACED, "rt_tracks_download: call rt_trace first");
    CK(cudaSetDevice(ctx->device));
    size_t n = (size_t)ctx->n_shard;
    if (n == 0) return RT_OK;
    const TrackSoA &t = ctx->t;
    std::vector<double> c0, c1, c2;
    int rc;
    if (p) {
        if ((rc = fetch_col(ctx, t.px, c0, n)) || (rc = fetch_col(ctx, t.py, c1, n))) return rc;
        for (size_t i = 0; i < n; ++i) {
            p[2 * i] = c0[i];
            p[2 * i + 1] = c1[i];
        }
    }
    if (q) {
        if ((rc = fetch_col(ctx, t.qx, c0, n)) || (rc = fetch_col(ctx, t.qy, c1, n))) return rc;
        for (size_t i = 0; i < n; ++i) {
            q[2 * i] = c0[i];
            q[2 * i + 1] = c1[i];
        }
    }
    if (abc) {
        if ((rc = fetch_col(ctx, t.a, c0, n)) || (rc = fetch_col(ctx, t.b, c1, n)) || (rc = fetch_col(ctx, t.c, c2, n))) return rc;
        for (size_t i = 0; i < n; ++i) {
            abc[3 * i] = c0[i];
            abc[3 * i + 1] = c1[i];
            abc[3 * i + 2] = c2[i];
        }
    }
    if (len) CK(cudaMemcpy(len, t.len, sizeof(double) * n, cudaMemcpyDeviceToHost));
    if (azim_idx || phi) {
        std::vector<int> az;
        if ((rc = fetch_col(ctx, t.azim, az, n))) return rc;
        for (size_t i = 0; i < n; ++i) {
            if (azim_idx) azim_idx[i] = az[i] + 1;
            if (phi) phi[i] = ctx->h_phi[az[i]];
        }
    }
    if (track_idx) CK(cudaMemcpy(track_idx, t.track_idx, sizeof(long long) * n, cudaMemcpyDeviceToHost));
    if (next_fwd_uid) CK(cudaMemcpy(next_fwd_uid, t.next_fwd, sizeof(long long) * n, cudaMemcpyDeviceToHost));
    if (next_bwd_uid) CK(cudaMemcpy(next_bwd_uid, t.next_bwd, sizeof(long long) * n, cudaMemcpyDeviceToHost));
    if (bc_fwd) CK(cudaMemcpy(bc_fwd, t.bc_fwd, n, cudaMemcpyDeviceToHost));
    if (bc_bwd) CK(cudaMemcpy(bc_bwd, t.bc_bwd, n, cudaMemcpyDeviceToHost));
    if (dir_fwd) CK(cudaMemcpy(dir_fwd, t.dir_fwd, n, cudaMemcpyDeviceToHost));
    if (dir_bwd) CK(cudaMemcpy(dir_bwd, t.dir_bwd, n, cudaMemcpyDeviceToHost));
    return RT_OK;
}

__global__ void k_split_points(const double *cum /* n+1 */, long long n, int n_parts, long long *bounds) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n_parts) return;
    if (r == 0) {
        bounds[0] = 1;
        return;
    }
    if (r == n_parts) {
        bounds[r] = n + 1;
        return;
    }
    double target = cum[n] * ((double)r / (double)n_parts);
    long long lo = 0, hi = n;  // first index with cum[idx] >= target
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if (cum[mid] < target)
            lo = mid + 1;
        else
            hi = mid;
    }
    bounds[r] = lo + 1;
}

extern "C" int rt_plan_shards(rt_ctx *ctx, int32_t n_azim_2, const int64_t *n_tracks_x, const int64_t *n_tracks_y,
                              const double *phi, const double *tan_phi, const double *dx_eff, const double *dy_eff,
                              int32_t n_parts, int64_t *bounds) {
    if (!ctx || !ctx->has_mesh) return fail(ctx, RT_ERR_ARG, "rt_plan_shards: upload a mesh first");
    if (n_parts < 1 || !bounds || !phi || !tan_phi || !dx_eff || !dy_eff) return fail(ctx, RT_ERR_ARG, "rt_plan_shards: bad arguments");
    CK(cudaSetDevice(ctx->device));
    int rc = upload_angle_tables(ctx, n_azim_2, n_tracks_x, n_tracks_y, phi, nullptr, nullptr, tan_phi, dx_eff, dy_eff);
    if (rc) return rc;
    ctx->traced = false;
    ctx->segmented = false;
    long long n = ctx->h_base[n_azim_2];
    DevBuf lens, cum, db;
    CK(ensure(lens, sizeof(double) * (size_t)n));
    CK(ensure(cum, sizeof(double) * ((size_t)n + 1)));
    CK(ensure(db, sizeof(long long) * ((size_t)n_parts + 1)));
    CK(ensure(ctx->b_err, sizeof(unsigned long long)));
    TraceParams P;
    fill_trace_params(ctx, P, nullptr);
    P.uid_begin = 1;
    P.n = n;
    P.t = TrackSoA{};
    P.len_only = (double *)lens.p;
    P.cost_w = ctx->edge_sum > 0.0 ? ctx->opt_band_cost * (kPi * ctx->area / ctx->edge_sum) : 0.0;  // band_cost segments, as a length
    k_trace<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(P);
    CK((exclusive_scan<double, double>(ctx, (const double *)lens.p, (double *)cum.p, n)));
    k_split_points<<<blocks_for(n_parts + 1, 64), 64, 0, ctx->stream>>>((const double *)cum.p, n, n_parts, (long long *)db.p);
    CK(cudaGetLastError());
    std::vector<long long> hb((size_t)n_parts + 1);
    CK(cudaMemcpyAsync(hb.data(), db.p, sizeof(long long) * hb.size(), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int r = 0; r <= n_parts; ++r) bounds[r] = hb[r];
    for (int r = 1; r <= n_parts; ++r) bounds[r] = std::max(bounds[r], bounds[r - 1]);
    release(lens);
    release(cum);
    release(db);
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------------
// segmentize!
// ------------------------------------------------------------------------------------------------------
__global__ void k_first_bad(const int *status, long long n, unsigned long long *out) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n && status[i] != 0) atomicMin(out, ((unsigned long long)i << 4) | (unsigned long long)(status[i] & 15));
}

__global__ void k_normalise(const double *in, double *out, int n, double denom) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] / denom;  // volumes ./= n_azim_2, src/trackgenerator.jl:386
}

extern "C" int rt_set_segment_capacity(rt_ctx *ctx, int64_t max_segments_resident) {
    if (!ctx || max_segments_resident < 0) return RT_ERR_ARG;
    ctx->cap_cfg = max_segments_resident;
    return RT_OK;
}

static int ensure_segment_buffers(rt_ctx *ctx, long long want) {
    if (want <= ctx->cap && ctx->b_seg_d.p) return RT_OK;
    release(ctx->b_seg_d);
    release(ctx->b_seg_e);
    ctx->cap = 0;
    size_t n = ((size_t)std::max<long long>(want, 1) + 15) & ~(size_t)15;  // every SoA column stays 32-byte aligned
    CK(ensure(ctx->b_seg_d, sizeof(double) * 5 * n));
    CK(ensure(ctx->b_seg_e, sizeof(int) * n));
    double *d = (double *)ctx->b_seg_d.p;
    ctx->s_px = d;
    ctx->s_py = d + n;
    ctx->s_qx = d + 2 * n;
    ctx->s_qy = d + 3 * n;
    ctx->s_len = d + 4 * n;
    ctx->s_elem = (int *)ctx->b_seg_e.p;
    ctx->cap = (long long)n;
    return RT_OK;
}

// fast transitions only accept chords that are certainly not dropped by isapprox(p, q) (src/track.jl:156) and long enough for
// the re-location argument (DESIGN.md): l > l_min = max(8*tiny, rtol * largest possible |point|)
static double lmin_of(const DevMesh &m, double tiny_step) {
    double nb = hypot(fmax(fabs(m.bbmin[0]), fabs(m.bbmax[0])), fmax(fabs(m.bbmin[1]), fabs(m.bbmax[1])));
    return fmax(8.0 * tiny_step, kRtol * nb * (1.0 + 1e-6) + 1e-300);
}

// ---- one attempt of rt_segmentize ----------------------------------------------------------------------------------------------
// What rt_segmentize does after an attempt
enum class Next {
    Done,
    RepeatCareful,  // the optimistic evaluation was cancelled on the device: the same pipeline, sized from the walk's result
    Sequential,     // count and fill disagreed / a geometric fast-path condition failed: fall back to mode 1
    Hybrid,         // the single walk's record pool ran out: fall back to mode 0
};

// One execution of a pipeline: its inputs, and what its driver leaves to the common tail of segmentize_attempt
struct Attempt {
    double rtol;
    bool want_vol;
    rt_batch_cb cb;
    void *cb_user;
    int index;                    // rt_batch::attempt
    Next next = Next::Done;
    double launches = 0;          // kernel launches (stats[0] when this attempt is the final one)
    bool first_bad_scan = false;  // k_first_bad finds the first failing track (the single walk's k_track_status reports it itself)
    bool defer_verify = false;    // the verification flag arrives with the final control read-back
    bool defer_total = false;     // ... and so do the segment total and the guard of the optimistic evaluation
};

static double crossings_per_length(const rt_ctx *ctx) { return ctx->edge_sum / (kPi * ctx->area); }

static void set_resident(rt_ctx *ctx, long long trk_begin, long long trk_end, long long off_base, long long nseg) {
    ctx->res_trk_begin = trk_begin;
    ctx->res_trk_end = trk_end;
    ctx->res_off_base = off_base;
    ctx->res_nseg = nseg;
}

// the Segment columns the fill / evaluation writes
static void bind_columns(const rt_ctx *ctx, WalkParams &P) {
    P.opx = ctx->s_px;
    P.opy = ctx->s_py;
    P.oqx = ctx->s_qx;
    P.oqy = ctx->s_qy;
    P.olen = ctx->s_len;
    P.oelem = ctx->s_elem;
}

// Segment columns sized from free memory (0.92 x free / 44 bytes per segment, counting the columns held now) for `want` segments
// (already limited by the capacity option): one batch takes what it needs if that fits, a walk in several batches everything that
// fits.  *cap: the capacity to cut the batches with.
static int size_columns(rt_ctx *ctx, long long want, bool take_all, size_t free_b, long long *cap) {
    const long long fit = (long long)((double)(free_b + ctx->b_seg_d.bytes + ctx->b_seg_e.bytes) * 0.92 / 44.0);
    *cap = take_all ? fit : std::min(want, fit);
    if (ctx->cap_cfg > 0) *cap = std::min(*cap, (long long)ctx->cap_cfg);
    return ensure_segment_buffers(ctx, *cap);
}

// The next batch of tracks, from track b on, whose segments fit `cap` (h_off: host copy of the offsets of the tracks from b0 on):
// P takes its tracks, its offset base and the warp units of the 32-track blocks overlapping it, in identity order.
static int cut_batch(rt_ctx *ctx, WalkParams &P, const std::vector<long long> &h_off, long long b0,
                     const std::vector<long long> &h_unit_base, long long b, long long cap, long long *nseg) {
    const long long lim = h_off[(size_t)(b - b0)] + cap;  // largest e with off[e] - off[b] <= cap
    const long long e = b0 + (long long)(std::upper_bound(h_off.begin() + (b - b0), h_off.end(), lim) - h_off.begin()) - 1;
    if (e <= b) return fail(ctx, RT_ERR_NOMEM, "rt_segmentize: one track needs more than the segment capacity");
    P.trk_begin = b;
    P.trk_end = e;
    P.offset_base = h_off[(size_t)(b - b0)];
    P.ch.order = nullptr;
    P.unit_begin = h_unit_base[(size_t)(b >> 5)];
    P.unit_end = h_unit_base[(size_t)((e - 1) >> 5) + 1];
    *nseg = h_off[(size_t)(e - b0)] - P.offset_base;
    return RT_OK;
}

// the reference's length check (src/track.jl:171-175) of the batch P describes, on the segment lengths it accumulated
static void launch_track_status(rt_ctx *ctx, const WalkParams &P, double rtol, const int *cancel, unsigned long long *bad) {
    if (P.trk_end <= P.trk_begin) return;
    EvalParams E{};
    E.t = ctx->t;
    E.offsets = P.offsets;
    E.trk_begin = P.trk_begin;
    E.trk_end = P.trk_end;
    E.offset_base = P.offset_base;
    E.olen = P.olen;
    E.status = P.status;
    E.tsum = P.tsum;
    E.rtol = rtol;
    E.cancel = cancel;
    E.bad = bad;
    k_track_status<<<blocks_for(P.trk_end - P.trk_begin, 128), 128, 0, ctx->stream>>>(E);
}

// waits for the batch and reads its verification flag
static int read_verify(rt_ctx *ctx, bool *failed) {
    ctx->h_pin[2] = 0;
    CK(cudaMemcpyAsync(&ctx->h_pin[2], d_verify(ctx), sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *failed = (int)ctx->h_pin[2] != 0;
    return RT_OK;
}

// the resident batch may be read: after a completed rt_segmentize, or from inside its batch callback
static bool resident_valid(const rt_ctx *ctx) { return ctx && (ctx->segmented || ctx->in_batch_cb); }

// the resident batch (rt_segments_device) to the caller's batch callback, if there is one
static int deliver_batch(rt_ctx *ctx, const Attempt &a) {
    if (!a.cb) return RT_OK;
    rt_batch bt;
    int rc = rt_segments_device(ctx, &bt);
    if (rc) return rc;
    bt.attempt = a.index;
    ctx->in_batch_cb = true;  // (the resident-batch calls accept the batch while the callback runs)
    const int stop = a.cb(&bt, a.cb_user);
    ctx->in_batch_cb = false;
    if (stop) return fail(ctx, RT_ERR_ARG, "rt_segmentize: batch callback asked to stop");
    return RT_OK;
}

// ---- chunk plan: cut tracks so that ~target_walkers independent walkers exist, >= chunk_segments segments each (n > 0) ----------
static int plan_chunks(rt_ctx *ctx, WalkParams &P, uint32_t flags, double *launches) {
    cudaStream_t st = ctx->stream;
    const long long n = ctx->n_shard;
    const DevMesh &m = ctx->m;
    const long long n_blocks = (n + 31) / 32;
    double rho = crossings_per_length(ctx);  // expected cell crossings per unit track length
    double est_total = ctx->sum_len * rho;
    double seg_target = fmax(ctx->opt_chunk_segments, est_total / ctx->opt_target_walkers);
    double chunk_len = (flags & RT_SEG_NO_CHUNKS) || !(rho > 0.0) ? INFINITY : seg_target / rho;
    rt_ctx::PlanKey key;
    key.gen = ctx->trace_gen;
    key.chunk_len = chunk_len;
    key.band = ctx->opt_band_chunks;
    key.band_min = ctx->opt_band_min;
    key.band_div = ctx->opt_band_div;
    key.order_grid = ctx->opt_order_grid + 1000 * ctx->opt_order_classes;
    key.n = n;
    const bool reuse = ctx->opt_plan_cache && key == ctx->plan_key && ctx->n_units > 0;
    ChunkPlan &ch = P.ch;
    if (!reuse) {
        ctx->plan_key = rt_ctx::PlanKey{};
        CK(ensure(ctx->b_nch, sizeof(int) * (size_t)n));
        CK(ensure(ctx->b_blk_chunks, sizeof(int) * (size_t)n_blocks));
        CK(ensure(ctx->b_unit_base, sizeof(long long) * ((size_t)n_blocks + 1)));
        PlanGeom pg{ctx->t.px, ctx->t.py, ctx->t.qx, ctx->t.qy, {m.bbmin[0], m.bbmin[1]}, {m.bbmax[0], m.bbmax[1]},
                    ctx->opt_band_chunks ? ctx->lmax : 0.0, ctx->opt_band_min * chunk_len, chunk_len / ctx->opt_band_div};
        CK(ensure(ctx->b_layout, sizeof(ChunkLayout) * (size_t)n));
        k_plan_chunks<<<blocks_for(n_blocks * 32, 128), 128, 0, st>>>(n, ctx->t.len, chunk_len, pg, (int *)ctx->b_nch.p,
                                                                     (ChunkLayout *)ctx->b_layout.p, (int *)ctx->b_blk_chunks.p);
        CK((exclusive_scan<int, long long>(ctx, (const int *)ctx->b_blk_chunks.p, (long long *)ctx->b_unit_base.p, n_blocks)));
        CK(cudaMemcpyAsync(&ctx->h_pin[0], (long long *)ctx->b_unit_base.p + n_blocks, sizeof(long long), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        ctx->n_units = ctx->h_pin[0];
        *launches += 5;
    }
    const long long n_units = ctx->n_units;
    size_t nc = (size_t)n_units * 32;
    CK(ensure(ctx->b_unit_block, sizeof(int) * (size_t)n_units));
    CK(ensure(ctx->b_ch_i, sizeof(int) * 5 * nc));
    CK(ensure(ctx->b_ch_d, sizeof(double) * 3 * nc));
    if (!reuse) {  // (slots no track owns are never written by the kernels, but the evaluation requests them before it knows that)
        CK(cudaMemsetAsync(ctx->b_ch_i.p, 0, sizeof(int) * 5 * nc, st));
        CK(cudaMemsetAsync(ctx->b_ch_d.p, 0, sizeof(double) * 3 * nc, st));
    }
    if (!reuse)
        k_fill_units<<<blocks_for(n_blocks, 128), 128, 0, st>>>(n_blocks, (const long long *)ctx->b_unit_base.p,
                                                                 (int *)ctx->b_unit_block.p);
    ch.nch = (int *)ctx->b_nch.p;
    ch.layout = (const ChunkLayout *)ctx->b_layout.p;
    ch.unit_block = (int *)ctx->b_unit_block.p;
    ch.unit_base = (long long *)ctx->b_unit_base.p;
    ch.n_units = n_units;
    int *ci = (int *)ctx->b_ch_i.p;
    ch.seed_cell = ci;
    ch.seed_kexit = ci + nc;
    ch.count = ci + 2 * nc;
    ch.endcode = ci + 3 * nc;
    ch.prefix = ci + 4 * nc;
    double *cd = (double *)ctx->b_ch_d.p;
    ch.seed_qx = cd;
    ch.seed_qy = cd + nc;
    ch.sum = cd + 2 * nc;
    P.unit_begin = 0;
    P.unit_end = n_units;
    // ---- execution orders (counting sorts of the units): the walk launches the units that start a track first and the short
    // ones last, in Morton order of their tiles inside each class; the evaluation, whose warps live for microseconds, keeps
    // the plain Morton order
    ch.order = nullptr;
    ctx->order_eval = nullptr;
    if (ctx->opt_order_grid > 0 && n_units < (1LL << 31)) {
        const bool two = ctx->opt_order_classes != 0;
        if (!reuse) {
            int G = std::min(ctx->opt_order_grid, 256);
            int gp = 1;
            while (gp < G) gp <<= 1;
            CK(ensure(ctx->b_order, sizeof(int) * (size_t)n_units * (two ? 2 : 1)));
            CK(ensure(ctx->b_okeys, sizeof(int) * (size_t)n_units));
            for (int pass = 0; pass < (two ? 2 : 1); ++pass) {
                const int classes = (two && pass == 0 && isfinite(chunk_len)) ? ctx->opt_order_classes : 1;
                size_t n_keys = (size_t)gp * gp * classes;
                CK(ensure(ctx->b_ohist, sizeof(int) * (3 * n_keys + 1)));
                int *hist = (int *)ctx->b_ohist.p, *ptrs = hist + n_keys, *cursor = ptrs + n_keys + 1;
                CK(cudaMemsetAsync(hist, 0, sizeof(int) * (3 * n_keys + 1), st));
                k_unit_keys<<<blocks_for(n_units, 256), 256, 0, st>>>(P, G, classes, gp * gp, chunk_len, chunk_len / ctx->opt_band_div, (int *)ctx->b_okeys.p, hist);
                CK((exclusive_scan<int, int>(ctx, hist, ptrs, (long long)n_keys)));
                k_unit_scatter<<<blocks_for(n_units, 256), 256, 0, st>>>(n_units, (const int *)ctx->b_okeys.p, ptrs, cursor,
                                                                        (int *)ctx->b_order.p + (size_t)pass * n_units);
                *launches += 5;
            }
        }
        ch.order = (const int *)ctx->b_order.p;
        ctx->order_eval = two ? (const int *)ctx->b_order.p + n_units : ch.order;
    }
    if (!reuse) ctx->plan_key = key;
    CK(cudaGetLastError());
    return RT_OK;
}

// ---- single-walk pipeline (mode 3): k_march counts AND records every chunk in one walk, k_eval3 evaluates the records -------
// The records live in a pool of kRecBlock-record blocks: block i < slots is the first block of chunk slot i of the batch, the
// blocks behind are claimed by the walkers as they need them.  Shards whose pool would not fit next to the Segment columns are
// processed in uid batches (whole 32-track blocks): count+record a batch, scan its offsets (carrying the running total), then
// evaluate it -- in sub-batches when its segments exceed the resident capacity.  Next::Hybrid asks for the call to be repeated
// with the hybrid pipeline (pool exhausted: the mesh is far denser along some chunks than the Cauchy-Crofton estimate).
static int segmentize_single(rt_ctx *ctx, WalkParams &P, Attempt &a) {
    cudaStream_t st = ctx->stream;
    const long long n = ctx->n_shard;
    const long long n_blocks = (n + 31) / 32;
    const long long n_units = P.ch.n_units;
    const size_t nn = (size_t)std::max<long long>(n, 1);
    const int *order_all = P.ch.order;
    CK(ensure(ctx->b_tsum, sizeof(double) * nn));  // (cleared per batch by k_seed, like the pool cursor and the volume accumulator)
    CK(ensure(ctx->b_pool_cursor, sizeof(int)));
    P.tsum = (double *)ctx->b_tsum.p;
    P.pool_cursor = (int *)ctx->b_pool_cursor.p;
    const double lmin_eval = ctx->opt_debug_verify_fail ? INFINITY : P.lmin;
    // the evaluation of the records of the tracks and units P describes (cancel: the guard of the optimistic evaluation)
    auto launch_eval = [&](const int *cancel) {
        WalkParams PE = P;
        PE.lmin = lmin_eval;
        PE.cancel = cancel;
        if (PE.ch.order) PE.ch.order = ctx->order_eval;
        k_eval3<<<blocks_for((PE.unit_end - PE.unit_begin) * 32 * 32, kEval3Threads), kEval3Threads, 0, st>>>(PE);
    };

    // ---- memory plan
    size_t free_b = 0, total_b = 0;
    bool have_mem = false;
    auto query_mem = [&]() -> cudaError_t {
        if (have_mem) return cudaSuccess;
        have_mem = true;
        return cudaMemGetInfo(&free_b, &total_b);
    };
    const long long slots_all = n_units * 32;
    const double est_total = ctx->sum_len * crossings_per_length(ctx);
    const double extra_per_slot = est_total * ctx->opt_pool_extra / kRecBlock / (double)std::max<long long>(slots_all, 1);
    const size_t block_bytes = sizeof(int) * (kRecBlock + 1);  // records + chain entry
    const long long spare = ctx->opt_pool_extra > 0.0 ? 4096 : 0;
    auto blocks_for_slots = [&](long long slots) { return slots + (long long)((double)slots * extra_per_slot) + spare; };
    long long max_slots = slots_all;
    if (ctx->opt_pool_slots > 0) max_slots = std::min(max_slots, std::max<long long>(32, ctx->opt_pool_slots & ~31LL));
    const size_t pool_have = std::min<size_t>(ctx->b_pool.bytes / (sizeof(int) * kRecBlock), ctx->b_pool_next.bytes / sizeof(int));
    if ((size_t)blocks_for_slots(std::min(max_slots, slots_all)) > pool_have) {
        CK(query_mem());
        const size_t avail = free_b + ctx->b_pool.bytes + ctx->b_pool_next.bytes + ctx->b_seg_d.bytes + ctx->b_seg_e.bytes;
        const size_t budget = (size_t)((double)avail * 0.15);  // ~9 pool bytes next to 44 Segment bytes per segment
        if ((size_t)blocks_for_slots(std::min(max_slots, slots_all)) * block_bytes > budget) {
            max_slots = (long long)((double)budget / ((double)block_bytes * (1.0 + extra_per_slot))) - 8192;
            max_slots &= ~31LL;
        }
        const long long pb = blocks_for_slots(std::min(max_slots, slots_all));
        if (max_slots < 32 || pb >= (1LL << 31)) {
            a.next = Next::Hybrid;
            return RT_OK;
        }
        if ((size_t)pb > pool_have) {
            if (max_slots < slots_all) {  // the Segment columns are re-fitted to what the pool leaves
                release(ctx->b_seg_d);
                release(ctx->b_seg_e);
                ctx->cap = 0;
            }
            release(ctx->b_pool);
            release(ctx->b_pool_next);
            CK(ensure(ctx->b_pool, sizeof(int) * (size_t)pb * kRecBlock));
            CK(ensure(ctx->b_pool_next, sizeof(int) * (size_t)pb));
            have_mem = false;
        }
    }
    P.pool = (int *)ctx->b_pool.p;
    P.pool_next = (int *)ctx->b_pool_next.p;
    P.pool_blocks = (int)std::min<size_t>(ctx->b_pool.bytes / (sizeof(int) * kRecBlock), ctx->b_pool_next.bytes / sizeof(int));
    if (ctx->opt_pool_extra <= 0.0) P.pool_blocks = (int)std::min<long long>(P.pool_blocks, blocks_for_slots(std::min(max_slots, slots_all)));

    const bool multi = max_slots < slots_all;
    std::vector<long long> h_unit_base;
    if (multi || ctx->cap_cfg > 0) {
        h_unit_base.resize((size_t)n_blocks + 1);
        CK(cudaMemcpyAsync(h_unit_base.data(), ctx->b_unit_base.p, sizeof(long long) * h_unit_base.size(), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    std::vector<long long> h_off;
    long long base = 0;  // segments of the batches already done
    long long B0 = 0;
    ctx->count_batches = 0;
    // phase times are accumulated over the batches (every batch ends with a stream synchronisation anyway)
    double acc[6] = {0, 0, 0, 0, 0, 0};
    auto take = [&](int ph) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->pev[ph][0], ctx->pev[ph][1]) == cudaSuccess) acc[ph] += (double)ms;
        ctx->pev_dirty[ph] = false;
    };
    while (B0 < n_blocks) {
        long long B1 = n_blocks;
        if (multi) {
            const long long lim = h_unit_base[(size_t)B0] + max_slots / 32;
            B1 = (long long)(std::upper_bound(h_unit_base.begin() + B0, h_unit_base.end(), lim) - h_unit_base.begin()) - 1;
            if (B1 <= B0) return fail(ctx, RT_ERR_NOMEM, "rt_segmentize: one block of 32 tracks needs more than the record pool");
        }
        const long long b = 32 * B0, e = std::min(32 * B1, n);
        const long long u0 = multi ? h_unit_base[(size_t)B0] : 0, u1 = multi ? h_unit_base[(size_t)B1] : n_units;
        const long long slots = (u1 - u0) * 32;
        ctx->count_batches += 1;
        // ---- seeds, count+record walk, per-track fix-up, offsets of the batch
        P.trk_begin = b;
        P.trk_end = e;
        P.unit_begin = u0;
        P.unit_end = u1;
        P.ch.order = multi ? nullptr : order_all;
        P.pool_slot_base = u0 * 32;
        P.vol = nullptr;
        P.offset_base = 0;
        P.cursor_init = (int)slots;
        P.zero_vol = (a.want_vol && B0 == 0) ? ctx->vol_acc : nullptr;  // (+1: the failed-rank flag of rt_volumes)
        P.zero_vol_n = (long long)P.m.n_cells + 1;
        if (ctx->opt_debug_clear_pool) CK(cudaMemsetAsync(ctx->b_pool.p, 0, ctx->b_pool.bytes, st));
        if (B0 > 0) tic(ctx, 2);  // (the first batch's count phase started with the chunk plan)
        k_seed<<<blocks_for(slots, 128), 128, 0, st>>>(P);
        k_march<<<blocks_for(slots, kMarchThreads), kMarchThreads, 0, st>>>(P);
        k_fixup_tracks<<<blocks_for(e - b, 128), 128, 0, st>>>(P);
        CK(cudaGetLastError());
        toc(ctx, 2);
        tic(ctx, 3);
        const bool optimistic = !multi && !a.cb && ctx->cap_cfg == 0 && ctx->opt_optimistic && !ctx->skip_optimistic_once &&
                                ctx->fit_gen == ctx->trace_gen && ctx->b_seg_d.p && ctx->cap > 0;
        ScanGuard guard{};
        if (optimistic) guard = ScanGuard{d_guard(ctx), base, ctx->cap, P.pool_cursor, P.pool_blocks};
        CK((exclusive_scan<int, long long>(ctx, (const int *)ctx->b_count.p + b, (long long *)ctx->b_offsets.p + b, e - b, base, guard)));
        toc(ctx, 3);
        a.launches += 6;
        CK(cudaMemcpyAsync(&ctx->h_pin[1], (long long *)ctx->b_offsets.p + e, sizeof(long long), cudaMemcpyDeviceToHost, st));
        if (!optimistic) CK(cudaMemcpyAsync(&ctx->h_pin[9], P.pool_cursor, sizeof(int), cudaMemcpyDeviceToHost, st));
        if (optimistic) {
            // ---- optimistic evaluation: no host round trip between the walk and the evaluation (see rt_ctx::opt_optimistic);
            // the guard (does the batch fit the Segment columns, did the pool hold every record?) is evaluated by the scan
            P.offset_base = base;
            bind_columns(ctx, P);
            P.vol = a.want_vol ? ctx->vol_acc : nullptr;
            tic(ctx, 4);
            launch_eval(d_guard(ctx));
            launch_track_status(ctx, P, a.rtol, d_guard(ctx), d_bad(ctx));
            a.launches += 2;
            CK(cudaGetLastError());
            toc(ctx, 4);
            // (the total, the resident count and the verification and guard flags come with the final read-back of the attempt)
            set_resident(ctx, b, e, base, 0);
            a.defer_total = a.defer_verify = true;
            return RT_OK;
        }
        CK(cudaStreamSynchronize(st));
        take(2);
        take(3);
        const long long batch_total = ctx->h_pin[1] - base;
        if ((long long)*(int *)&ctx->h_pin[9] > (long long)P.pool_blocks) {  // some walker found the pool empty
            a.next = Next::Hybrid;
            return RT_OK;
        }
        ctx->total_segments = base + batch_total;
        // ---- Segment columns: everything of this batch if it fits, else as much as fits
        const long long want = ctx->cap_cfg > 0 ? std::min(batch_total, (long long)ctx->cap_cfg) : batch_total;
        if (want > ctx->cap || !ctx->b_seg_d.p) {
            CK(query_mem());
            long long fitted = 0;
            int rc = size_columns(ctx, want, multi, free_b, &fitted);
            if (rc) return rc;
            have_mem = false;
        }
        const long long cap = ctx->cap_cfg > 0 ? std::min(ctx->cap, (long long)ctx->cap_cfg) : ctx->cap;
        P.offset_base = base;
        bind_columns(ctx, P);
        P.vol = a.want_vol ? ctx->vol_acc : nullptr;
        const bool split = batch_total > cap;
        ctx->fit_gen = (!multi && !split) ? ctx->trace_gen : ~0ULL;  // (the next call with these tracks may skip this round trip)
        if (split) {
            if (h_unit_base.empty()) {  // (one walk batch whose segments do not fit after all: the unit ranges are needed now)
                h_unit_base.resize((size_t)n_blocks + 1);
                CK(cudaMemcpyAsync(h_unit_base.data(), ctx->b_unit_base.p, sizeof(long long) * h_unit_base.size(), cudaMemcpyDeviceToHost, st));
            }
            h_off.resize((size_t)(e - b) + 1);
            CK(cudaMemcpyAsync(h_off.data(), (long long *)ctx->b_offsets.p + b, sizeof(long long) * h_off.size(), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        for (long long sb = b; sb < e; sb = P.trk_end) {
            long long nseg = batch_total;
            if (split) {
                int rc = cut_batch(ctx, P, h_off, b, h_unit_base, sb, cap, &nseg);
                if (rc) return rc;
            }
            tic(ctx, 4);
            if (nseg > 0) launch_eval(nullptr);
            launch_track_status(ctx, P, a.rtol, nullptr, d_bad(ctx));
            a.launches += 2;
            CK(cudaGetLastError());
            set_resident(ctx, P.trk_begin, P.trk_end, P.offset_base, nseg);
            toc(ctx, 4);
            if (!a.cb && !multi && !split) {
                // one batch, nobody waits for it: the verification flag is read with the final read-back of the attempt, which
                // saves one host synchronisation per call; the fill time is collected lazily
                a.defer_verify = true;
                ctx->phase_ms[2] = acc[2];
                ctx->phase_ms[3] = acc[3];
                return RT_OK;
            }
            bool failed = false;
            int rc = read_verify(ctx, &failed);
            if (rc) return rc;
            take(4);
            if (failed) {
                a.next = Next::Sequential;
                return RT_OK;
            }
            rc = deliver_batch(ctx, a);
            if (rc) return rc;
        }
        base += batch_total;
        B0 = B1;
    }
    for (int ph = 2; ph <= 4; ++ph) ctx->phase_ms[ph] = acc[ph];
    return RT_OK;
}

// ---- two-pass pipelines: count -> scan -> fill (possibly in uid batches over a recycled buffer)
//   mode 1 (sequential): k_walk<false> counts, k_walk<true> fills (walk.cuh);
//   mode 0 (hybrid):     k_march counts by sign tests (march.cuh; no record pool, so it records nothing), k_walk<true> fills
//                        and re-derives the same decisions from the exact geometry, k_track_status runs the length check
//                        (src/track.jl:171-175) after the fill.  A fill that disagrees with the count fails the verification:
//                        Next::Sequential.
static int segmentize_two_pass(rt_ctx *ctx, WalkParams &P, uint32_t flags, bool hybrid, Attempt &a) {
    cudaStream_t st = ctx->stream;
    const long long n = ctx->n_shard;
    const size_t nn = (size_t)std::max<long long>(n, 1);
    // (+1: the failed-rank flag of rt_volumes)
    if (a.want_vol) CK(cudaMemsetAsync(ctx->vol_acc, 0, sizeof(double) * ((size_t)ctx->m.n_cells + 1), st));
    // ---- seeds, count pass, per-track fix-up
    if (n > 0) {
        const long long n_units = P.ch.n_units;
        k_seed<<<blocks_for(n_units * 32, 128), 128, 0, st>>>(P);
        if (hybrid) {
            k_march<<<blocks_for(n_units * 32, kMarchThreads), kMarchThreads, 0, st>>>(P);
        } else {
            P.vol = (a.want_vol && (flags & RT_SEG_COUNT_ONLY)) ? ctx->vol_acc : nullptr;
            if (ctx->mixed)
                k_walk<false, true><<<blocks_for(n_units * 32, kWalkThreads), kWalkThreads, 0, st>>>(P);
            else
                k_walk<false><<<blocks_for(n_units * 32, kWalkThreads), kWalkThreads, 0, st>>>(P);
        }
        k_fixup_tracks<<<blocks_for(n, 128), 128, 0, st>>>(P);
        a.launches += 3;
        a.first_bad_scan = true;
    }
    CK(cudaGetLastError());
    toc(ctx, 2);
    // ---- scan
    tic(ctx, 3);
    long long total = 0;
    if (n > 0) {
        CK((exclusive_scan<int, long long>(ctx, (const int *)ctx->b_count.p, (long long *)ctx->b_offsets.p, n)));
        a.launches += 3;
        CK(cudaMemcpyAsync(&ctx->h_pin[1], (long long *)ctx->b_offsets.p + n, sizeof(long long), cudaMemcpyDeviceToHost, st));
    }
    toc(ctx, 3);
    CK(cudaStreamSynchronize(st));
    if (n > 0) total = ctx->h_pin[1];
    ctx->total_segments = total;
    ctx->phase_ms[4] = 0.0;
    ctx->pev_dirty[4] = false;
    if ((flags & RT_SEG_COUNT_ONLY) || n == 0) return RT_OK;

    // ---- fill pass
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    long long cap = 0;
    int rc = size_columns(ctx, ctx->cap_cfg > 0 ? std::min(total, (long long)ctx->cap_cfg) : total, false, free_b, &cap);
    if (rc) return rc;
    if (hybrid) {
        CK(ensure(ctx->b_tsum, sizeof(double) * nn));
        CK(cudaMemsetAsync(ctx->b_tsum.p, 0, sizeof(double) * nn, st));
    }
    bind_columns(ctx, P);
    P.tsum = hybrid ? (double *)ctx->b_tsum.p : nullptr;
    P.vol = a.want_vol ? ctx->vol_acc : nullptr;
    P.counters = nullptr;
    if (ctx->opt_debug_verify_fail && hybrid) CK(cudaMemsetAsync(d_verify(ctx), 1, 1, st));
    const bool split = total > cap;
    std::vector<long long> h_off, h_unit_base;
    if (split) {
        h_off.resize((size_t)n + 1);
        CK(cudaMemcpy(h_off.data(), ctx->b_offsets.p, sizeof(long long) * ((size_t)n + 1), cudaMemcpyDeviceToHost));
        h_unit_base.resize((size_t)((n + 31) / 32) + 1);
        CK(cudaMemcpy(h_unit_base.data(), ctx->b_unit_base.p, sizeof(long long) * h_unit_base.size(), cudaMemcpyDeviceToHost));
    }
    tic(ctx, 4);
    for (long long b = 0; b < n; b = P.trk_end) {
        long long nseg = total;
        if (split) {
            rc = cut_batch(ctx, P, h_off, 0, h_unit_base, b, cap, &nseg);
            if (rc) return rc;
        }
        if (ctx->mixed)
            k_walk<true, true><<<blocks_for((P.unit_end - P.unit_begin) * 32, kWalkThreads), kWalkThreads, 0, st>>>(P);
        else
            k_walk<true><<<blocks_for((P.unit_end - P.unit_begin) * 32, kWalkThreads), kWalkThreads, 0, st>>>(P);
        a.launches += 1;
        if (hybrid) {
            launch_track_status(ctx, P, a.rtol, nullptr, nullptr);
            a.launches += 1;
        }
        CK(cudaGetLastError());
        set_resident(ctx, P.trk_begin, P.trk_end, P.offset_base, nseg);
        if (hybrid) {
            bool failed = false;
            rc = read_verify(ctx, &failed);
            if (rc) return rc;
            if (failed) {
                a.next = Next::Sequential;
                toc(ctx, 4);
                return RT_OK;
            }
        }
        rc = deliver_batch(ctx, a);
        if (rc) return rc;
    }
    toc(ctx, 4);
    return RT_OK;
}

// One attempt of rt_segmentize in pipeline `mode` (segmentize_single or segmentize_two_pass); a.next says whether it stands.
static int segmentize_attempt(rt_ctx *ctx, double tiny_step, int32_t k, int32_t max_iter, uint32_t flags, int mode, Attempt &a,
                              unsigned long long *bad_out) {
    cudaStream_t st = ctx->stream;
    const long long n = ctx->n_shard;
    const int n2 = ctx->n2;
    const DevMesh &m = ctx->m;
    *bad_out = ~0ULL;
    // ---- control block: counters, "no bad track", flags
    for (int q = 0; q < 8; ++q) ctx->h_pin[kPinCtrlInit + q] = 0;
    ctx->h_pin[kPinCtrlInit + 4] = -1LL;
    CK(cudaMemcpyAsync(ctx->b_ctrl.p, &ctx->h_pin[kPinCtrlInit], 64, cudaMemcpyHostToDevice, st));
    if (n == 0) CK(cudaMemsetAsync(ctx->b_offsets.p, 0, sizeof(long long) * 2, st));  // (otherwise the scan writes all n + 1 entries)
    set_resident(ctx, 0, 0, 0, 0);

    WalkParams P{};
    P.m = m;
    P.t = ctx->t;
    const double *ad = (const double *)ctx->b_ang_d.p;
    P.ang.phi = ad;
    P.ang.sinp = ad + n2;
    P.ang.cosp = ad + 2 * n2;
    P.ang.delta_eff = ad + 6 * n2;
    P.tiny = tiny_step;
    P.rtol = mode == 1 ? a.rtol : -1.0;  // sign-test count: the length check runs after the fill (k_track_status)
    P.k = k;
    P.max_iter = max_iter;
    P.flags = flags;
    P.lmin = lmin_of(m, tiny_step);
    P.lmax = ctx->lmax;
    P.smax = ctx->smax;
    P.count = (int *)ctx->b_count.p;
    P.status = (int *)ctx->b_status.p;
    P.offsets = (const long long *)ctx->b_offsets.p;
    P.counters = d_counters(ctx);
    P.verify_fail = d_verify(ctx);
    P.n_tracks = n;
    P.trk_begin = 0;
    P.trk_end = n;

    tic(ctx, 2);  // (the count phase of the first batch includes the chunk plan)
    if (n > 0) {
        int rc = plan_chunks(ctx, P, flags, &a.launches);
        if (rc) return rc;
    }
    int rc = mode == 3 && n > 0 ? segmentize_single(ctx, P, a) : segmentize_two_pass(ctx, P, flags, mode == 0, a);
    if (rc || a.next != Next::Done) return rc;

    ctx->voln_done = false;
    if (a.want_vol && m.n_cells > 0 && ctx->vol_acc && !(ctx->comm && ctx->coll_stream)) {
        // volumes ./= n_azim_2 right behind the evaluation (rt_volumes would launch it after the host has seen the call return:
        // one more host round trip with the GPU idle); with a communicator the all-reduce comes first and rt_volumes does both
        CK(ensure(ctx->b_voln, sizeof(double) * ((size_t)m.n_cells + 1)));
        tic(ctx, 5);
        k_normalise<<<blocks_for(m.n_cells, 256), 256, 0, st>>>(ctx->vol_acc, (double *)ctx->b_voln.p, m.n_cells, (double)ctx->n2);
        CK(cudaGetLastError());
        toc(ctx, 5);
        ctx->voln_done = true;
        a.launches += 1;
    }
    if (a.first_bad_scan) {
        k_first_bad<<<blocks_for(n, 256), 256, 0, st>>>((const int *)ctx->b_status.p, n, d_bad(ctx));
        a.launches += 1;
    }
    CK(cudaMemcpyAsync(&ctx->h_pin[kPinCtrl], ctx->b_ctrl.p, 64, cudaMemcpyDeviceToHost, st));  // counters, first bad track, flags: one copy
    CK(cudaStreamSynchronize(st));
    const int flag_verify = (int)(ctx->h_pin[kPinCtrl + 5] & 0xffffffffLL), flag_guard = (int)((unsigned long long)ctx->h_pin[kPinCtrl + 5] >> 32);
    if (a.defer_total) {  // optimistic evaluation: the total arrives only now
        if (flag_guard) {  // cancelled on the device (Segment columns or record pool too small): repeat on the careful path
            ctx->skip_optimistic_once = true;
            ctx->optimistic_cancels += 1;
            ctx->fit_gen = ~0ULL;
            a.next = Next::RepeatCareful;
            return RT_OK;
        }
        ctx->total_segments = ctx->h_pin[1];
        ctx->res_nseg = ctx->h_pin[1];
    }
    if (a.defer_verify && flag_verify) {
        a.next = Next::Sequential;
        return RT_OK;
    }
    if (n > 0) *bad_out = (unsigned long long)ctx->h_pin[kPinCtrl + 4];
    ctx->stats[0] += a.launches;
    for (int q = 0; q < 4; ++q) ctx->stats[1 + q] = (double)(unsigned long long)ctx->h_pin[kPinCtrl + q];
    return RT_OK;
}

extern "C" int rt_segmentize(rt_ctx *ctx, double tiny_step, int32_t k, double rtol, int32_t max_iter, const double *delta_eff,
                             uint32_t flags, rt_batch_cb cb, void *cb_user, int64_t *n_segments_total, int64_t *first_bad_uid,
                             int32_t *bad_status) {
    if (!ctx) return RT_ERR_ARG;
    if (ctx->in_batch_cb) return fail(ctx, RT_ERR_ARG, "rt_segmentize: called from inside a batch callback");
    // (what rt_correct_volumes may use inside this call's batch callback)
    ctx->prev_vol_valid = ctx->segmented && ctx->vol_valid && ctx->b_voln.p;
    // (whatever goes wrong below, the results of an earlier call are no longer "the last segmentize!": rt_volumes must see that)
    ctx->segmented = false;
    ctx->vol_valid = false;
    if (!ctx->traced)
        return fail(ctx, RT_ERR_NOT_TRACED, "Segmentation is intended after tracing. Please, call `trace!` first!");
    if (k < 1 || max_iter < 0) return fail(ctx, RT_ERR_ARG, "rt_segmentize: bad k / max_iter");
    if (k > kMaxK)
        return fail(ctx, RT_ERR_ARG, "rt_segmentize: k = %d exceeds RT_MAX_K = %d (the k-nearest-node fallback of find_element keeps a fixed-size candidate list)", (int)k, kMaxK);
    const bool want_vol = !(flags & RT_SEG_NO_VOLUMES);
    if (want_vol && !delta_eff) return fail(ctx, RT_ERR_ARG, "rt_segmentize: delta_eff is required unless RT_SEG_NO_VOLUMES");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const long long n = ctx->n_shard;
    const int n2 = ctx->n2;
    DevMesh &m = ctx->m;
    ctx->segmented = false;
    ctx->vol_valid = false;

    if (ctx->mixed) flags |= RT_SEG_LITERAL | RT_SEG_NO_CHUNKS | RT_SEG_SEQUENTIAL;  // quadrilaterals: the reference's walk, step by step
    // count-only with volumes: the volumes are summed by the count walk itself, where every chunk runs on its own (its own max_iter
    // cap, blind to an error or the track end in an earlier chunk) and the fix-up cannot take back what a dropped chunk added.
    // One walker per track stops exactly where the reference loop does.
    if ((flags & RT_SEG_COUNT_ONLY) && want_vol) flags |= RT_SEG_NO_CHUNKS;
    if (!ctx->mixed && ctx->clear_tiny != tiny_step) {
        k_finalize_clear<<<blocks_for(m.n_cells, 128), 128, 0, st>>>(m, (CellRec *)ctx->b_cells.p, (HalfEdge *)ctx->b_he.p,
                                                                     (const float *)ctx->b_qual.p, (const float *)ctx->b_bdist.p,
                                                                     (const MeshScalars *)ctx->b_sc.p,
                                                                     (const float *)ctx->b_node_reach.p, tiny_step, lmin_of(m, tiny_step));
        CK(cudaGetLastError());
        ctx->clear_tiny = tiny_step;
    }
    if (want_vol) {
        // (pageable source: the call returns once the n2 values are staged, no synchronisation needed before the caller reuses them)
        if (!ctx->has_delta || ctx->h_delta.size() != (size_t)n2 || memcmp(ctx->h_delta.data(), delta_eff, sizeof(double) * n2) != 0) {
            CK(cudaMemcpyAsync((double *)ctx->b_ang_d.p + 6 * (size_t)n2, delta_eff, sizeof(double) * n2, cudaMemcpyHostToDevice, st));
            ctx->h_delta.assign(delta_eff, delta_eff + n2);
        }
        ctx->has_delta = true;
        CK(ensure(ctx->b_vol, sizeof(double) * ((size_t)m.n_cells + 1)));
        ctx->vol_acc = (double *)ctx->b_vol.p;
        if (ctx->comm && ctx->coll_stream) {  // alternate, and wait until the collective of two calls ago has released the buffer
            ctx->vol_cur ^= 1;
            if (ctx->vol_cur) {
                CK(ensure(ctx->b_vol_alt, sizeof(double) * ((size_t)m.n_cells + 1)));
                ctx->vol_acc = (double *)ctx->b_vol_alt.p;
            }
            if (ctx->ev_vol_used[ctx->vol_cur]) CK(cudaStreamWaitEvent(st, ctx->ev_vol_free[ctx->vol_cur], 0));
        }
    }
    size_t nn = (size_t)std::max<long long>(n, 1);
    CK(ensure(ctx->b_count, sizeof(int) * nn));
    CK(ensure(ctx->b_status, sizeof(int) * nn));
    CK(ensure(ctx->b_offsets, sizeof(long long) * (nn + 1)));
    CK(ensure(ctx->b_ctrl, 64));

    // the configured pipeline unless a flag asks for behaviour only the sequential kernels have
    int mode = (flags & (RT_SEG_SEQUENTIAL | RT_SEG_COUNT_ONLY)) ? 1 : ctx->opt_pipeline;
    ctx->stats[0] = 0;
    ctx->verify_fallbacks = 0;
    unsigned long long bad = ~0ULL;
    if (mode == 3 && (flags & RT_SEG_LITERAL)) mode = 1;  // (literal-only walks have nothing to gain from per-segment evaluation)
    for (int attempt = 0; attempt < 4; ++attempt) {
        Attempt a{rtol, want_vol, cb, cb_user, attempt};
        int rc = segmentize_attempt(ctx, tiny_step, k, max_iter, flags, mode, a, &bad);
        if (rc) return rc;
        if (a.next == Next::Done) break;
        if (a.next == Next::RepeatCareful) continue;  // the optimistic evaluation did not fit: sized from the walk's result this time
        mode = a.next == Next::Hybrid ? 0 : 1;
        ctx->verify_fallbacks += 1;
    }
    ctx->skip_optimistic_once = false;
    if (n_segments_total) *n_segments_total = ctx->total_segments;
    if (first_bad_uid) *first_bad_uid = 0;
    if (bad_status) *bad_status = 0;
    ctx->segmented = true;
    ctx->vol_valid = want_vol;
    if (bad != ~0ULL) {
        long long idx = (long long)(bad >> 4);
        int stt = (int)(bad & 15);
        if (first_bad_uid) *first_bad_uid = ctx->uid_begin + idx;
        if (bad_status) *bad_status = stt;
        const char *msg = stt == RT_TRACK_TRY_K
                              ? "Try increasing `k`. If the problem persists, raise an issue, this might be a case that hasn't been presented before."
                              : (stt == RT_TRACK_LENGTH ? "has a length that do not match the sum of its segments lengths with the provided tolerance `rtol`."
                                                        : "walk failed");
        return fail(ctx, RT_ERR_TRACK, "Track with `uid` %lld: %s (status %d)", ctx->uid_begin + idx, msg, stt);
    }
    return RT_OK;
}

extern "C" int rt_segment_offsets(rt_ctx *ctx, int64_t *offsets, int32_t *status) {
    if (!ctx || !ctx->segmented) return fail(ctx, RT_ERR_ARG, "rt_segment_offsets: call rt_segmentize first");
    CK(cudaSetDevice(ctx->device));
    size_t n = (size_t)ctx->n_shard;
    if (offsets) CK(cudaMemcpy(offsets, ctx->b_offsets.p, sizeof(long long) * (n + 1), cudaMemcpyDeviceToHost));
    if (status && n) CK(cudaMemcpy(status, ctx->b_status.p, sizeof(int) * n, cudaMemcpyDeviceToHost));
    return RT_OK;
}

extern "C" int rt_segments_download(rt_ctx *ctx, double *px, double *py, double *qx, double *qy, double *len, int32_t *element) {
    if (!resident_valid(ctx)) return fail(ctx, RT_ERR_ARG, "rt_segments_download: call rt_segmentize first");
    CK(cudaSetDevice(ctx->device));
    size_t n = (size_t)ctx->res_nseg;
    if (n == 0) return RT_OK;
    cudaStream_t st = ctx->stream;
    if (px) CK(cudaMemcpyAsync(px, ctx->s_px, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    if (py) CK(cudaMemcpyAsync(py, ctx->s_py, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    if (qx) CK(cudaMemcpyAsync(qx, ctx->s_qx, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    if (qy) CK(cudaMemcpyAsync(qy, ctx->s_qy, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    if (len) CK(cudaMemcpyAsync(len, ctx->s_len, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    if (element) CK(cudaMemcpyAsync(element, ctx->s_elem, sizeof(int) * n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return RT_OK;
}

extern "C" int rt_segments_download_compact(rt_ctx *ctx, double *qx, double *qy, double *len, int32_t *element, int64_t max_exceptions,
                                            int64_t *exc_index, double *exc_px, double *exc_py, int64_t *n_exceptions) {
    if (!resident_valid(ctx)) return fail(ctx, RT_ERR_ARG, "rt_segments_download_compact: call rt_segmentize first");
    if (max_exceptions < 0 || !n_exceptions || (max_exceptions > 0 && (!exc_index || !exc_px || !exc_py)))
        return fail(ctx, RT_ERR_ARG, "rt_segments_download_compact: bad exception buffers");
    CK(cudaSetDevice(ctx->device));
    const long long n = ctx->res_nseg;
    *n_exceptions = 0;
    if (n == 0) return RT_OK;
    cudaStream_t st = ctx->stream;
    // the exception list is built on a side stream (a 0.3 ms kernel over the resident columns) while the four columns that do
    // cross the bus are already on their way
    if (!ctx->aux_stream) {
        CK(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->ev_aux, cudaEventDisableTiming));
    }
    cudaStream_t ax = ctx->aux_stream;
    const size_t cap = (size_t)max_exceptions;
    CK(ensure(ctx->b_exc, 16 + cap * 24));
    unsigned long long *d_cnt = (unsigned long long *)ctx->b_exc.p;
    long long *d_idx = (long long *)((char *)ctx->b_exc.p + 16);
    double *d_px = (double *)(d_idx + cap), *d_py = d_px + cap;
    CK(cudaEventRecord(ctx->ev_aux, st));  // (the evaluation that wrote the columns)
    CK(cudaStreamWaitEvent(ax, ctx->ev_aux, 0));
    CK(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), ax));
    k_p_exceptions<<<blocks_for(n, 256), 256, 0, ax>>>(n, ctx->s_px, ctx->s_py, ctx->s_qx, ctx->s_qy, (long long)cap, d_cnt, d_idx, d_px, d_py);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&ctx->h_pin[11], d_cnt, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ax));
    if (qx) CK(cudaMemcpyAsync(qx, ctx->s_qx, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (qy) CK(cudaMemcpyAsync(qy, ctx->s_qy, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (len) CK(cudaMemcpyAsync(len, ctx->s_len, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (element) CK(cudaMemcpyAsync(element, ctx->s_elem, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(ax));
    const long long k = ctx->h_pin[11];
    *n_exceptions = k;
    if (k > 0 && k <= (long long)cap) {
        CK(cudaMemcpyAsync(exc_index, d_idx, sizeof(long long) * (size_t)k, cudaMemcpyDeviceToHost, ax));
        CK(cudaMemcpyAsync(exc_px, d_px, sizeof(double) * (size_t)k, cudaMemcpyDeviceToHost, ax));
        CK(cudaMemcpyAsync(exc_py, d_py, sizeof(double) * (size_t)k, cudaMemcpyDeviceToHost, ax));
        CK(cudaStreamSynchronize(ax));
    }
    CK(cudaStreamSynchronize(st));
    if (k > (long long)cap)
        return fail(ctx, RT_ERR_NOMEM, "rt_segments_download_compact: %lld exceptions, room for %lld (call again with larger buffers)", k, (long long)cap);
    return RT_OK;
}

extern "C" int rt_segments_device(rt_ctx *ctx, rt_batch *view) {
    if (!ctx || !view) return RT_ERR_ARG;
    view->uid_begin = ctx->uid_begin + ctx->res_trk_begin;
    view->uid_end = ctx->uid_begin + ctx->res_trk_end;
    view->n_segments = ctx->res_nseg;
    view->d_offsets = (const int64_t *)ctx->b_offsets.p;
    view->offset_base = ctx->res_off_base;
    view->d_px = ctx->s_px;
    view->d_py = ctx->s_py;
    view->d_qx = ctx->s_qx;
    view->d_qy = ctx->s_qy;
    view->d_len = ctx->s_len;
    view->d_element = ctx->s_elem;
    view->stream = (void *)ctx->stream;
    view->attempt = 0;
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------------
// sweep-facing device views (SURVEY 8f-1)
// ------------------------------------------------------------------------------------------------------
extern "C" int rt_tracks_device(rt_ctx *ctx, rt_track_view *v) {
    if (!ctx || !v) return RT_ERR_ARG;
    if (!ctx->traced) return fail(ctx, RT_ERR_NOT_TRACED, "rt_tracks_device: call rt_trace first");
    const TrackSoA &t = ctx->t;
    v->uid_begin = ctx->uid_begin;
    v->n_tracks = ctx->n_shard;
    v->d_px = t.px;
    v->d_py = t.py;
    v->d_qx = t.qx;
    v->d_qy = t.qy;
    v->d_len = t.len;
    v->d_a = t.a;
    v->d_b = t.b;
    v->d_c = t.c;
    v->d_azim = t.azim;
    v->d_track_idx = (const int64_t *)t.track_idx;
    v->d_next_fwd = (const int64_t *)t.next_fwd;
    v->d_next_bwd = (const int64_t *)t.next_bwd;
    v->d_bc_fwd = (const int8_t *)t.bc_fwd;
    v->d_bc_bwd = (const int8_t *)t.bc_bwd;
    v->d_dir_fwd = (const int8_t *)t.dir_fwd;
    v->d_dir_bwd = (const int8_t *)t.dir_bwd;
    v->stream = (void *)ctx->stream;
    return RT_OK;
}

extern "C" int rt_quadrature_device(rt_ctx *ctx, rt_quad_view *v, double *omega_host) {
    if (!ctx || !v) return RT_ERR_ARG;
    if (ctx->n2 < 2) return fail(ctx, RT_ERR_NOT_TRACED, "rt_quadrature_device: call rt_trace first");
    CK(cudaSetDevice(ctx->device));
    const int n2 = ctx->n2;
    CK(ensure(ctx->b_omega, sizeof(double) * (size_t)n2));
    const double *ad = (const double *)ctx->b_ang_d.p;
    k_weights<<<blocks_for(n2 / 2, 64), 64, 0, ctx->stream>>>(n2, ad, (double *)ctx->b_omega.p);
    CK(cudaGetLastError());
    v->n_azim_2 = n2;
    v->d_phi = ad;
    v->d_sin = ad + n2;
    v->d_cos = ad + 2 * n2;
    v->d_delta_eff = ctx->has_delta ? ad + 6 * n2 : nullptr;
    v->d_omega = (const double *)ctx->b_omega.p;
    if (omega_host) CK(cudaMemcpyAsync(omega_host, ctx->b_omega.p, sizeof(double) * (size_t)n2, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

extern "C" int rt_optical_lengths(rt_ctx *ctx, int32_t n_groups, const double *sigma_t, int32_t layout, const double **d_tau,
                                  double *tau_host) {
    if (!ctx || n_groups < 1 || !sigma_t || (layout != 0 && layout != 1)) return fail(ctx, RT_ERR_ARG, "rt_optical_lengths: bad arguments");
    if (!resident_valid(ctx)) return fail(ctx, RT_ERR_ARG, "rt_optical_lengths: call rt_segmentize first");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const long long n_seg = ctx->res_nseg;
    const size_t n_sig = (size_t)ctx->m.n_cells * (size_t)n_groups, n_tau = (size_t)std::max<long long>(n_seg, 1) * (size_t)n_groups;
    CK(ensure(ctx->b_sigma, sizeof(double) * n_sig));
    CK(ensure(ctx->b_tau, sizeof(double) * n_tau));
    CK(cudaMemcpyAsync(ctx->b_sigma.p, sigma_t, sizeof(double) * n_sig, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(ctx->ev2[0], st));
    if (n_seg > 0)
        k_tau<<<blocks_for(n_seg * n_groups, 256), 256, 0, st>>>(n_seg, n_groups, ctx->s_len, ctx->s_elem, (const double *)ctx->b_sigma.p,
                                                               layout, (double *)ctx->b_tau.p);
    CK(cudaEventRecord(ctx->ev2[1], st));
    CK(cudaGetLastError());
    if (tau_host && n_seg > 0)
        CK(cudaMemcpyAsync(tau_host, ctx->b_tau.p, sizeof(double) * (size_t)n_seg * n_groups, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev2[0], ctx->ev2[1]);
    ctx->tau_ms = ms;
    if (d_tau) *d_tau = (const double *)ctx->b_tau.p;
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------------
// exact element volumes and the volume correction (SURVEY 8f-2)
// ------------------------------------------------------------------------------------------------------
static int ensure_areas(rt_ctx *ctx) {
    if (ctx->mixed) return fail(ctx, RT_ERR_ARG, "element_volume is defined for triangles (src/trackgenerator.jl:402-411): triangle meshes only");
    if (ctx->area_valid) return RT_OK;
    const int nc = ctx->m.n_cells;
    CK(ensure(ctx->b_area, sizeof(double) * (size_t)nc));
    k_element_volumes<<<blocks_for(nc, 256), 256, 0, ctx->stream>>>(nc, ctx->m.cell_nodes, ctx->m.xy, (double *)ctx->b_area.p);
    CK(cudaGetLastError());
    ctx->area_valid = true;
    return RT_OK;
}

extern "C" int rt_element_volumes(rt_ctx *ctx, double *areas, const double **d_areas) {
    if (!ctx || !ctx->has_mesh) return fail(ctx, RT_ERR_ARG, "rt_element_volumes: upload a mesh first");
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_areas(ctx);
    if (rc) return rc;
    if (areas) CK(cudaMemcpyAsync(areas, ctx->b_area.p, sizeof(double) * (size_t)ctx->m.n_cells, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (d_areas) *d_areas = (const double *)ctx->b_area.p;
    return RT_OK;
}

extern "C" int rt_correct_volumes(rt_ctx *ctx, double *factors, const double **d_factors) {
    // inside a batch callback: the volumes of the call before the running one (its own are summed only as far as its batches go)
    const bool have_vol = ctx && (ctx->in_batch_cb ? ctx->prev_vol_valid : ctx->segmented && ctx->vol_valid && ctx->b_voln.p);
    if (!have_vol)
        return fail(ctx, RT_ERR_ARG, ctx && ctx->in_batch_cb
                                         ? "rt_correct_volumes: inside a batch callback it needs an earlier rt_segmentize with volumes"
                                         : "rt_correct_volumes: run rt_segmentize with volumes enabled and rt_volumes first");
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_areas(ctx);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    const int nc = ctx->m.n_cells;
    if (ctx->voln_ready >= 0) CK(cudaStreamWaitEvent(st, ctx->ev_vol_free[ctx->voln_ready], 0));  // the all-reduced volumes
    CK(ensure(ctx->b_factor, sizeof(double) * (size_t)nc));
    k_volume_factors<<<blocks_for(nc, 256), 256, 0, st>>>(nc, (const double *)ctx->b_area.p, (const double *)ctx->b_voln.p, (double *)ctx->b_factor.p);
    if (ctx->res_nseg > 0)
        k_scale_lengths<<<blocks_for(ctx->res_nseg, 256), 256, 0, st>>>(ctx->res_nseg, ctx->s_elem, (const double *)ctx->b_factor.p, ctx->s_len);
    CK(cudaGetLastError());
    if (factors) CK(cudaMemcpyAsync(factors, ctx->b_factor.p, sizeof(double) * (size_t)nc, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (d_factors) *d_factors = (const double *)ctx->b_factor.p;
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------------
// point location outside the walk
// ------------------------------------------------------------------------------------------------------
extern "C" int rt_find_elements(rt_ctx *ctx, int64_t n, const double *xy, int32_t k, int32_t *element, const int32_t **d_element) {
    if (!ctx) return RT_ERR_ARG;
    if (!ctx->has_mesh) return fail(ctx, RT_ERR_ARG, "rt_find_elements: upload a mesh first");
    if (k < 1 || k > kMaxK) return fail(ctx, RT_ERR_ARG, "rt_find_elements: k = %d outside [1, RT_MAX_K = %d]", (int)k, kMaxK);
    if (n < 0 || (n > 0 && !xy)) return fail(ctx, RT_ERR_ARG, "rt_find_elements: n = %lld points at %p", (long long)n, (const void *)xy);
    // a NaN distance never compares less than another: the ring search would keep the first node it visits and never meet its
    // stopping bound, i.e. scan the whole grid twice for a meaningless answer
    for (int64_t i = 0; i < 2 * n; ++i)
        if (!std::isfinite(xy[i]))
            return fail(ctx, RT_ERR_ARG, "rt_find_elements: point %lld has a non-finite coordinate", (long long)(i / 2));
    ctx->locate_knn = 0.0;
    ctx->locate_ms = 0.0;
    if (n > 0) {
        CK(cudaSetDevice(ctx->device));
        cudaStream_t st = ctx->stream;
        CK(ensure(ctx->b_loc_xy, sizeof(double2) * (size_t)n));
        CK(ensure(ctx->b_loc_elem, sizeof(int) * (size_t)n));
        CK(ensure(ctx->b_loc_knn, sizeof(unsigned long long)));
        CK(cudaMemcpyAsync(ctx->b_loc_xy.p, xy, sizeof(double2) * (size_t)n, cudaMemcpyHostToDevice, st));
        CK(cudaMemsetAsync(ctx->b_loc_knn.p, 0, sizeof(unsigned long long), st));
        CK(cudaEventRecord(ctx->ev2[0], st));
        if (ctx->mixed)
            k_find_elements<true><<<blocks_for(n, kLocateThreads), kLocateThreads, 0, st>>>(
                ctx->m, n, (const double2 *)ctx->b_loc_xy.p, k, (int *)ctx->b_loc_elem.p, (unsigned long long *)ctx->b_loc_knn.p);
        else
            k_find_elements<false><<<blocks_for(n, kLocateThreads), kLocateThreads, 0, st>>>(
                ctx->m, n, (const double2 *)ctx->b_loc_xy.p, k, (int *)ctx->b_loc_elem.p, (unsigned long long *)ctx->b_loc_knn.p);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev2[1], st));
        unsigned long long knn = 0;
        CK(cudaMemcpyAsync(&knn, ctx->b_loc_knn.p, sizeof(knn), cudaMemcpyDeviceToHost, st));
        if (element) CK(cudaMemcpyAsync(element, ctx->b_loc_elem.p, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->ev2[0], ctx->ev2[1]));
        ctx->locate_knn = (double)knn;
        ctx->locate_ms = ms;
    }
    if (d_element) *d_element = (const int32_t *)ctx->b_loc_elem.p;
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------------
// volumes + NCCL
// ------------------------------------------------------------------------------------------------------
static int load_nccl(rt_ctx *ctx) {
    NcclApi &a = ctx->nccl;
    if (a.lib) return RT_OK;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *nm : names) {
        a.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (a.lib) break;
    }
    if (!a.lib) return fail(ctx, RT_ERR_NCCL, "dlopen(libnccl.so.2) failed: %s", dlerror());
    a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(a.lib, "ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))dlsym(a.lib, "ncclCommInitRank");
    a.AllReduce = (decltype(a.AllReduce))dlsym(a.lib, "ncclAllReduce");
    a.CommDestroy = (decltype(a.CommDestroy))dlsym(a.lib, "ncclCommDestroy");
    a.GetErrorString = (decltype(a.GetErrorString))dlsym(a.lib, "ncclGetErrorString");
    if (!a.GetUniqueId || !a.CommInitRank || !a.AllReduce || !a.CommDestroy) return fail(ctx, RT_ERR_NCCL, "NCCL symbols missing");
    return RT_OK;
}

extern "C" int rt_comm_unique_id(rt_ctx *ctx, char id[128]) {
    if (!ctx || !id) return RT_ERR_ARG;
    int rc = load_nccl(ctx);
    if (rc) return rc;
    ncclUniqueId u;
    ncclResult_t r = ctx->nccl.GetUniqueId(&u);
    if (r != 0) return fail(ctx, RT_ERR_NCCL, "ncclGetUniqueId: %s", ctx->nccl.GetErrorString ? ctx->nccl.GetErrorString(r) : "?");
    memcpy(id, u.internal, 128);
    return RT_OK;
}

extern "C" int rt_comm_init(rt_ctx *ctx, int32_t n_ranks, int32_t rank, const char id[128]) {
    if (!ctx || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return RT_ERR_ARG;
    int rc = load_nccl(ctx);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    ncclUniqueId u;
    memcpy(u.internal, id, 128);
    ncclResult_t r = ctx->nccl.CommInitRank(&ctx->comm, n_ranks, u, rank);
    if (r != 0) return fail(ctx, RT_ERR_NCCL, "ncclCommInitRank: %s", ctx->nccl.GetErrorString ? ctx->nccl.GetErrorString(r) : "?");
    if (!ctx->coll_stream) {
        if (cudaStreamCreateWithFlags(&ctx->coll_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_fill_done, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_vol_free[0], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_vol_free[1], cudaEventDisableTiming) != cudaSuccess)
            return fail(ctx, RT_ERR_CUDA, "rt_comm_init: cannot create the collective stream");
    }
    ctx->n_ranks = n_ranks;
    ctx->rank = rank;
    return RT_OK;
}

extern "C" int rt_volumes(rt_ctx *ctx, double *volumes) {
    if (!ctx) return RT_ERR_ARG;
    const bool have = ctx->segmented && ctx->vol_valid;
    const bool coll = ctx->comm && ctx->coll_stream;
    if (!have && !(coll && ctx->has_mesh)) return fail(ctx, RT_ERR_ARG, "rt_volumes: run rt_segmentize with volumes enabled first");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    int nc = ctx->m.n_cells;
    CK(ensure(ctx->b_voln, sizeof(double) * ((size_t)nc + 1)));
    const double *src = ctx->vol_acc ? ctx->vol_acc : (const double *)ctx->b_vol.p;
    if (!have) {
        // This rank's rt_segmentize failed, but its peers are (or will be) inside the all-reduce: join it with a zero contribution
        // and a raised flag in the extra slot, so that nobody hangs and every rank learns that the sums are incomplete.
        CK(cudaStreamSynchronize(ctx->coll_stream));  // (an earlier collective may still be reading b_vol)
        CK(ensure(ctx->b_vol, sizeof(double) * ((size_t)nc + 1)));
        CK(cudaMemsetAsync(ctx->b_vol.p, 0, sizeof(double) * ((size_t)nc + 1), st));
        const double one = 1.0;
        CK(cudaMemcpyAsync((double *)ctx->b_vol.p + nc, &one, sizeof(double), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
        src = (const double *)ctx->b_vol.p;
    }
    if (coll) {
        // the ONLY collective of the path: sum of per-element delta*len over the uid shards -- on its own stream, behind the
        // evaluation that produced the sums and in front of nothing but the next collective.  Element nc of the buffers counts the
        // ranks whose rt_segmentize failed.
        cudaStream_t cs = ctx->coll_stream;
        CK(cudaEventRecord(ctx->ev_fill_done, st));
        CK(cudaStreamWaitEvent(cs, ctx->ev_fill_done, 0));
        CK(cudaEventRecord(ctx->pev[5][0], cs));
        ncclResult_t r = ctx->nccl.AllReduce(src, ctx->b_voln.p, (size_t)nc + 1, ncclFloat64, ncclSum, ctx->comm, cs);
        if (r != 0) return fail(ctx, RT_ERR_NCCL, "ncclAllReduce: %s", ctx->nccl.GetErrorString ? ctx->nccl.GetErrorString(r) : "?");
        ctx->collectives += 1;
        k_normalise<<<blocks_for(nc, 256), 256, 0, cs>>>((const double *)ctx->b_voln.p, (double *)ctx->b_voln.p, nc, (double)ctx->n2);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->pev[5][1], cs));
        ctx->pev_dirty[5] = true;
        if (have) {
            CK(cudaEventRecord(ctx->ev_vol_free[ctx->vol_cur], cs));
            ctx->ev_vol_used[ctx->vol_cur] = true;
            ctx->voln_ready = ctx->vol_cur;
        }
        if (volumes || !have) CK(cudaStreamSynchronize(cs));
        if (!have) return fail(ctx, RT_ERR_ARG, "rt_volumes: this rank's rt_segmentize failed; it joined the all-reduce with a zero contribution and the failed-rank flag");
    } else {
        if (!ctx->voln_done) {  // (rt_segmentize normalises right behind the evaluation)
            tic(ctx, 5);
            k_normalise<<<blocks_for(nc, 256), 256, 0, st>>>(src, (double *)ctx->b_voln.p, nc, (double)ctx->n2);
            CK(cudaGetLastError());
            toc(ctx, 5);
        }
        ctx->voln_ready = -1;
        if (volumes) CK(cudaStreamSynchronize(st));  // (the copy below runs on the legacy stream, which does not wait for ours)
    }
    if (volumes) {
        CK(cudaMemcpy(volumes, ctx->b_voln.p, sizeof(double) * (size_t)nc, cudaMemcpyDeviceToHost));
        if (coll) {
            double failed = 0.0;
            CK(cudaMemcpy(&failed, (const double *)ctx->b_voln.p + nc, sizeof(double), cudaMemcpyDeviceToHost));
            if (failed != 0.0)
                return fail(ctx, RT_ERR_PEER, "rt_volumes: rt_segmentize failed on %d rank(s) of the communicator: the volumes miss their tracks", (int)failed);
        }
    }
    return RT_OK;
}


// ------------------------------------------------------------------------------------------------------
// self-test: the shared-reciprocal division of geom.cuh must equal the IEEE `/` bit for bit
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long &x) {
    unsigned long long z = (x += 0x9e3779b97f4a7c15ull);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__global__ void k_selftest_division(long long n, unsigned long long seed, int exp_span, unsigned long long *mismatch) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long st = seed + 0x632be59bd9b4e019ull * (unsigned long long)(i + 1);
    unsigned long long bad = 0;
    for (int rep = 0; rep < 64; ++rep) {
        // denominators and numerators with random sign, random mantissa and an exponent within +-exp_span of 1.0; every 16th
        // numerator is an exact zero / a power of two / has an all-ones mantissa (the classical hard cases)
        unsigned long long r1 = splitmix64(st), r2 = splitmix64(st), r3 = splitmix64(st);
        int e1 = 1023 + (int)(r3 % (2 * exp_span + 1)) - exp_span, e2 = 1023 + (int)((r3 >> 20) % (2 * exp_span + 1)) - exp_span;
        e1 = min(max(e1, 0), 2046);
        e2 = min(max(e2, 1), 2046);
        unsigned long long mx = r1 & 0xfffffffffffffull, mn = r2 & 0xfffffffffffffull;
        int kind = (int)((r3 >> 44) & 15);
        if (kind == 1) mx = 0;
        if (kind == 2) mx = 0xfffffffffffffull;
        if (kind == 3) mn = 0xfffffffffffffull;
        if (kind == 4) mn = 0;
        double x = __longlong_as_double((long long)(((r1 >> 63) << 63) | ((unsigned long long)e1 << 52) | mx));
        double d = __longlong_as_double((long long)(((r2 >> 63) << 63) | ((unsigned long long)e2 << 52) | mn));
        if (kind == 5) x = 0.0;
        if (kind == 6) x = -0.0;
        Recip r = recip_prepare(d);
        double q1 = div_shared(x, r), q2 = x / d;
        if (__double_as_longlong(q1) != __double_as_longlong(q2)) bad++;
    }
    if (bad) atomicAdd(mismatch, bad);
}

extern "C" int rt_selftest_division(rt_ctx *ctx, int64_t n_threads, uint64_t seed, int32_t exp_span, int64_t *mismatches) {
    if (!ctx || !mismatches || n_threads < 1 || exp_span < 0 || exp_span > 1022) return RT_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    DevBuf d;
    CK(ensure(d, sizeof(unsigned long long)));
    CK(cudaMemsetAsync(d.p, 0, sizeof(unsigned long long), ctx->stream));
    k_selftest_division<<<blocks_for(n_threads, 256), 256, 0, ctx->stream>>>(n_threads, seed, exp_span, (unsigned long long *)d.p);
    CK(cudaGetLastError());
    unsigned long long h = 0;
    CK(cudaMemcpyAsync(&h, d.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    release(d);
    *mismatches = (int64_t)h;
    return RT_OK;
}

extern "C" int rt_stats(rt_ctx *ctx, double stats[8]) {
    if (!ctx || !stats) return RT_ERR_ARG;
    cudaSetDevice(ctx->device);
    collect_phase_ms(ctx);
    ctx->stats[5] = ctx->phase_ms[2];
    ctx->stats[6] = ctx->phase_ms[4];
    ctx->stats[7] = ctx->phase_ms[3];
    memcpy(stats, ctx->stats, sizeof(ctx->stats));
    return RT_OK;
}

extern "C" int rt_info(rt_ctx *ctx, const char *key, double *value) {
    if (!ctx || !key || !value) return RT_ERR_ARG;
    std::string k(key);
    if (k == "verify_fallbacks")
        *value = ctx->verify_fallbacks;
    else if (k == "tau_ms")
        *value = ctx->tau_ms;
    else if (k == "n_units")
        *value = (double)ctx->n_units;
    else if (k == "segment_capacity")
        *value = (double)ctx->cap;
    else if (k == "rho")  // expected cell crossings per unit track length (Cauchy-Crofton): sum of edge lengths / (pi * area)
        *value = ctx->area > 0.0 ? ctx->edge_sum / (kPi * ctx->area) : 0.0;
    else if (k == "band_cost")
        *value = ctx->opt_band_cost;
    else if (k == "count_batches")
        *value = (double)ctx->count_batches;
    else if (k == "optimistic_cancels")
        *value = (double)ctx->optimistic_cancels;
    else if (k == "collectives")
        *value = (double)ctx->collectives;
    else if (k == "locate_knn")
        *value = ctx->locate_knn;
    else if (k == "locate_ms")
        *value = ctx->locate_ms;
    else
        return fail(ctx, RT_ERR_ARG, "rt_info: unknown key %s", key);
    return RT_OK;
}

// diagnostics of the last chunk plan (tools/): out = {chunks with work, void seeds (j >= 1), mean segments per working chunk,
// max segments of a chunk, sum over the units of their longest chunk, sum over the units of their mean chunk, chunk slots, units}
extern "C" int rt_debug_chunk_stats(rt_ctx *ctx, double out[8]) {
    if (!ctx || !out || !ctx->segmented || ctx->n_units <= 0) return fail(ctx, RT_ERR_ARG, "rt_debug_chunk_stats: call rt_segmentize first");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    const long long n = ctx->n_shard, n_units = ctx->n_units, n_blocks = (n + 31) / 32;
    const size_t nc = (size_t)n_units * 32;
    std::vector<int> nch((size_t)n), ublk((size_t)n_units), seed(nc), cnt(nc);
    std::vector<long long> ubase((size_t)n_blocks + 1);
    CK(cudaMemcpy(nch.data(), ctx->b_nch.p, sizeof(int) * nch.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ublk.data(), ctx->b_unit_block.p, sizeof(int) * ublk.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ubase.data(), ctx->b_unit_base.p, sizeof(long long) * ubase.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(seed.data(), ctx->b_ch_i.p, sizeof(int) * nc, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(cnt.data(), (const int *)ctx->b_ch_i.p + 2 * nc, sizeof(int) * nc, cudaMemcpyDeviceToHost));
    double work = 0, voids = 0, sum = 0, mx = 0;
    for (long long u = 0; u < n_units; ++u) {
        const long long b = ublk[(size_t)u];
        const int j = (int)(u - ubase[(size_t)b]);
        for (int l = 0; l < 32; ++l) {
            const long long t = 32 * b + l;
            if (t >= n || j >= nch[(size_t)t]) continue;
            const size_t c = (size_t)u * 32 + l;
            if (j >= 1 && seed[c] < 0) voids += 1;
            if (cnt[c] > 0) {
                work += 1;
                sum += cnt[c];
                mx = std::max(mx, (double)cnt[c]);
            }
        }
    }
    const double mean = work > 0 ? sum / work : 0.0;
    // how evenly a unit's work is spread over its 32 lanes: sum over the units of the LONGEST chunk (what the warp has to wait for)
    // and of the mean chunk of the unit
    double over15 = 0, over2 = 0;
    for (long long u = 0; u < n_units; ++u) {
        const long long b = ublk[(size_t)u];
        const int j = (int)(u - ubase[(size_t)b]);
        double umax = 0, usum = 0;
        for (int l = 0; l < 32; ++l) {
            const long long t = 32 * b + l;
            if (t >= n || j >= nch[(size_t)t]) continue;
            const double c = (double)std::max(cnt[(size_t)u * 32 + l], 0);
            umax = std::max(umax, c);
            usum += c;
        }
        over15 += umax;
        over2 += usum / 32.0;
    }
    out[0] = work;
    out[1] = voids;
    out[2] = mean;
    out[3] = mx;
    out[4] = over15;
    out[5] = over2;
    out[6] = (double)nc;
    out[7] = (double)n_units;
    return RT_OK;
}

extern "C" int rt_phase_ms(rt_ctx *ctx, double ms[6]) {
    if (!ctx || !ms) return RT_ERR_ARG;
    cudaSetDevice(ctx->device);
    collect_phase_ms(ctx);
    memcpy(ms, ctx->phase_ms, sizeof(ctx->phase_ms));
    return RT_OK;
}

extern "C" int rt_timer_start(rt_ctx *ctx) {
    if (!ctx) return RT_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (ctx->coll_stream) CK(cudaStreamSynchronize(ctx->coll_stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventRecord(ctx->tev[0], ctx->stream));
    return RT_OK;
}

extern "C" int rt_timer_stop(rt_ctx *ctx, double *elapsed_ms) {
    if (!ctx || !elapsed_ms) return RT_ERR_ARG;
    if (ctx->voln_ready >= 0) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_vol_free[ctx->voln_ready], 0));  // outstanding collective
    CK(cudaEventRecord(ctx->tev[1], ctx->stream));
    CK(cudaEventSynchronize(ctx->tev[1]));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->tev[0], ctx->tev[1]));
    *elapsed_ms = (double)ms;
    return RT_OK;
}

extern "C" int rt_set_option(rt_ctx *ctx, const char *name, double value) {
    if (!ctx || !name) return RT_ERR_ARG;
    std::string n(name);
    if (n == "chunk_segments" && value >= 1.0)
        ctx->opt_chunk_segments = value;
    else if (n == "target_walkers" && value >= 1.0)
        ctx->opt_target_walkers = value;
    else if (n == "order_grid" && value >= 0.0 && value <= 256.0)
        ctx->opt_order_grid = (int)value;
    else if (n == "pipeline" && (value == 0.0 || value == 1.0 || value == 3.0))
        ctx->opt_pipeline = (int)value;
    else if (n == "debug_clear_pool")
        ctx->opt_debug_clear_pool = value != 0.0;
    else if (n == "band_cost" && value >= 0.0)
        ctx->opt_band_cost = value;
    else if (n == "order_classes" && value >= 0.0 && value <= 64.0)
        ctx->opt_order_classes = (int)value;
    else if (n == "plan_cache")
        ctx->opt_plan_cache = value != 0.0;
    else if (n == "optimistic")
        ctx->opt_optimistic = value != 0.0;
    else if (n == "band_chunks")
        ctx->opt_band_chunks = value != 0.0;
    else if (n == "band_min" && value >= 0.0)
        ctx->opt_band_min = value;
    else if (n == "band_div" && value >= 1.0 && value <= 64.0)
        ctx->opt_band_div = value;
    else if (n == "pool_slots" && value >= 0.0)
        ctx->opt_pool_slots = (long long)value;
    else if (n == "pool_extra" && value >= 0.0)
        ctx->opt_pool_extra = value;
    else if (n == "debug_verify_fail")
        ctx->opt_debug_verify_fail = value != 0.0;
    else
        return fail(ctx, RT_ERR_ARG, "rt_set_option: unknown option or bad value: %s", name);
    return RT_OK;
}
