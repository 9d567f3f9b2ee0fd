/*
 * rt_b200.h -- C ABI of librt_b200.so: the B200 (sm_100a) implementation of the trace! -> segmentize!
 * hot path of RayTracing.jl v0.2.3.
 *
 * The reference has no FFI of its own: its boundary is the Julia public API (SURVEY.md 8b).  Each entry
 * point below names the reference function whose work it replaces (file:line relative to the reference
 * root); INTEGRATION.md shows the Julia `ccall` glue a maintainer adds on top.  Plain pointers and sizes
 * only.  All functions return RT_OK (0) or a negative rt_status; rt_last_error(ctx) holds a message.
 *
 * Index conventions: mesh tables cross the ABI 1-BASED exactly as Gridap stores them (Table.data /
 * Table.ptrs), track uids and element ids are 1-based as in the reference.  Host arrays are caller
 * owned and only read/written during the call.  There is no CPU fallback: every call needs a CUDA device.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rt_ctx rt_ctx;

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_CUDA = -1,          /* CUDA runtime error (message has the detail) */
    RT_ERR_ARG = -2,           /* invalid argument / call order */
    RT_ERR_NO_EXIT = -4,       /* DomainError("could not found track exit point.")  trackgenerator.jl:219 */
    RT_ERR_BC_MISMATCH = -5,   /* error("Boundaries do not match!")                 trackgenerator.jl:244 */
    RT_ERR_NOT_ON_BOUNDARY = -6, /* error("Point do not lie in the boundary.")      boundary.jl:59 */
    RT_ERR_NOT_TRACED = -7,    /* error("Segmentation is intended after tracing...") trackgenerator.jl:360 */
    RT_ERR_TRACK = -8,         /* a track failed; see first_bad_uid / bad_status of rt_segmentize */
    RT_ERR_NCCL = -9,
    RT_ERR_NOMEM = -10,
    RT_ERR_PEER = -11          /* rt_volumes: another rank's rt_segmentize failed (the all-reduced sums are incomplete) */
} rt_status;

/* per-track status written by rt_segmentize (the reference throws at the first such track) */
enum {
    RT_TRACK_OK = 0,
    RT_TRACK_TRY_K = 1,   /* "Try increasing `k`..."                 src/track.jl:141 */
    RT_TRACK_LENGTH = 2,  /* sum of segment lengths != track length  src/track.jl:171-175 */
    RT_TRACK_RUNAWAY = 3, /* walk did not terminate (guard, no reference counterpart) */
    RT_TRACK_UNDEF = 4    /* x_int1 undefined in intersections()     src/intersection.jl:81-95 */
};

/* boundary-condition codes = the reference's @enum BoundaryType (src/boundary.jl:12-16) */
enum { RT_VACUUM = 0, RT_REFLECTIVE = 1, RT_PERIODIC = 2 };
/* @enum DirectionType (src/track.jl:11-14) */
enum { RT_FORWARD = 0, RT_BACKWARD = 1 };

#define RT_MAX_K 32

/* walk flags for rt_segmentize */
enum {
    RT_SEG_DEFAULT = 0,
    RT_SEG_LITERAL = 1,     /* disable the adjacency fast path: every step re-locates like src/track.jl:122 */
    RT_SEG_NO_VOLUMES = 2,  /* skip the fused fill_volumes accumulation */
    RT_SEG_COUNT_ONLY = 4,  /* count + scan only (no segment buffers are written).  Without RT_SEG_NO_VOLUMES the volumes are
                               those of exactly the segments a full call produces (max_iter cap and failing tracks included):
                               they are summed by the count walk, which then runs one walker per track (as RT_SEG_NO_CHUNKS) */
    RT_SEG_NO_CHUNKS = 8,   /* one walker per track (no sub-track chunks) */
    RT_SEG_SEQUENTIAL = 16  /* sequential walk kernels only (the self-verifying pipelines fall back to them by themselves) */
};

/* ---- context ------------------------------------------------------------------------------------- */
int rt_create(rt_ctx **out, int device);
void rt_destroy(rt_ctx *ctx);
const char *rt_last_error(const rt_ctx *ctx);
const char *rt_version(void);

/* Pinned host memory helpers so callers can stage downloads at full PCIe speed. */
int rt_host_alloc(void **ptr, size_t bytes);
int rt_host_free(void *ptr);

/* ---- mesh: replaces Mesh(model) (src/mesh.jl:24-31) + KDTree(grid) (src/mesh.jl:38-42) ---------------
 * Uploads the flattened Gridap model and builds, on the device, the cell->neighbour table, per-cell and
 * per-edge records (general_form of every edge, src/intersection.jl:11-18) and the uniform node grid
 * that answers the exact nearest-node queries the reference asks its KD-tree (src/mesh.jl:107,123).
 * xy = x0,y0,x1,y1,... ; cell_ptrs/cell_data = get_cell_node_ids(grid) ; node_cell_ptrs/node_cell_data =
 * get_faces(topology, 0, 2) ; bb_min/bb_max = bounding_box(grid) (src/mesh.jl:53-69). Triangles only.
 * Ingestion at scale: node_cell_ptrs/node_cell_data may both be NULL -- the vertex -> cells table is then built on the
 * device (cells around a node in ascending cell id, Gridap's order) -- and bb_min/bb_max may both be NULL -- the bounding
 * box is then an exact min/max reduction on the device (the reference's `min(xs...)` splat, src/mesh.jl:60-62, does not
 * scale to million-node meshes).  rt_mesh_bbox / rt_mesh_node_cells return what was built. */
int rt_mesh_upload(rt_ctx *ctx, int32_t n_nodes, const double *xy, int32_t n_cells, const int32_t *cell_ptrs,
                   const int32_t *cell_data, const int32_t *node_cell_ptrs, const int32_t *node_cell_data,
                   const double bb_min[2], const double bb_max[2]);
int rt_mesh_bbox(rt_ctx *ctx, double bb_min[2], double bb_max[2]);
/* 1-based CSR like Gridap's Table{Int32}; either pointer may be NULL. node_cell_data has 3*n_cells entries. */
int rt_mesh_node_cells(rt_ctx *ctx, int32_t *node_cell_ptrs /* n_nodes+1 */, int32_t *node_cell_data);
/* cell -> neighbour across edge (i, i%3+1) in the cell's stored node order, 1-based, 0 = boundary */
int rt_mesh_neighbours(rt_ctx *ctx, int32_t *cell_nbr /* 3*n_cells */);

/* ---- trace!: replaces trace!(t) (src/trackgenerator.jl:134-280) + next_tracks (:282-348) ------------
 * One kernel over (phi, track) pairs.  The per-angle tables are computed by the CALLER with its own
 * libm (Julia's when Julia calls) because sin/cos/tan/atan are not reproducible across libms:
 * phi = tg.azimuthal_quadrature.phis, sin/cos/tan of it, dx_eff/dy_eff = the local dx/dy of trace!.
 * bcs = top,bottom,right,left.  Only uids in [uid_begin, uid_end) (1-based, end exclusive) are generated
 * on this context: that is the multi-GPU shard.  n_tracks_x/y are the constructor's counts
 * (src/trackgenerator.jl:96-108). */
int rt_trace(rt_ctx *ctx, int32_t n_azim_2, const int64_t *n_tracks_x, const int64_t *n_tracks_y,
             const double *phi, const double *sin_phi, const double *cos_phi, const double *tan_phi,
             const double *dx_eff, const double *dy_eff, const int32_t bcs[4], int64_t uid_begin,
             int64_t uid_end);
/* SoA over the shard's uids (index uid - uid_begin). Any pointer may be NULL.
 * p,q: 2 doubles per track; abc: 3 per track (Track fields, src/track.jl:42-57). */
int rt_tracks_download(rt_ctx *ctx, int64_t *azim_idx, int64_t *track_idx, double *p, double *q, double *phi,
                       double *len, double *abc, int8_t *bc_fwd, int8_t *bc_bwd, int8_t *dir_fwd,
                       int8_t *dir_bwd, int64_t *next_fwd_uid, int64_t *next_bwd_uid);
/* Split [1, n_total] into n_parts contiguous uid ranges of equal total track length (bounds has
 * n_parts+1 entries, bounds[0]=1, bounds[n_parts]=n_total+1). Same tables as rt_trace. */
int rt_plan_shards(rt_ctx *ctx, int32_t n_azim_2, const int64_t *n_tracks_x, const int64_t *n_tracks_y,
                   const double *phi, const double *tan_phi, const double *dx_eff, const double *dy_eff,
                   int32_t n_parts, int64_t *bounds);

/* ---- segmentize!: replaces segmentize!(t; k, rtol) (src/trackgenerator.jl:357-369), i.e. the loop over
 * _segmentize_track! (src/track.jl:106-178) and fill_volumes (src/trackgenerator.jl:371-386) -----------
 * count pass -> exclusive scan -> fill pass (+ fused per-element sum of delta_eff*len).
 * tiny_step: TrackGenerator kwarg; k, rtol: segmentize! kwargs; max_iter: MAX_ITER (src/track.jl:104).
 * 1 <= k <= RT_MAX_K: the k-nearest-node fallback of find_element (src/mesh.jl:123) keeps a fixed-size candidate list;
 * larger values are rejected with RT_ERR_ARG instead of being clamped silently (the reference has no limit).
 * delta_eff: tg.azimuthal_quadrature.deltas (n_azim_2 values) or NULL with RT_SEG_NO_VOLUMES.
 * If the shard's segments exceed the context's segment capacity (rt_set_segment_capacity) the fill runs
 * in uid batches over a recycled buffer and `cb` (may be NULL) is called once per batch.  While `cb` runs, the batch it receives
 * is the resident batch: rt_segments_download, rt_segments_download_compact, rt_optical_lengths and rt_correct_volumes may be called
 * from inside it and act on that batch (outside a callback they need a completed rt_segmentize).  `cb` must not call rt_segmentize.
 * Returns RT_ERR_TRACK if any track failed (first_bad_uid, bad_status say which, like the reference's
 * first thrown error); the other tracks are still segmentized. */
typedef struct rt_batch {
    int64_t uid_begin, uid_end;   /* tracks in this batch */
    int64_t n_segments;           /* segments in this batch */
    const int64_t *d_offsets;     /* DEVICE: offsets of the shard's tracks (n_shard+1), global to the shard */
    int64_t offset_base;          /* subtract from d_offsets[uid-shard_begin] to index the arrays below */
    const double *d_px, *d_py, *d_qx, *d_qy, *d_len; /* DEVICE SoA */
    const int32_t *d_element;     /* DEVICE, 1-based element ids */
    void *stream;                 /* cudaStream_t the batch was produced on */
    int32_t attempt;              /* 1: the call restarted sequentially after a failed verification; drop attempt-0 batches */
} rt_batch;
typedef int (*rt_batch_cb)(const rt_batch *batch, void *user);

int rt_set_segment_capacity(rt_ctx *ctx, int64_t max_segments_resident);
int rt_segmentize(rt_ctx *ctx, double tiny_step, int32_t k, double rtol, int32_t max_iter,
                  const double *delta_eff, uint32_t flags, rt_batch_cb cb, void *cb_user,
                  int64_t *n_segments_total, int64_t *first_bad_uid, int32_t *bad_status);
/* per-track segment counts / offsets / status of the shard after rt_segmentize (host copies) */
int rt_segment_offsets(rt_ctx *ctx, int64_t *offsets /* n_shard+1 */, int32_t *status /* n_shard or NULL */);
/* Segment(p, q, len, element) records (src/segment.jl:23-33) of the resident batch (the whole shard when
 * it fitted), SoA, in uid order then walk order. Any pointer may be NULL.  Also valid inside the batch callback of rt_segmentize. */
int rt_segments_download(rt_ctx *ctx, double *px, double *py, double *qx, double *qy, double *len,
                         int32_t *element);
/* The same records over a thinner wire: 28 instead of 44 bytes per segment cross the bus.  Inside a track, `p` of a segment is
 * `q` of the one before it (src/track.jl:165: the walk continues from q), so only q, len and element are copied; the positions
 * where p differs in any bit from the preceding q -- the first segment of every track, the neighbourhood of the few segments the
 * literal walk produced -- come as an unordered exception list (index into the resident batch, px, py).  The caller rebuilds
 * p[i] = q[i-1] and patches the listed positions: the result is bit-identical to rt_segments_download (tests/test_gpu_parity.py).
 * *n_exceptions receives the number of exceptions found; if it exceeds max_exceptions the call returns RT_ERR_NOMEM after the
 * columns have been copied, and can be repeated with larger buffers.  Column pointers may be NULL.  Also valid inside the batch
 * callback of rt_segmentize. */
int rt_segments_download_compact(rt_ctx *ctx, double *qx, double *qy, double *len, int32_t *element, int64_t max_exceptions,
                                 int64_t *exc_index, double *exc_px, double *exc_py, int64_t *n_exceptions);
/* device-resident view of the resident batch for on-GPU consumers (transport sweeps) */
int rt_segments_device(rt_ctx *ctx, rt_batch *view);

/* ---- what a transport sweep consumes besides the Segment records, kept on the device (SURVEY.md 8f-1) -------------
 * Device-resident view of the shard's Track records (src/track.jl:42-57): the cyclic links next_track_fwd/bwd
 * (src/trackgenerator.jl:282-348, as 1-based GLOBAL uids), link directions and boundary conditions are what the sweep
 * follows from one track to the next; d_azim indexes the per-angle tables of rt_quad_view (0-based). */
typedef struct rt_track_view {
    int64_t uid_begin, n_tracks;                      /* track i of the arrays has uid = uid_begin + i */
    const double *d_px, *d_py, *d_qx, *d_qy, *d_len;  /* track.p, track.q, track.l */
    const double *d_a, *d_b, *d_c;                    /* track.ABC */
    const int32_t *d_azim;                            /* azim_idx - 1 */
    const int64_t *d_track_idx, *d_next_fwd, *d_next_bwd;
    const int8_t *d_bc_fwd, *d_bc_bwd, *d_dir_fwd, *d_dir_bwd; /* RT_VACUUM.. / RT_FORWARD.. */
    void *stream;
} rt_track_view;
int rt_tracks_device(rt_ctx *ctx, rt_track_view *view);

/* Per-angle tables on the device: phi, sin, cos (as passed to rt_trace), delta_eff (as passed to rt_segmentize, NULL before),
 * and the azimuthal weights omega of init_weights! (src/azimuthal_quad.jl:35-53), computed on the device from phi with the
 * reference's formula; omega_host (n_azim_2 doubles) receives a copy when not NULL. */
typedef struct rt_quad_view {
    int32_t n_azim_2;
    const double *d_phi, *d_sin, *d_cos, *d_delta_eff, *d_omega;
} rt_quad_view;
int rt_quadrature_device(rt_ctx *ctx, rt_quad_view *view, double *omega_host);

/* tau[s][g] = sigma_t[element(s)][g] * len(s) for every segment of the resident batch: the `tau::Vector{T}` of each Segment
 * (src/segment.jl:27), which the reference leaves empty for the transport code.  sigma_t: HOST array, n_cells x n_groups
 * (element-major).  layout 0: tau[s*n_groups + g] (the reference's per-segment vectors, concatenated); layout 1:
 * tau[g*n_segments + s].  *d_tau receives the device buffer (owned by the context, valid until the next call);
 * tau_host, when not NULL, receives a copy.  Inside the batch callback of rt_segmentize: tau of the batch the callback received. */
int rt_optical_lengths(rt_ctx *ctx, int32_t n_groups, const double *sigma_t, int32_t layout, const double **d_tau,
                       double *tau_host);

/* ---- exact element volumes and the volume correction (SURVEY 8f-2) -------------------------------------
 * rt_element_volumes: element_volume(mesh, node_ids) = 1/2*abs((x2-x1) x (x3-x1)) for every cell (src/trackgenerator.jl:402-411),
 * computed on the device; `areas` (n_cells, may be NULL) receives a copy, *d_areas (may be NULL) the device buffer.
 * rt_correct_volumes: the step the reference only announces ("correct volumes by changing segment lengths",
 * src/trackgenerator.jl:388-397, flag `volume_correction` :48): after rt_segmentize + rt_volumes, every resident segment length
 * is multiplied by factor[element] = area[element] / volumes[element] (1 where no track crosses the element), so that the
 * traced volumes of the corrected lengths equal the exact areas.  p and q are left untouched.  `factors` / *d_factors: the
 * n_cells factors (host copy / device buffer; either may be NULL).  With batched segments the factors need the volumes of all
 * tracks: run one rt_segmentize with volumes (+ rt_volumes), then a SECOND rt_segmentize whose batch callback calls
 * rt_correct_volumes for every batch.  Inside a callback the factors come from the normalised volumes of the previous completed
 * rt_segmentize (RT_ERR_ARG if that call had none, e.g. RT_SEG_NO_VOLUMES); the correcting call itself may run with or without
 * RT_SEG_NO_VOLUMES, and its own traced volumes are those of the lengths BEFORE correction (they are summed before the callback
 * runs). */
int rt_element_volumes(rt_ctx *ctx, double *areas, const double **d_areas);
int rt_correct_volumes(rt_ctx *ctx, double *factors, const double **d_factors);

/* ---- point location: find_element(mesh, x, k) (src/mesh.jl:103-146) outside the walk ---------------------------------------
 * For n points: xy = x0,y0,x1,y1,... (HOST), element[i] = 1-based cell or -1 (no cell passes the tolerant test, like the reference).
 * The answer is the walk's own find_element: the first passing cell around the nearest node in Gridap's order, then around the k
 * nearest other nodes.  Needs rt_mesh_upload only.  1 <= k <= RT_MAX_K.  Non-finite coordinates are rejected (RT_ERR_ARG, the
 * message names the first such point).  Triangle and mixed meshes.  Nearest-node distance ties go to the lowest node id (the
 * oracle's choice; NearestNeighbors.jl documents none).  n = 0 launches nothing.  element (may be NULL) receives a host copy;
 * *d_element (may be NULL) the device buffer (owned by the context, valid until the next call).  Runs on the context's stream and
 * leaves what rt_segmentize produced untouched (resident batch, offsets, volumes, rt_stats, rt_phase_ms): it may also be called
 * inside the batch callback of rt_segmentize.  rt_info "locate_knn" / "locate_ms" describe the last call. */
int rt_find_elements(rt_ctx *ctx, int64_t n, const double *xy, int32_t k, int32_t *element, const int32_t **d_element);

/* ---- volumes: replaces the tail of fill_volumes (src/trackgenerator.jl:378-386) -----------------------
 * volumes[e] = (sum over this context's segments of delta_eff[azim]*len) / n_azim_2, after an NCCL
 * all-reduce across the communicator set up with rt_comm_init (skipped when there is none).  With a communicator the
 * collective runs on a stream of its own, ordered behind the rt_segmentize that produced the sums: with volumes == NULL the
 * call only enqueues it (it then overlaps with the caller's next rt_segmentize); with a host pointer the call waits for it and
 * copies the result.  Every rank must call rt_volumes once per rt_segmentize, in the same order -- ALSO when its rt_segmentize
 * returned an error (RT_ERR_TRACK leaves valid sums; after any other error the rank joins the collective with a zero contribution
 * and raises a flag that travels with the sums): the call then returns that rank's error, and every rank that asks for the
 * volumes (host pointer) gets RT_ERR_PEER instead of silently incomplete sums.  Nobody is left waiting inside the all-reduce. */
int rt_volumes(rt_ctx *ctx, double *volumes /* n_cells, or NULL */);

/* ---- multi-GPU: one context per process/GPU, tracks sharded by uid range, mesh replicated -----------
 * rank 0 calls rt_comm_unique_id and ships the 128 bytes to the other ranks (MPI / torch.distributed /
 * Julia Distributed); then every rank calls rt_comm_init. NCCL is resolved with dlopen at this point. */
int rt_comm_unique_id(rt_ctx *ctx, char id[128]);
int rt_comm_init(rt_ctx *ctx, int32_t n_ranks, int32_t rank, const char id[128]);

/* ---- instrumentation -----------------------------------------------------------------------------
 * stats[0..7] of the last rt_segmentize: kernel launches, fast transitions, slow (literal) iterations,
 * nearest-node queries, knn queries, count-pass ms, fill-pass ms, scan+volumes ms. */
int rt_stats(rt_ctx *ctx, double stats[8]);
/* named scalars: "verify_fallbacks", "n_units", "segment_capacity", "count_batches"
 * (uid batches of the single-walk pipeline's count walk) of the last rt_segmentize; "optimistic_cancels" (calls of this context
 * whose evaluation, launched behind the walk without reading the segment total back, was cancelled by the device-side guard and
 * repeated); "collectives" (ncclAllReduce calls this context has issued in rt_volumes, including the joins of a rank whose
 * rt_segmentize failed: the ranks of a communicator that call rt_volumes as documented below agree on it); "rho", "band_cost"
 * (shard planning); "tau_ms" (k_tau alone) of the last rt_optical_lengths; "locate_knn" (points that entered the k-nearest-node
 * branch of find_element) and "locate_ms" (k_find_elements alone) of the last rt_find_elements */
int rt_info(rt_ctx *ctx, const char *key, double *value);
/* CUDA-event time (ms) of the last call's device work, by phase: 0 upload+prep, 1 trace, 2 count,
 * 3 scan, 4 fill, 5 volumes(+allreduce) */
int rt_phase_ms(rt_ctx *ctx, double ms[6]);
/* diagnostics of the last rt_segmentize's chunk plan (after the fix-up): {chunks with work, void seeds, mean and max segments per
 * working chunk, sum over the warp units of their longest / of their mean chunk (lane balance of the walk), chunk slots, warp units} */
int rt_debug_chunk_stats(rt_ctx *ctx, double out[8]);

/* self-test: 64*n_threads random quotients x/d (exponents within +-exp_span of 1.0, zeros, powers of two, all-ones
 * mantissas) through the shared-reciprocal division the walk kernels use, compared bit for bit with the IEEE `/`. */
int rt_selftest_division(rt_ctx *ctx, int64_t n_threads, uint64_t seed, int32_t exp_span, int64_t *mismatches);

/* tuning knobs: "chunk_segments" (minimum expected segments per sub-track chunk, default 208),
 * "target_walkers" (chunks are sized so that about this many walkers exist, default 148*2048*4),
 * "order_grid" (G: walkers are launched in Morton order of a G x G tiling of the domain, default 32, 0 = uid order),
 * "order_classes" (duration bins of the walk's launch order, longest units first, Morton order inside a bin; default 3, 0 = spatial
 * order only),
 * "pipeline" (3: ONE sign-test walk that counts and records every chunk + one lane per segment [default]; 0: sign-test count
 * walk + geometric fill walk; 1: sequential geometric walks only.  0 and 3 verify themselves and restart in mode 1 on any
 * disagreement; 3 restarts in mode 0 when its record
 * pool runs out), "band_chunks" (0: uniform chunks also where a track
 * runs along the bounding box), "band_min" / "band_div" (a head or tail of a track that stays inside the boundary band for more
 * than band_min regular chunk lengths [0.0625] is cut into chunks band_div times shorter than the regular ones [8]), "pool_slots" / "pool_extra" (test hooks: chunk slots per count batch, spare record blocks),
 * "debug_verify_fail", "debug_clear_pool" (test hooks), "plan_cache" (0: rebuild the chunk plan in every call), "optimistic" (0: always read
 * the segment total back before the evaluation is launched) */
int rt_set_option(rt_ctx *ctx, const char *name, double value);
/* CUDA-event stopwatch on the context's launching stream (bench harness: torch.cuda.Event cannot see it). */
int rt_timer_start(rt_ctx *ctx);
int rt_timer_stop(rt_ctx *ctx, double *elapsed_ms);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
