// walk.cuh -- the segmentation walk: _segmentize_track! (src/track.jl:106-178) as a count pass and a
// fill pass.  Two ways to take a step, producing identical results:
//
//   LITERAL  re-locate xp = q + tiny*(cos phi, sin phi) exactly like the reference (find_element through the
//            nearest node, tolerant barycentric test, inboundary, intersections over all three edges);
//   FAST     when the exit point of the current cell is provably generic (DESIGN.md, "fast-path
//            equivalence"), the reference's next accepted cell is the neighbour across the exit edge and its
//            chord is (shared-edge hit, hit on the one other crossed edge); only that one line/line
//            intersection is evaluated, with the reference's own formula so p, q, len are bit-identical.
//
// Parallel decomposition: a track is cut into CHUNKS at seed points x_j = p + (j/n)*len*(cos, sin).  A seed is
// valid when x_j lies in a cell C whose chord is generic; the state "C has just been pushed" is then history
// independent (intersections() only depends on the cell and the track), so walker j starts from it while walker
// j-1 stops at its first push of C (DESIGN.md, "chunk hand-off").  Invalid seeds are void: the previous walker
// simply continues.  One thread per (track, chunk); a warp holds the same chunk index of 32 consecutive tracks,
// i.e. 32 adjacent parallel rays marching through the same cells.  Threads of a warp alternate between a batch
// of FAST transitions and one LITERAL run-until-push, so the rare literal steps execute together.
#pragma once
#include "mesh_dev.cuh"

namespace rt {

struct AngleTabs {
    const double *phi, *sinp, *cosp, *delta_eff;  // per azimuthal index (0-based), n_azim_2 entries
};

struct TrackSoA {
    double *px, *py, *qx, *qy, *len, *a, *b, *c;
    int *azim;  // 0-based azimuthal index
    long long *track_idx;
    signed char *bc_fwd, *bc_bwd, *dir_fwd, *dir_bwd;
    long long *next_fwd, *next_bwd;
};

// chunk bookkeeping; per-chunk arrays are indexed cidx = unit*32 + lane, consecutive chunks of a track are 32 apart
struct ChunkPlan {
    int *nch;               // per track: number of chunks (>= 1)
    const struct ChunkLayout *layout;  // per track: where the chunks start (k_plan_chunks)
    int *unit_block;        // per warp-unit: which block of 32 consecutive tracks
    long long *unit_base;   // per block: first unit; [n_blocks] = n_units
    long long n_units;
    const int *order;       // execution order of the units (spatially sorted), or nullptr = identity
    int *seed_cell;         // >= 0: valid seed (cell already pushed by the previous walker); -1: void
    int *seed_kexit;
    double *seed_qx, *seed_qy;
    int *count;             // segments pushed by this chunk (count pass; final after fix-up)
    double *sum;            // sum of their lengths
    int *endcode;           // END_* | status << 8
    int *prefix;            // exclusive prefix of final counts inside the track
};

enum { END_HANDOFF = 0, END_TRACK = 1, END_ERROR = 2, END_CAP = 3 };

struct WalkParams {
    DevMesh m;
    long long n_tracks;     // tracks of the shard
    long long trk_begin, trk_end;  // fill pass: only tracks in [trk_begin, trk_end) (batching); count pass: all
    long long unit_begin, unit_end;
    TrackSoA t;
    AngleTabs ang;
    ChunkPlan ch;
    double tiny, rtol, lmin;
    double lmax, smax;  // longest mesh edge, largest |coordinate| (error bounds of the two-stage pipeline)
    int k, max_iter;
    unsigned flags;
    int *count;   // per track (fix-up output)
    int *status;  // per track
    const long long *offsets;  // shard-local exclusive scan of count
    long long offset_base;
    double *opx, *opy, *oqx, *oqy, *olen;
    int *oelem;
    double *vol;                   // unnormalised sum(delta_eff*len) per element, or nullptr
    unsigned long long *counters;  // [fast transitions, literal iterations, nn queries, knn queries] or nullptr
    int *verify_fail;
    const int *cancel;             // optimistic evaluation: set by the scan (ScanGuard) when the batch does not fit (nullptr: not used)
    double *tsum;                  // self-verifying pipelines: per-track sum of segment lengths
    // single-walk pipeline (k_march + k_eval3): pool of record blocks
    int *pool;                     // pool_blocks * kRecBlock records
    int *pool_next;                // per block: the chunk's next block
    int *pool_cursor;              // next unclaimed block
    int pool_blocks;
    long long pool_slot_base;      // chunk slot (unit*32 + lane) whose first block is block 0
    // start-of-batch initialisations folded into k_seed (each used to be a memset / copy in front of the first kernel)
    int cursor_init;               // first unclaimed block = chunk slots of the batch
    double *zero_vol;              // volume accumulator to clear (first batch of a call), or nullptr
    long long zero_vol_n;
};

constexpr int kRecBlock = 256;  // records per pool block (a multiple of 32): with the default chunks of at most ~208 segments a walker
                                // rarely needs a second block, so the claiming atomic stays off the hot path

// smallest sine of a crossing angle the cheap filter of the sign-test walks accepts is 1 / RT_KAPPA_INV (DESIGN.md, "cheap filter")
#ifndef RT_KAPPA_INV
#define RT_KAPPA_INV 1024.0
#endif
enum { MODE_FAST = 0, MODE_SLOW = 1, MODE_DONE = 2 };
constexpr int kFastBatch = 16;
constexpr long long kRunaway = 4000000;
constexpr int kMaxChunksPerTrack = 4096;

// ---- chunk planning -----------------------------------------------------------------------------------
// Chunk layout of a track.  Every track starts and ends on the bounding box; while it is within one cell of a bounding-box line
// it walks through boundary-band cells, where every transition is examined exactly on the slow side of the walk kernels (several
// microseconds instead of one gather).  For the angles closest to the axes that stretch is dozens of cells long at each end (the
// whole track for the rows next to the boundary): one regular chunk of it is a serial chain that outlasts the rest of the launch.
// Such a head / tail (longer than band_min regular chunks) is therefore cut into chunks band_div times shorter:
//     [0, head) in n_head chunks | the middle in n_mid regular chunks | [len - tail, len) in the remaining chunks
struct ChunkLayout {
    float head, tail;  // lengths of the finely chunked ends (0: none)
    int n_head, n_mid;
};
struct PlanGeom {
    const double *px, *py, *qx, *qy;
    double bbmin[2], bbmax[2];
    double band;  // width of the boundary band that counts (the longest mesh edge); 0: uniform chunks only
    double band_min;  // a head / tail gets chunks of its own when it is longer than this
    double band_len;  // ... of this length (both derived from the regular chunk length, see rt_ctx::opt_band_min)
};

// length of the initial part of a track of length `len` whose coordinate a(s) = a0 + s * (a1 - a0) / len stays within `band` of lo / hi
__device__ __forceinline__ double prefix_in_band(double len, double a0, double a1, double lo, double hi, double band) {
    const double da = (a1 - a0) / len;
    double r = 0.0;
    if (a0 < lo + band) r = fmax(r, da > 0.0 ? fmin(len, (lo + band - a0) / da) : len);
    if (a0 > hi - band) r = fmax(r, da < 0.0 ? fmin(len, (hi - band - a0) / da) : len);
    return r;
}

// seed point of chunk j (0 <= j <= n) as a distance from the track's start
__device__ __forceinline__ double chunk_start(const ChunkLayout &L, double len, int n, int j) {
    if (L.n_head == 0 && L.n_mid == n) return len * ((double)j / (double)n);  // uniform (the common case)
    const double head = (double)L.head, tail = (double)L.tail;
    if (j < L.n_head) return head * ((double)j / (double)L.n_head);
    if (j < L.n_head + L.n_mid) return head + (len - head - tail) * ((double)(j - L.n_head) / (double)L.n_mid);
    const int n_tail = n - L.n_head - L.n_mid;
    return n_tail > 0 ? (len - tail) + tail * ((double)(j - L.n_head - L.n_mid) / (double)n_tail) : len;
}

__global__ void k_plan_chunks(long long n_tracks, const double *len, double chunk_len, const __grid_constant__ PlanGeom G, int *nch,
                              ChunkLayout *layout, int *blk_chunks) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    int n = 0;
    if (t < n_tracks) {
        const double l = len[t];
        auto count = [](double x) { return x >= 1.0 ? (x > (double)kMaxChunksPerTrack ? kMaxChunksPerTrack : (int)x) : 1; };
        ChunkLayout L{0.0f, 0.0f, 0, 0};
        double head = 0.0, tail = 0.0;
        if (isfinite(chunk_len) && G.band > 0.0 && l > 0.0) {
            head = fmax(prefix_in_band(l, G.px[t], G.qx[t], G.bbmin[0], G.bbmax[0], G.band),
                        prefix_in_band(l, G.py[t], G.qy[t], G.bbmin[1], G.bbmax[1], G.band));
            tail = fmax(prefix_in_band(l, G.qx[t], G.px[t], G.bbmin[0], G.bbmax[0], G.band),
                        prefix_in_band(l, G.qy[t], G.py[t], G.bbmin[1], G.bbmax[1], G.band));
            if (!(head > G.band_min)) head = 0.0;  // an ordinary end: a few band cells, not worth chunks of its own
            if (!(tail > G.band_min)) tail = 0.0;
        }
        if (head == 0.0 && tail == 0.0) {
            n = count(ceil(l / chunk_len));
            L.n_mid = n;
        } else if (head + tail >= l) {  // the whole track runs along the boundary
            n = count(ceil(l / G.band_len));
            L.n_mid = n;
        } else {
            const int nh = head > 0.0 ? count(ceil(head / G.band_len)) : 0, nt = tail > 0.0 ? count(ceil(tail / G.band_len)) : 0;
            const int nm = count(ceil((l - head - tail) / chunk_len));
            if (nh + nm + nt <= kMaxChunksPerTrack) {
                n = nh + nm + nt;
                L.head = (float)head;
                L.tail = (float)tail;
                L.n_head = nh;
                L.n_mid = nm;
            } else {
                n = count(ceil(l / chunk_len));
                L.n_mid = n;
            }
        }
        nch[t] = n;
        layout[t] = L;
    }
    int mx = __reduce_max_sync(0xffffffffu, n);
    if ((threadIdx.x & 31) == 0 && t < n_tracks) blk_chunks[t >> 5] = mx;
}

__global__ void k_fill_units(long long n_blocks, const long long *unit_base, int *unit_block) {
    long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    for (long long u = unit_base[b]; u < unit_base[b + 1]; ++u) unit_block[u] = (int)b;
}


// ---- spatial execution order of the units ------------------------------------------------------------------------------
// Units (= warps) are independent, so their launch order is free.  Sorting them by the Morton index of the G x G tile
// that holds the chunk's mid point makes the walkers that are resident at the same time work on the same part of the
// mesh: the half-edge records they gather then hit in L1/L2 instead of HBM (the whole table does not fit the cache).
__device__ __forceinline__ unsigned morton2(unsigned x, unsigned y) {
    auto spread = [](unsigned v) {
        v = (v | (v << 8)) & 0x00ff00ffu;
        v = (v | (v << 4)) & 0x0f0f0f0fu;
        v = (v | (v << 2)) & 0x33333333u;
        v = (v | (v << 1)) & 0x55555555u;
        return v;
    };
    return spread(x) | (spread(y) << 1);
}

__global__ void k_unit_keys(const __grid_constant__ WalkParams P, int G, int classes, int keys_per_class, double chunk_len, double band_len,
                            int *keys, int *hist) {
    long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (u >= P.ch.n_units) return;
    int b = P.ch.unit_block[u];
    int j = (int)(u - P.ch.unit_base[b]);
    long long t = min(32LL * b + 16, P.n_tracks - 1);
    int n = P.ch.nch[t];
    int jj = min(j, n - 1);
    int az = P.t.azim[t];
    const ChunkLayout L = P.ch.layout[t];
    double s = 0.5 * (chunk_start(L, P.t.len[t], n, jj) + chunk_start(L, P.t.len[t], n, jj + 1));
    double x = P.t.px[t] + s * P.ang.cosp[az], y = P.t.py[t] + s * P.ang.sinp[az];
    double fx = (x - P.m.bbmin[0]) / (P.m.bbmax[0] - P.m.bbmin[0]), fy = (y - P.m.bbmin[1]) / (P.m.bbmax[1] - P.m.bbmin[1]);
    int ix = min(max((int)(fx * G), 0), G - 1), iy = min(max((int)(fy * G), 0), G - 1);
    int key = (int)morton2((unsigned)ix, (unsigned)iy);
    // Longest units first, shortest last (LPT list scheduling): a unit lives for about a third of the whole walk kernel, so the
    // units that start last decide how long the SMs that are already out of work have to wait (ncu, cfg3, spatial order only:
    // the SMs were active for 0.69 of the kernel's duration on average).  Expected duration of a unit, in regular chunks:
    // its length (a chunk of a track end that runs along the bounding box is 8x shorter, but all its steps take the slow side),
    // plus one for the chunk that starts a track (literal start, boundary band), plus a quarter for the one that ends it.
    // `classes` duration bins, longest first; inside a bin the spatial (Morton) order is kept.
    if (classes > 1) {
        const int n_head = L.n_head, n_mid = L.n_mid;
        const bool band = !(n_head == 0 && n_mid == n) && (jj < n_head || jj >= n_head + n_mid);
        const double len_j = chunk_start(L, P.t.len[t], n, jj + 1) - chunk_start(L, P.t.len[t], n, jj);
        double d = len_j / (band ? band_len : chunk_len) + (j == 0 ? 1.0 : 0.0) + (jj == n - 1 ? 0.25 : 0.0);
        d = fmin(fmax(d, 0.0), 2.0);
        int bin = (int)((2.0 - d) * 0.5 * classes);
        bin = min(max(bin, 0), classes - 1);
        key += bin * keys_per_class;
    }
    keys[u] = key;
    atomicAdd(&hist[key], 1);
}

__global__ void k_unit_scatter(long long n_units, const int *keys, const int *ptrs, int *cursor, int *order) {
    long long u = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (u >= n_units) return;
    int key = keys[u];
    order[ptrs[key] + atomicAdd(&cursor[key], 1)] = (int)u;
}

struct TrackCtx {
    Line trk;
    double g, sx, sy, tlen, delta;
    bool right;
};

__device__ __forceinline__ bool cell_clean(const CellRec &r, const Line &trk, double g, double clear) {
    double thr = g * clear;
    return (fabs(trk.a * r.vx[0] + trk.b * r.vy[0] + trk.c) >= thr) && (fabs(trk.a * r.vx[1] + trk.b * r.vy[1] + trk.c) >= thr) &&
           (fabs(trk.a * r.vx[2] + trk.b * r.vy[2] + trk.c) >= thr);
}

// distance of a point from the nearest bounding-box line
__device__ __forceinline__ double bbox_dist(const DevMesh &m, double x, double y) {
    return fmin(fmin(fabs(x - m.bbmin[0]), fabs(x - m.bbmax[0])), fmin(fabs(y - m.bbmin[1]), fabs(y - m.bbmax[1])));
}

// ---- seeds: one thread per chunk j >= 1 ------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_seed(const __grid_constant__ WalkParams P) {
    long long gw = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (P.pool_cursor) {  // clear what the walk and the evaluation of this batch accumulate into
        const long long gtid = blockIdx.x * (long long)blockDim.x + threadIdx.x, gsz = gridDim.x * (long long)blockDim.x;
        if (gtid == 0) *P.pool_cursor = P.cursor_init;
        if (P.tsum)
            for (long long i = P.trk_begin + gtid; i < P.trk_end; i += gsz) P.tsum[i] = 0.0;
        if (P.zero_vol)
            for (long long i = gtid; i < P.zero_vol_n; i += gsz) P.zero_vol[i] = 0.0;
    }
    long long slot = P.unit_begin + gw;
    if (slot >= P.unit_end) return;
    long long unit = P.ch.order ? P.ch.order[slot] : slot;
    const DevMesh &m = P.m;
    int b = P.ch.unit_block[unit];
    int j = (int)(unit - P.ch.unit_base[b]);
    long long t = 32LL * b + lane;
    long long cidx = unit * 32 + lane;
    if (t >= P.n_tracks) return;
    int n = P.ch.nch[t];
    if (j >= n) return;
    P.ch.seed_cell[cidx] = -1;  // (every field is written: the evaluation requests the seed point of a chunk before it knows whether it needs it)
    P.ch.seed_kexit[cidx] = 0;
    P.ch.seed_qx[cidx] = 0.0;
    P.ch.seed_qy[cidx] = 0.0;
    if (j == 0) return;
    int az = P.t.azim[t];
    Line trk{P.t.a[t], P.t.b[t], P.t.c[t]};
    double s = chunk_start(P.ch.layout[t], P.t.len[t], n, j);
    double x = P.t.px[t] + s * P.ang.cosp[az], y = P.t.py[t] + s * P.ang.sinp[az];
    bool right = P.ang.phi[az] < kPi / 2;
    int c = locate_by_walk(m, x, y);  // (any cell near the seed point that the walk pushes will do: no need for the reference's search)
    if (c < 0) c = find_element(m, x, y, 2, nullptr);
    if (c < 0) return;
    const CellRec &r = m.cells[c];
    if (!isfinite(r.clear)) return;  // degenerate cells never seed
    // Boundary-band cells (clear stored negative) seed only when the whole chord keeps the distance from the bounding box that
    // the fast path asks of an entry point (checked below).  Exactness never depends on this test (a seed cell the serial walk
    // does not push just costs the work of the chunks behind it, see DESIGN.md "chunks"); without such seeds a track that runs
    // along a boundary row of cells is walked by ONE thread from end to end.
    const bool band = r.clear < 0.0f;
    double clear = (double)fabsf(r.clear);
    double g = sqrt(trk.a * trk.a + trk.b * trk.b);
    if (!cell_clean(r, trk, g, clear)) return;
    // the seed point itself must be well inside (not merely tolerantly inside) the cell
    {
        double x1 = r.vx[0], y1 = r.vy[0], x2 = r.vx[1], y2 = r.vy[1], x3 = r.vx[2], y3 = r.vy[2];
        double d = x1 * (y2 - y3) + y1 * (x3 - x2) + (x2 * y3 - y2 * x3);
        double l1 = ((y2 - y3) * x + (x3 - x2) * y + (x2 * y3 - x3 * y2)) / d;
        double l2 = ((y3 - y1) * x + (x1 - x3) * y + (x3 * y1 - x1 * y3)) / d;
        double l3 = ((y1 - y2) * x + (x2 - x1) * y + (x1 * y2 - x2 * y1)) / d;
        const double mrg = 1e-6;
        if (!(l1 > mrg && l2 > mrg && l3 > mrg)) return;
    }
    P2 p, q;
    int e_p, e_q;
    if (intersections(m, c, trk, right, p, q, e_p, e_q) != 0) return;
    if (e_q < 0 || e_p < 0) return;
    double l = norm2(p.x - q.x, p.y - q.y);
    if (!(l > P.lmin)) return;
    if (band) {
        const double need = 0.25 * l + 8.0 * P.tiny;
        if (!(bbox_dist(m, p.x, p.y) > need && bbox_dist(m, q.x, q.y) > need && bbox_dist(m, x, y) > need)) return;
    }
    P.ch.seed_cell[cidx] = c;
    P.ch.seed_kexit[cidx] = e_q;
    P.ch.seed_qx[cidx] = q.x;
    P.ch.seed_qy[cidx] = q.y;
}

// ---- 256-bit read-only loads / 256-bit stores (LDG.E.ENL2.256 / STG.E.ENL2.256 on sm_100a) with L2 eviction policies:
// the half-edge table is re-read by every track that crosses a cell (keep: evict_last), the segment records are
// written once and never read by this kernel (stream: evict_first), so the output does not flush the mesh out of L2.
__device__ __forceinline__ unsigned long long l2_policy_keep() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ unsigned long long l2_policy_stream() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void ldg256_keep(const void *p, unsigned long long pol, double &a, double &b, double &c, double &d) {
    asm volatile("ld.global.nc.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p), "l"(pol));
}
__device__ __forceinline__ void stg256_stream(void *p, unsigned long long pol, double a, double b, double c, double d) {
    asm volatile("st.global.L2::cache_hint.v4.f64 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg128_stream(void *p, unsigned long long pol, int a, int b, int c, int d) {
    asm volatile("st.global.L2::cache_hint.v4.s32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d), "l"(pol) : "memory");
}

constexpr int kWalkThreads = 128;
constexpr int kStage = 8;  // fill pass: staged segments per thread (a ring; complete aligned quads are flushed at warp-uniform points)
// resident blocks per SM the register allocator must allow (without it ptxas picks ~56-72 registers and spills the walk state)
#ifndef RT_WALK_MIN_BLOCKS
#define RT_WALK_MIN_BLOCKS 4
#endif

// ---- the literal walk: src/track.jl:119-168 iterated until ONE segment is pushed (or the walk ends) ------------------
struct LitIn {
    double a, b, c;   // track.ABC
    double sx, sy;    // tiny_step * (cos phi, sin phi)
    double x, y;      // xp = advance_step(x, tiny, phi) is the first point examined
    int prev;         // prev_element (-1: none)
    bool right;       // isless(phi, pi/2)
    bool at_start;    // isempty(segments) and this walker owns the track start
};
struct LitOut {
    int code;    // 0: pushed a segment, END_TRACK, END_ERROR
    int status;  // RT_TRACK_* when code == END_ERROR
    int e, e_q;  // pushed cell, local exit edge (-1: no single exit edge)
    double px, py, qx, qy, l;
    unsigned iters;
    unsigned long long nq[2];  // nearest-node / knn queries
};

template <bool MIXED = false>
__device__ RT_LITERAL_CALL void literal_until_push(const WalkParams &P, const LitIn &in, LitOut &out) {
    const DevMesh &m = P.m;
    Line trk{in.a, in.b, in.c};
    double xpx = in.x + in.sx, xpy = in.y + in.sy;  // advance_step, src/point.jl:43 / src/track.jl:114,165
    int prev = in.prev;
    out.code = END_ERROR;
    out.status = 0;
    out.e = out.e_q = -1;
    out.iters = 0;
    out.nq[0] = out.nq[1] = 0;
    while (true) {
        if (++out.iters > (unsigned)kRunaway) {
            out.status = 3;
            return;
        }
        // find_element's result is discarded on boundary steps (src/track.jl:122-134): test the boundary first
        if (inboundary(m, xpx, xpy, P.tiny)) {
            if (in.at_start) {
                xpx = xpx + in.sx;
                xpy = xpy + in.sy;
                continue;
            }
            out.code = END_TRACK;
            return;
        }
        int e = find_element<MIXED>(m, xpx, xpy, 2, out.nq);
        if (e < 0) {
            e = find_element<MIXED>(m, xpx, xpy, P.k, out.nq);
            if (e < 0) {
                out.status = 1;  // "Try increasing `k`", src/track.jl:141
                return;
            }
        }
        if (e == prev) {
            xpx = xpx + in.sx;
            xpy = xpy + in.sy;
            continue;
        }
        P2 p, q;
        int e_p, e_q;
        int rc = intersections<MIXED>(m, e, trk, in.right, p, q, e_p, e_q);
        if (rc) {
            out.status = rc;
            return;
        }
        if (isapprox_pt(p, q)) {  // src/track.jl:156-159
            xpx = xpx + in.sx;
            xpy = xpy + in.sy;
            continue;
        }
        out.code = 0;
        out.e = e;
        out.e_q = e_q;
        out.px = p.x;
        out.py = p.y;
        out.qx = q.x;
        out.qy = q.y;
        out.l = norm2(p.x - q.x, p.y - q.y);
        return;
    }
}

// ---- the walk ----------------------------------------------------------------------------------------------
// POINTS = false (RT_SEG_LENGTHS_ONLY, fill pass only): the ring stages and the flushes write len and element alone
template <bool FILL, bool MIXED = false, bool POINTS = true>
__global__ void __launch_bounds__(kWalkThreads, RT_WALK_MIN_BLOCKS) k_walk(const __grid_constant__ WalkParams P) {
    const unsigned FULL = 0xffffffffu;
    const DevMesh &m = P.m;
    // fill pass: every thread stages its segments in a ring of kStage slots and writes complete, aligned groups of four as full
    // 32-byte sectors; the flushes happen at points that are uniform across the warp (every fourth fast iteration and once per
    // outer iteration), so the lanes of a warp execute them together although their output positions differ modulo 4
    constexpr int kCols = POINTS ? 5 : 1;  // staged double columns: px, py, qx, qy, len / len
    constexpr int kLen = kCols - 1;
    __shared__ double s_buf[FILL ? kCols * kStage * kWalkThreads : 1];
    __shared__ int s_el[FILL ? kStage * kWalkThreads : 1];
    const int tid = threadIdx.x;
    long long gw = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    long long slot = P.unit_begin + gw;
    if (slot >= P.unit_end) return;  // whole warp
    long long unit = P.ch.order ? P.ch.order[slot] : slot;
    int blk = P.ch.unit_block[unit];
    int j = (int)(unit - P.ch.unit_base[blk]);
    long long t = 32LL * blk + lane;
    long long cidx = unit * 32 + lane;

    int mode = MODE_DONE;
    double ta = 0, tb = 0, tc = 0, g = 0;
    int az = 0;
    bool right = true;
    int nseg = 0, status = 0, endcode = END_TRACK;
    double sum = 0.0;
    long long out = 0;
    // fast state: last pushed cell `cur` with exit point (qx, qy); the encoded half-edge `enc` through which the next
    // cell is entered (-1: boundary); the two end points of that edge (e1, e2) with their signed distances (s1, s2) from
    // the track line; f: e1 is the half-edge's SECOND vertex v_k+1 (else its first, v_k)
    int cur = -1, enc = -1;
    bool f = false, clean = false;
    double e1x = 0, e1y = 0, e2x = 0, e2y = 0, s1 = 0, s2 = 0, qx = 0, qy = 0;
    float clearA = INFINITY;
    double rax = 0, ray = 0, rw0 = 0, rw1 = 0;  // the (prefetched) record of half-edge `enc`
    int stop_cell = -1;  // count pass: hand-off cell of the next valid chunk
    int limit = P.max_iter;
    int n_litpush = 0;  // segments pushed by the literal path (the others are fast transitions)
    const bool literal_only = (P.flags & 1u) != 0;
    bool active = false;
    const unsigned long long pol_keep = l2_policy_keep();
    const unsigned long long pol_stream = FILL ? l2_policy_stream() : 0ull;

    // arm the fast path after cell e was pushed with exit edge e_q (local index) and exit point (ex, ey)
    auto arm = [&](int e, int e_q, double ex, double ey) {
        const CellRec &r = m.cells[e];
        cur = e;
        qx = ex;
        qy = ey;
        clearA = fabsf(r.clear);
        double v0 = ta * r.vx[0] + tb * r.vy[0] + tc, v1 = ta * r.vx[1] + tb * r.vy[1] + tc, v2 = ta * r.vx[2] + tb * r.vy[2] + tc;
        double thr = g * (double)clearA;
        int e_n = e_q == 2 ? 0 : e_q + 1;
        s1 = e_q == 0 ? v0 : (e_q == 1 ? v1 : v2);
        s2 = e_q == 0 ? v1 : (e_q == 1 ? v2 : v0);
        clean = (fabs(v0) >= thr) && (fabs(v1) >= thr) && (fabs(v2) >= thr) && ((s1 > 0) != (s2 > 0));
        e1x = r.vx[e_q];
        e1y = r.vy[e_q];
        e2x = r.vx[e_n];
        e2y = r.vy[e_n];
        enc = m.twin[3 * e + e_q];
        f = (enc & 1) != 0;  // (e1, e2) is the neighbour's (v_k, v_k+1) unless the twin runs in the opposite order
        if (enc >= 0) ldg256_keep(m.he + (enc >> 3), pol_keep, rax, ray, rw0, rw1);
    };

    if (t < P.n_tracks && t >= P.trk_begin && t < P.trk_end) {
        int n = P.ch.nch[t];
        int seed = (j < n) ? (j == 0 ? -2 : P.ch.seed_cell[cidx]) : -1;
        active = (seed != -1);
        if (FILL && active) {
            limit = P.ch.count[cidx];
            active = limit > 0;
        }
        if (active) {
            az = P.t.azim[t];
            ta = P.t.a[t];
            tb = P.t.b[t];
            tc = P.t.c[t];
            double phi = P.ang.phi[az];
            right = phi < kPi / 2;         // isless(phi, pi/2), src/intersection.jl:153
            g = sqrt(ta * ta + tb * tb);
            if (FILL) out = P.offsets[t] - P.offset_base + P.ch.prefix[cidx];
            if (j == 0) {
                qx = P.t.px[t];  // the literal walk starts from advance_step(track.p), src/track.jl:114
                qy = P.t.py[t];
                mode = MODE_SLOW;
            } else {
                arm(seed, P.ch.seed_kexit[cidx], P.ch.seed_qx[cidx], P.ch.seed_qy[cidx]);  // k_seed verified `clean`
                mode = (literal_only || !clean) ? MODE_SLOW : MODE_FAST;
            }
            if (!FILL) {
                for (int jj = j + 1; jj < n; ++jj) {
                    int sc = P.ch.seed_cell[cidx + 32LL * (jj - j)];
                    if (sc >= 0) {
                        stop_cell = sc;
                        break;
                    }
                }
                if (j > 0 && stop_cell == cur) {  // next seed sits in the same cell: this chunk is empty
                    endcode = END_HANDOFF;
                    mode = MODE_DONE;
                }
                if (limit <= 0) {  // while i < MAX_ITER never runs
                    endcode = END_CAP;
                    mode = MODE_DONE;
                }
            }
        }
    }

    long long wpos = out;  // fill pass: every staged segment before this output position has been written
    // write the complete aligned quads among the staged segments [wpos, out + nseg); all = true: everything (chunk end)
    auto flush = [&](bool all) {
        if (!FILL) return;
        const long long o_next = out + nseg;
        const long long head = (wpos + 3) & ~3LL;  // unaligned chunk start: scalar stores up to the first sector boundary
        const long long stop = all ? o_next : (o_next & ~3LL);
        if ((wpos & 3) && head <= stop) {
            for (; wpos < head; ++wpos) {
                const int kk = (int)(wpos & (kStage - 1));
                if (POINTS) {
                    P.opx[wpos] = s_buf[(0 * kStage + kk) * kWalkThreads + tid];
                    P.opy[wpos] = s_buf[(1 * kStage + kk) * kWalkThreads + tid];
                    P.oqx[wpos] = s_buf[(2 * kStage + kk) * kWalkThreads + tid];
                    P.oqy[wpos] = s_buf[(3 * kStage + kk) * kWalkThreads + tid];
                }
                P.olen[wpos] = s_buf[(kLen * kStage + kk) * kWalkThreads + tid];
                P.oelem[wpos] = s_el[kk * kWalkThreads + tid];
            }
        }
        while (!(wpos & 3) && wpos + 4 <= stop) {
            const int k0 = (int)(wpos & (kStage - 1));
            double *dst[5] = {P.opx, P.opy, P.oqx, P.oqy, P.olen};
#pragma unroll
            for (int a = POINTS ? 0 : 4; a < 5; ++a)
                stg256_stream(dst[a] + wpos, pol_stream, s_buf[((a - 4 + kLen) * kStage + k0 + 0) * kWalkThreads + tid],
                              s_buf[((a - 4 + kLen) * kStage + k0 + 1) * kWalkThreads + tid],
                              s_buf[((a - 4 + kLen) * kStage + k0 + 2) * kWalkThreads + tid],
                              s_buf[((a - 4 + kLen) * kStage + k0 + 3) * kWalkThreads + tid]);
            stg128_stream(P.oelem + wpos, pol_stream, s_el[(k0 + 0) * kWalkThreads + tid], s_el[(k0 + 1) * kWalkThreads + tid],
                          s_el[(k0 + 2) * kWalkThreads + tid], s_el[(k0 + 3) * kWalkThreads + tid]);
            wpos += 4;
        }
        if (all) {
            for (; wpos < o_next; ++wpos) {
                const int kk = (int)(wpos & (kStage - 1));
                if (POINTS) {
                    P.opx[wpos] = s_buf[(0 * kStage + kk) * kWalkThreads + tid];
                    P.opy[wpos] = s_buf[(1 * kStage + kk) * kWalkThreads + tid];
                    P.oqx[wpos] = s_buf[(2 * kStage + kk) * kWalkThreads + tid];
                    P.oqy[wpos] = s_buf[(3 * kStage + kk) * kWalkThreads + tid];
                }
                P.olen[wpos] = s_buf[(kLen * kStage + kk) * kWalkThreads + tid];
                P.oelem[wpos] = s_el[kk * kWalkThreads + tid];
            }
        }
    };

    auto push = [&](int e, double ax, double ay, double bx, double by, double l) {
        if (FILL) {
            const int k = (int)((out + nseg) & (kStage - 1));
            if (POINTS) {
                s_buf[(0 * kStage + k) * kWalkThreads + tid] = ax;
                s_buf[(1 * kStage + k) * kWalkThreads + tid] = ay;
                s_buf[(2 * kStage + k) * kWalkThreads + tid] = bx;
                s_buf[(3 * kStage + k) * kWalkThreads + tid] = by;
            }
            s_buf[(kLen * kStage + k) * kWalkThreads + tid] = l;
            s_el[k * kWalkThreads + tid] = e + 1;
        }
        if (P.vol) atomicAdd(&P.vol[e], P.ang.delta_eff[az] * l);  // volumes[i] += delta_s[a]*l, src/trackgenerator.jl:382
        sum += l;
        nseg += 1;
        if (nseg >= limit) {  // while i < MAX_ITER (src/track.jl:119) / this chunk's final count in the fill pass
            endcode = END_CAP;
            mode = MODE_DONE;
        } else if (!FILL && e == stop_cell) {
            endcode = END_HANDOFF;
            mode = MODE_DONE;
        }
    };

    while (__any_sync(FULL, mode != MODE_DONE)) {
        // ------------------------------------------------------------------ FAST phase
#pragma unroll 1
        for (int it = 0; it < kFastBatch; ++it) {
            if (!__any_sync(FULL, mode == MODE_FAST)) break;
            if (mode != MODE_FAST) continue;
            bool ok = false;
            if (enc >= 0) {
                const double ax = rax, ay = ray, w0 = rw0, w1 = rw1;
                const float clearf = __int_as_float(__double2loint(w1));
                const float clearB = fabsf(clearf);
                const double sa = ta * ax + tb * ay + tc;
                const double thr = g * (double)fmaxf(clearA, clearB);
                // the entry edge is crossed (s1, s2 of opposite sign): the exit edge joins the apex with the end point that
                // lies on the other side of the track line
                const bool opp1 = (sa > 0) != (s1 > 0);
                const bool clear_ok = (fabs(sa) >= thr) && (fabs(s1) >= thr) && (fabs(s2) >= thr);
                const double kx = opp1 ? e1x : e2x, ky = opp1 ? e1y : e2y, ks = opp1 ? s1 : s2;
                // exit through edge k+1 = (v_k+1, apex) iff the kept end point is v_k+1, else through k+2 = (apex, v_k).  The
                // record of the half-edge behind that exit is requested NOW: its latency overlaps the arithmetic below.
                const bool exit1 = (opp1 == f);
                const int nenc = exit1 ? __double2loint(w0) : __double2hiint(w0);
                if (nenc >= 0) ldg256_keep(m.he + (nenc >> 3), pol_keep, rax, ray, rw0, rw1);
                // general_form of the exit edge (kept end point, apex), src/intersection.jl:11-18,57.  Its orientation is free:
                // reversing the edge negates (A, B, C) exactly and intersection() is invariant under that negation bit for bit.
                const double A = ky - ay, B = ax - kx, C = kx * ay - ax * ky;
                const Recip rn = recip_prepare(sqrt(A * A + B * B + C * C));
                // (the quotients are only used if `dok` stays true: otherwise the transition is left to the literal walk)
                bool dok = rn.ok;
                const double La = div_try<true>(A, rn, dok), Lb = div_try<true>(B, rn, dok), Lc = div_try<true>(C, rn, dok);
                // intersection(track.ABC, L), src/intersection.jl:127-138 (operands are finite here, so isapprox(a, b) reduces
                // to |a - b| <= rtol * max(|a|, |b|))
                const double a = tb * La, b = Lb * ta;
                const double fa = fabs(a), fb = fabs(b);
                const bool par = fabs(a - b) <= kRtol * (fa > fb ? fa : fb);
                const Recip rd = recip_prepare(a - b);
                dok = dok && rd.ok;
                const double Xx = div_try<false>(tc * Lb - Lc * tb, rd, dok), Xy = div_try<false>(ta * Lc - La * tc, rd, dok);
                const int kin = (enc >> 1) & 3;
                // int_points are stored in edge-index order; order_intersection_points (src/intersection.jl:151-159) must put
                // the entry point first
                const bool kin_lt_kout = (kin == 0) || (kin == 1 && exit1);
                const bool in_first = right ? (kin_lt_kout ? (qx < Xx) : !(Xx < qx)) : (kin_lt_kout ? (qx > Xx) : !(Xx > qx));
                const double dx = qx - Xx, dy = qy - Xy;
                const double l = sqrt(dx * dx + dy * dy);  // Segment(p, q): norm(p - q), src/segment.jl:32
                bool accept = dok && clear_ok && !par && in_first && l > P.lmin;
                // cells touching the bounding-box band: the re-location points must not be `inboundary`
                if (clearf < 0.0f && accept) accept = bbox_dist(m, qx, qy) > 0.25 * l + 8.0 * P.tiny;
                // the walker state needed only by the next fast transition is updated unconditionally (the literal path re-arms it)
                const int cellB = (enc >> 3) / 3;
                e1x = kx;
                e1y = ky;
                s1 = ks;
                e2x = ax;
                e2y = ay;
                s2 = sa;
                f = (exit1 == ((nenc & 1) != 0));
                enc = nenc;
                clearA = clearB;
                if (accept) {
                    const double pxx = qx, pyy = qy;
                    cur = cellB;
                    qx = Xx;
                    qy = Xy;
                    ok = true;
                    push(cellB, pxx, pyy, Xx, Xy, l);
                }
            }
            if (!ok) mode = MODE_SLOW;  // re-locate literally from advance_step(q, tiny, phi), src/track.jl:165-166
            if ((it & 3) == 3) flush(false);
        }
        flush(false);
        // ------------------------------------------------------------------ LITERAL phase (until one push)
        if (mode == MODE_SLOW) {
            // advance_step: x + step*Point2D(cos phi, sin phi), src/point.jl:43
            LitIn in{ta, tb, tc, P.tiny * P.ang.cosp[az], P.tiny * P.ang.sinp[az], qx, qy, cur, right, j == 0 && nseg == 0};
            LitOut o;
            literal_until_push<MIXED>(P, in, o);
            if (P.counters) {
                atomicAdd(&P.counters[1], (unsigned long long)o.iters);
                atomicAdd(&P.counters[2], o.nq[0]);
                if (o.nq[1]) atomicAdd(&P.counters[3], o.nq[1]);
            }
            if (o.code == 0) {
                n_litpush++;
                push(o.e, o.px, o.py, o.qx, o.qy, o.l);
                cur = o.e;
                qx = o.qx;
                qy = o.qy;
                if (mode != MODE_DONE && !literal_only && o.e_q >= 0) {
                    arm(o.e, o.e_q, o.qx, o.qy);
                    if (clean) mode = MODE_FAST;
                }
            } else {
                endcode = o.code;
                status = o.status;
                mode = MODE_DONE;
            }
        }
    }

    flush(true);
    if (!FILL && t < P.n_tracks && j < P.ch.nch[t]) {
        P.ch.count[cidx] = active ? nseg : 0;
        P.ch.sum[cidx] = sum;
        P.ch.endcode[cidx] = active ? (endcode | (status << 8)) : (END_HANDOFF | (0 << 8));
    }
    if (FILL && active && P.tsum) {  // hybrid pipeline: the counts came from the sign-test walk (k_march, march.cuh)
        atomicAdd(&P.tsum[t], sum);
        if (nseg != limit) atomicExch(P.verify_fail, 1);  // this walk ended before producing the counted segments
    }
    if (P.counters) {
        unsigned long long v = active ? (unsigned long long)(nseg - n_litpush) : 0ull;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(FULL, v, o);
        if (lane == 0 && v) atomicAdd(&P.counters[0], v);
    }
}

// ---- per-track fix-up: combine the chunks of a track exactly like one serial walk would have ended ----------
//  * a chunk that ended with an error / at the track end / at the MAX_ITER cap ends the track: later chunks are dropped
//  * the total is capped at max_iter (src/track.jl:119); the length check (src/track.jl:171-175) uses the chunk sums
__global__ void k_fixup_tracks(const __grid_constant__ WalkParams P) {
    long long t = P.trk_begin + blockIdx.x * (long long)blockDim.x + threadIdx.x;  // tracks [trk_begin, trk_end) of the shard
    if (t >= P.trk_end) return;
    int n = P.ch.nch[t];
    long long blk = t >> 5;
    int lane = (int)(t & 31);
    long long c0 = P.ch.unit_base[blk] * 32 + lane;
    int total = 0, status = 0;
    double sum = 0.0;
    bool open = true, truncated = false;
    // (the loads of an iteration do not depend on the running state: requested unconditionally, four iterations at a time)
#pragma unroll 4
    for (int j = 0; j < n; ++j) {
        long long cidx = c0 + 32LL * j;
        const int seed_c = P.ch.seed_cell[cidx], cnt_c = P.ch.count[cidx], ec = P.ch.endcode[cidx];
        const double sum_c = P.ch.sum[cidx];
        bool valid = (j == 0) || seed_c >= 0;
        int cnt = (valid && open) ? cnt_c : 0;
        if (valid && open) {
            int end = ec & 255, st = ec >> 8;
            if (total + cnt >= P.max_iter) {
                if (total + cnt > P.max_iter) truncated = true;
                cnt = P.max_iter - total;
                open = false;
            }
            sum += sum_c;
            if (end == END_ERROR) {
                status = st;
                open = false;
            } else if (end != END_HANDOFF) {
                open = false;  // END_TRACK, or END_CAP inside one chunk
            }
        }
        P.ch.prefix[cidx] = total;
        P.ch.count[cidx] = cnt;
        total += cnt;
    }
    // P.rtol < 0: the two-stage pipeline checks the length after the evaluation (k_track_check)
    if (P.rtol >= 0.0 && status == 0 && (truncated || !isapprox(P.t.len[t], sum, 0.0, P.rtol))) status = 2;
    P.count[t] = total;
    P.status[t] = status;
}

// ---- per-track length check after the fill --------------------------------------------------------------------------------
struct EvalParams {
    TrackSoA t;
    const long long *offsets;      // shard-local exclusive scan of the per-track counts (n_tracks + 1)
    long long trk_begin, trk_end;  // tracks of this batch
    long long offset_base;         // offsets[trk_begin]
    const double *olen;            // segment lengths of this batch
    int *status;   // per track
    double *tsum;  // per track: sum of segment lengths (atomics)
    double rtol;
    const int *cancel;  // optimistic evaluation cancelled (scan.cuh ScanGuard): nothing to check
    unsigned long long *bad;  // min over the failing tracks of (track << 4 | status), or nullptr
};

// isapprox(track.l, sum(l.(segments)); rtol)  src/track.jl:171-175.  The atomically accumulated sum differs from the
// reference's left-to-right sum by at most ~n*eps relative; only when the comparison is that close to its threshold is the
// track re-summed left to right from the segment records.
__global__ void k_track_status(const __grid_constant__ EvalParams P) {
    long long t = P.trk_begin + blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= P.trk_end) return;
    if (P.cancel && *P.cancel) return;
    const int st0 = P.status[t];
    if (st0 != 0) {  // (failed in the walk)
        if (P.bad) atomicMin(P.bad, ((unsigned long long)t << 4) | (unsigned long long)(st0 & 15));
        return;
    }
    const double len = P.t.len[t];
    double sum = P.tsum[t];
    const double tol = P.rtol * fmax(fabs(len), fabs(sum));
    const double slack = 1e-10 * fmax(fabs(len), fabs(sum));
    if (fabs(fabs(len - sum) - tol) <= slack) {
        long long b = P.offsets[t] - P.offset_base, e = P.offsets[t + 1] - P.offset_base;
        sum = 0.0;
        for (long long s = b; s < e; ++s) sum += P.olen[s];
    }
    if (!isapprox(len, sum, 0.0, P.rtol)) {
        P.status[t] = 2;
        if (P.bad) atomicMin(P.bad, ((unsigned long long)t << 4) | 2ull);
    }
}

}  // namespace rt
