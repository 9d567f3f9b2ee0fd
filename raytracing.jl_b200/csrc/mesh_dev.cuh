// mesh_dev.cuh -- device-resident flattened mesh, its preparation kernels, and the literal point
// location of the reference (find_element / point_in_triangle / inboundary, src/mesh.jl:91-176) with the
// KD-tree of NearestNeighbors.jl replaced by an exact uniform-grid nearest-node search.
#pragma once
#include "geom.cuh"

namespace rt {

// 64-byte per-cell record read once per fast transition (two 32 B sectors, no dependent gathers).
struct __align__(32) CellRec {
    double vx[3];
    double vy[3];
    int nbr[3];   // 0-based cell across edge k = (k, (k+1)%3); -1 on the boundary
    float clear;  // required perpendicular clearance of the track from this cell's vertices; +inf = always literal
};
static_assert(sizeof(CellRec) == 64, "CellRec must be 64 bytes");

// 32-byte per-(cell, edge) record: general_form(P_k, P_k+1) (src/intersection.jl:57) and |P_k - P_k+1|.
struct __align__(32) EdgeRec {
    double a, b, c, len;
};

// 32-byte record (ONE sector) of the directed half-edge h = 3*cell + k, read when a track ENTERS `cell` through its
// edge k = (v_k, v_k+1).  The walker carries the coordinates of v_k and v_k+1 (they are the end points of the edge it
// left the previous cell through), so the apex completes the triangle and general_form of the exit edge
// (src/intersection.jl:57) is evaluated on the fly from the same node coordinates, in the cell's stored orientation.
struct __align__(32) HalfEdge {
    double ax, ay;  // apex v_k+2
    int tw1, tw2;   // entry half-edge of the neighbour across edge k+1 = (v_k+1, apex) / k+2 = (apex, v_k),
                    // encoded (3*cell' + k') << 3 | k' << 1 | flip (flip: end points in opposite order); -1 on the boundary
    float clear;    // = CellRec::clear of this cell
    float clear2;   // l_min / sigma: a lone vertex at least this far from the track line has a chord longer than l_min
};
static_assert(sizeof(HalfEdge) == 32, "HalfEdge must be 32 bytes");

struct DevMesh {
    const HalfEdge *he;  // [3*cell + k]
    const int *twin;     // [3*cell + k]: encoded entry half-edge of the neighbour across edge k (as tw1/tw2)
    int n_nodes, n_cells;
    const double2 *xy;      // node coordinates
    const int *cell_nodes;  // 3*n_cells, 0-based, stored (Gridap) order; mixed meshes: the CSR data of cell_ptrs
    const int *cell_ptrs;   // nullptr: every cell is a triangle.  Otherwise 0-based CSR offsets (n_cells + 1) of a MIXED mesh of
                            // 3- and 4-node cells (SURVEY 8f-4): only the literal walk runs on it, from xy / cell_nodes directly
    const int *nc_ptrs;     // node -> cells CSR, 0-based, caller's order (src/mesh.jl:27)
    const int *nc_data;
    const CellRec *cells;
    const EdgeRec *edges;  // [3*cell + k]
    // uniform node grid
    int gx, gy;
    double g0x, g0y, gh, ginv;
    const int *grid_ptrs;   // gx*gy + 1
    const int *grid_nodes;  // node ids binned
    const int *cell_bin;    // gx*gy: a cell whose centroid lies in the bin (-1: none) -- entry point of the seed location walk
    double bbmin[2], bbmax[2];
};

// ------------------------------------------------------------------------------------------------
// preparation kernels (run once per rt_mesh_upload)
// ------------------------------------------------------------------------------------------------

__global__ void k_to_zero_based(const int32_t *in, int *out, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] - 1;
}

// ---- device-side ingestion (SURVEY 8f-3): the tables the reference takes from Gridap / computes with a splat ----------------
// bounding_box(grid) (src/mesh.jl:53-69) = min / max over all node coordinates: an exact, order-independent reduction.
__device__ __forceinline__ void atomic_min_double_any(double *addr, double v) {
    unsigned long long *a = (unsigned long long *)addr, old = *a, assumed;
    do {
        assumed = old;
        if (!(v < __longlong_as_double((long long)assumed))) break;
        old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
    } while (old != assumed);
}
__device__ __forceinline__ void atomic_max_double_any(double *addr, double v) {
    unsigned long long *a = (unsigned long long *)addr, old = *a, assumed;
    do {
        assumed = old;
        if (!(v > __longlong_as_double((long long)assumed))) break;
        old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
    } while (old != assumed);
}
// bb = {min x, min y, max x, max y}, initialised to {+inf, +inf, -inf, -inf}
__global__ void k_bbox(const double2 *xy, int n_nodes, double *bb) {
    double mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_nodes; i += gridDim.x * blockDim.x) {
        const double2 p = xy[i];
        mnx = fmin(mnx, p.x);
        mny = fmin(mny, p.y);
        mxx = fmax(mxx, p.x);
        mxy = fmax(mxy, p.y);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mnx = fmin(mnx, __shfl_down_sync(0xffffffffu, mnx, o));
        mny = fmin(mny, __shfl_down_sync(0xffffffffu, mny, o));
        mxx = fmax(mxx, __shfl_down_sync(0xffffffffu, mxx, o));
        mxy = fmax(mxy, __shfl_down_sync(0xffffffffu, mxy, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomic_min_double_any(&bb[0], mnx);
        atomic_min_double_any(&bb[1], mny);
        atomic_max_double_any(&bb[2], mxx);
        atomic_max_double_any(&bb[3], mxy);
    }
}

// vertex -> cells table = get_faces(get_grid_topology(model), 0, 2) (src/mesh.jl:27): cells around each node in ASCENDING cell
// id (the order find_element scans them in, src/mesh.jl:110).  count -> scan -> fill (atomic cursor) -> per-node sort.
__global__ void k_nc_count(int n_cells, const int *cell_nodes, int *deg) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < 3 * (int64_t)n_cells) atomicAdd(&deg[cell_nodes[t]], 1);
}
__global__ void k_nc_fill(int n_cells, const int *cell_nodes, const int *ptrs, int *cursor, int *data) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= 3 * (int64_t)n_cells) return;
    const int node = cell_nodes[t];
    data[ptrs[node] + atomicAdd(&cursor[node], 1)] = (int)(t / 3);
}
__global__ void k_nc_sort(int n_nodes, const int *ptrs, int *data) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const int b = ptrs[i], e = ptrs[i + 1];
    for (int q = b + 1; q < e; ++q) {  // insertion sort: the valence of a mesh node is small
        const int v = data[q];
        int r = q - 1;
        while (r >= b && data[r] > v) {
            data[r + 1] = data[r];
            --r;
        }
        data[r + 1] = v;
    }
}

// one thread per (cell, edge): the neighbour is the other cell around node a that also contains node b
__global__ void k_neighbours(int n_cells, const int *cell_nodes, const int *nc_ptrs, const int *nc_data, int *nbr) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= 3 * (int64_t)n_cells) return;
    int c = (int)(t / 3), k = (int)(t % 3);
    int a = cell_nodes[3 * c + k], b = cell_nodes[3 * c + (k + 1) % 3];
    int found = -1;
    for (int q = nc_ptrs[a]; q < nc_ptrs[a + 1]; ++q) {
        int c2 = nc_data[q];
        if (c2 == c) continue;
        const int *n2 = &cell_nodes[3 * c2];
        if (n2[0] == b || n2[1] == b || n2[2] == b) {
            found = c2;
            break;
        }
    }
    nbr[t] = found;
}

struct MeshScalars {
    double lmax;      // longest edge
    double smax;      // largest |coordinate|
    double edge_sum;  // sum over (cell, edge) of the edge length (interior edges counted twice)
    double area;      // total mesh area
};

__device__ __forceinline__ void atomic_max_double(double *addr, double v) {
    // values are non-negative: ordering of the bit patterns equals ordering of the doubles
    atomicMax((unsigned long long *)addr, (unsigned long long)__double_as_longlong(v));
}

// mixed meshes (3- and 4-node cells): the density scalars only -- edges are consecutive stored nodes, like in intersections()
// (src/intersection.jl:46-51); the area of a quadrilateral is the shoelace sum over its stored cycle
__global__ void k_mesh_scalars_generic(int n_cells, const int *cell_ptrs, const int *cell_nodes, const double2 *xy, MeshScalars *sc) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells) return;
    const int b = cell_ptrs[c], nn = cell_ptrs[c + 1] - b;
    double lmax = 0.0, smax = 0.0, esum = 0.0, a2 = 0.0;
    for (int i = 0; i < nn; ++i) {
        const double2 p = xy[cell_nodes[b + i]], q = xy[cell_nodes[b + (i + 1 == nn ? 0 : i + 1)]];
        const double l = norm2(p.x - q.x, p.y - q.y);
        lmax = fmax(lmax, l);
        esum += l;
        smax = fmax(smax, fmax(fabs(p.x), fabs(p.y)));
        a2 += p.x * q.y - q.x * p.y;
    }
    atomic_max_double(&sc->lmax, lmax);
    atomic_max_double(&sc->smax, smax);
    atomicAdd(&sc->edge_sum, esum);
    atomicAdd(&sc->area, 0.5 * fabs(a2));
}

// per cell: vertex coordinates, neighbours, edge records, geometric quality numbers
// qual[c] = (1 + 8*eps*(S/hmin)^2/rtol) / sigma, sigma = min sine of the interior angles; bdist[c] = min distance of
// the cell's vertices from the bounding-box lines.  (clear is finalised per segmentize call, it depends on tiny_step.)
__global__ void k_cell_records(DevMesh m, const int *nbr, CellRec *cells, EdgeRec *edges, float *qual, float *bdist,
                               MeshScalars *sc) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = c < m.n_cells;
    if (!live) c = m.n_cells - 1;  // keep the warp converged for the reductions below; results are not stored
    P2 v[3];
    for (int k = 0; k < 3; ++k) {
        double2 p = m.xy[m.cell_nodes[3 * c + k]];
        v[k].x = p.x;
        v[k].y = p.y;
    }
    CellRec r;
    double lmax = 0.0, smax = 0.0, bd = INFINITY;
    double len[3];
    for (int k = 0; k < 3; ++k) {
        int j = (k + 1) % 3;
        r.vx[k] = v[k].x;
        r.vy[k] = v[k].y;
        r.nbr[k] = nbr[3 * c + k];
        Line l = general_form(v[k], v[j]);
        EdgeRec e;
        e.a = l.a;
        e.b = l.b;
        e.c = l.c;
        e.len = norm2(v[k].x - v[j].x, v[k].y - v[j].y);
        if (live) edges[3 * c + k] = e;
        len[k] = e.len;
        lmax = fmax(lmax, e.len);
        smax = fmax(smax, fmax(fabs(v[k].x), fabs(v[k].y)));
        bd = fmin(bd, fmin(fmin(fabs(v[k].x - m.bbmin[0]), fabs(v[k].x - m.bbmax[0])),
                           fmin(fabs(v[k].y - m.bbmin[1]), fabs(v[k].y - m.bbmax[1]))));
    }
    double area2 = fabs((v[1].x - v[0].x) * (v[2].y - v[0].y) - (v[2].x - v[0].x) * (v[1].y - v[0].y));
    // sine of the angle at vertex k = 2*Area / (product of the two edges meeting there)
    double s0 = area2 / (len[0] * len[2]), s1 = area2 / (len[0] * len[1]), s2 = area2 / (len[1] * len[2]);
    double sigma = fmin(s0, fmin(s1, s2));
    double hmin = area2 / lmax;
    r.clear = INFINITY;
    if (live) {
        cells[c] = r;
        qual[c] = (sigma > 0.0 && hmin > 0.0) ? (float)(1.0 / sigma) : INFINITY;
        bdist[c] = (float)bd;
    } else {
        len[0] = len[1] = len[2] = 0.0;
        area2 = 0.0;
    }
    // hmin feeds the lambda rounding-error term; stash via a second pass using smax (global), see k_finalize_clear
    // Cauchy-Crofton: a random line crosses edge_sum / (pi * area) cell edges per unit length (chunk sizing only)
    double es = len[0] + len[1] + len[2], ar = 0.5 * area2;
    for (int o = 16; o > 0; o >>= 1) {  // one atomic per warp and scalar (one per thread on a single address took 1.3 of the upload's 2.2 ms)
        es += __shfl_down_sync(0xffffffffu, es, o);
        ar += __shfl_down_sync(0xffffffffu, ar, o);
        lmax = fmax(lmax, __shfl_down_sync(0xffffffffu, lmax, o));
        smax = fmax(smax, __shfl_down_sync(0xffffffffu, smax, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomic_max_double(&sc->lmax, lmax);
        atomic_max_double(&sc->smax, smax);
        atomicAdd(&sc->edge_sum, es);
        atomicAdd(&sc->area, ar);
    }
}

// clear[c] for one (tiny_step) value; see DESIGN.md "fast-path equivalence" for the derivation.
//   reach R = (8*rtol + 64*eps*(S/hmin_c)^2) * Lmax      (how far outside a cell its tolerant test can pass)
//   clear_c = 8 * R / sigma_c ; stored NEGATIVE for cells with a vertex inside the bounding-box band (the fast path
//   then also checks that the re-location points are not `inboundary`), +inf for degenerate cells (always literal)
__device__ __forceinline__ double cell_hmin(const DevMesh &m, const CellRec &r, int c) {
    double lmax = 0.0;
    for (int k = 0; k < 3; ++k) lmax = fmax(lmax, m.edges[3 * c + k].len);
    double area2 = fabs((r.vx[1] - r.vx[0]) * (r.vy[2] - r.vy[0]) - (r.vx[2] - r.vx[0]) * (r.vy[1] - r.vy[0]));
    return area2 / lmax;
}

// reach of every cell, max-reduced onto its nodes (so a cell can take the max over its whole vertex star)
__global__ void k_node_reach(DevMesh m, const CellRec *cells, const MeshScalars *sc, float *node_reach) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m.n_cells) return;
    double hmin = cell_hmin(m, cells[c], c);
    double ratio = sc->smax / hmin;
    double reach = (8.0 * kRtol + 64.0 * 2.220446049250313e-16 * ratio * ratio) * sc->lmax;
    float rf = (float)reach;
    if (!(rf >= reach)) rf = nextafterf(rf, INFINITY);
    if (!(hmin > 0.0) || !isfinite(reach)) rf = INFINITY;
    for (int k = 0; k < 3; ++k) atomicMax((unsigned *)&node_reach[m.cell_nodes[3 * c + k]], __float_as_uint(rf));
}

__global__ void k_finalize_clear(DevMesh m, CellRec *cells, HalfEdge *he, const float *qual, const float *bdist,
                                 const MeshScalars *sc, const float *node_reach, double tiny, double lmin) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m.n_cells) return;
    const CellRec &r = cells[c];
    double hmin = cell_hmin(m, r, c);
    double reach = 0.0;
    for (int k = 0; k < 3; ++k) reach = fmax(reach, (double)node_reach[m.cell_nodes[3 * c + k]]);
    double clear = 8.0 * reach * (double)qual[c] * 1.001;
    bool boundary = !((double)bdist[c] > 16.0 * tiny + 1e-12 * sc->smax);
    float cf = (float)clear;
    if (!(cf >= clear)) cf = nextafterf(cf, INFINITY);
    if (!isfinite(clear) || !(hmin > 0.0))
        cf = INFINITY;
    else if (boundary)
        cf = -cf;
    cells[c].clear = cf;
    // chord >= d * sin(gamma) >= d * sigma for a lone vertex at distance d from the track line (the cheap filter of k_march, march.cuh)
    double c2 = lmin * 1.001 * (double)qual[c];
    float c2f = (float)c2;
    if (!(c2f >= c2)) c2f = nextafterf(c2f, INFINITY);
    if (!isfinite(c2)) c2f = INFINITY;
    for (int k = 0; k < 3; ++k) {
        he[3 * c + k].clear = cf;
        he[3 * c + k].clear2 = c2f;
    }
}

// twin[3c+k]: where a track that leaves cell c through edge k = (v_k, v_k+1) enters the neighbour
__global__ void k_twins(int n_cells, const int *cell_nodes, const int *nbr, int *twin) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= 3 * (int64_t)n_cells) return;
    int c = (int)(t / 3), k = (int)(t % 3);
    int n1 = nbr[t];
    int enc = -1;
    if (n1 >= 0) {
        int a = cell_nodes[3 * c + k], b = cell_nodes[3 * c + (k + 1) % 3];
        const int *nn = &cell_nodes[3 * n1];
        for (int kk = 0; kk < 3; ++kk) {
            int a2 = nn[kk], b2 = nn[(kk + 1) % 3];
            if (a2 == b && b2 == a) enc = ((3 * n1 + kk) << 3) | (kk << 1) | 1;  // opposite order (consistently oriented pair)
            if (a2 == a && b2 == b) enc = ((3 * n1 + kk) << 3) | (kk << 1) | 0;
        }
    }
    twin[t] = enc;
}

__global__ void k_half_edges(DevMesh m, const CellRec *cells, const int *twin, HalfEdge *he) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= 3 * (int64_t)m.n_cells) return;
    int c = (int)(t / 3), k = (int)(t % 3);
    int k1 = (k + 1) % 3, k2 = (k + 2) % 3;
    const CellRec &r = cells[c];
    HalfEdge h;
    h.ax = r.vx[k2];
    h.ay = r.vy[k2];
    h.tw1 = twin[3 * c + k1];
    h.tw2 = twin[3 * c + k2];
    h.clear = INFINITY;
    h.clear2 = INFINITY;
    he[t] = h;
}

// ---- uniform node grid -------------------------------------------------------------------------
__device__ __forceinline__ int grid_bin(const DevMesh &m, double x, double y) {
    int bx = (int)floor((x - m.g0x) * m.ginv);
    int by = (int)floor((y - m.g0y) * m.ginv);
    bx = min(max(bx, 0), m.gx - 1);
    by = min(max(by, 0), m.gy - 1);
    return by * m.gx + bx;
}

__global__ void k_grid_count(DevMesh m, int *counts) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m.n_nodes) return;
    double2 p = m.xy[i];
    atomicAdd(&counts[grid_bin(m, p.x, p.y)], 1);
}

__global__ void k_grid_fill(DevMesh m, const int *ptrs, int *cursor, int *nodes) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m.n_nodes) return;
    double2 p = m.xy[i];
    int b = grid_bin(m, p.x, p.y);
    int pos = atomicAdd(&cursor[b], 1);
    nodes[ptrs[b] + pos] = i;
}

// ---- cheap point location for the seeds of the sub-track chunks (k_seed) ------------------------------------------------------
// A seed only has to name SOME cell the serial walk pushes near the nominal seed point (DESIGN.md "chunks": exactness never
// depends on the seed, only efficiency does), so it does not need the reference's find_element with its nearest-node search
// and tolerant barycentric tests: jump to a cell whose centroid lies in the point's grid bin and walk towards the point through
// the neighbour table, deciding every step from the signs of the three edge functions (no division).  Returns the cell that
// contains (x, y), or -1 when the walk does not get there (empty bin, hole, too far): the caller falls back to find_element.
__global__ void k_cell_bins(DevMesh m, const CellRec *cells, int *cell_bin) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= m.n_cells) return;
    const CellRec &r = cells[c];
    const double cx = (r.vx[0] + r.vx[1] + r.vx[2]) / 3.0, cy = (r.vy[0] + r.vy[1] + r.vy[2]) / 3.0;
    atomicMax(&cell_bin[grid_bin(m, cx, cy)], c);
}

__device__ __forceinline__ int locate_by_walk(const DevMesh &m, double x, double y) {
    int c = m.cell_bin[grid_bin(m, x, y)];
    for (int it = 0; it < 16 && c >= 0; ++it) {
        const CellRec &r = m.cells[c];
        const double x1 = r.vx[0], y1 = r.vy[0], x2 = r.vx[1], y2 = r.vy[1], x3 = r.vx[2], y3 = r.vy[2];
        const double d = (x2 - x1) * (y3 - y1) - (x3 - x1) * (y2 - y1);  // twice the signed area: orientation of the stored nodes
        double e0 = (x2 - x1) * (y - y1) - (x - x1) * (y2 - y1);         // edge k = (v_k, v_k+1): same sign as d on the inner side
        double e1 = (x3 - x2) * (y - y2) - (x - x2) * (y3 - y2);
        double e2 = (x1 - x3) * (y - y3) - (x - x3) * (y1 - y3);
        if (d < 0.0) {
            e0 = -e0;
            e1 = -e1;
            e2 = -e2;
        }
        int k = -1;
        double mn = 0.0;
        if (e0 < mn) {
            mn = e0;
            k = 0;
        }
        if (e1 < mn) {
            mn = e1;
            k = 1;
        }
        if (e2 < mn) k = 2;
        if (k < 0) return c;
        c = r.nbr[k];
    }
    return -1;
}

// ------------------------------------------------------------------------------------------------
// literal point location
// ------------------------------------------------------------------------------------------------

// largest `k` of segmentize!(t; k) (src/mesh.jl:123): the candidate list of the exact kNN search is a fixed-size array;
// rt_segmentize rejects larger values with RT_ERR_ARG (the reference itself has no limit)
constexpr int kMaxK = 32;

struct KBest {
    double d2[kMaxK];
    int id[kMaxK];
    int n, k;
};

__device__ __forceinline__ bool cand_less(double d2a, int ida, double d2b, int idb) {
    return d2a < d2b || (d2a == d2b && ida < idb);
}

__device__ __forceinline__ void kbest_insert(KBest &s, double d2, int id) {
    if (s.n == s.k && !cand_less(d2, id, s.d2[s.k - 1], s.id[s.k - 1])) return;
    int pos = s.n < s.k ? s.n : s.k - 1;
    while (pos > 0 && cand_less(d2, id, s.d2[pos - 1], s.id[pos - 1])) {
        s.d2[pos] = s.d2[pos - 1];
        s.id[pos] = s.id[pos - 1];
        --pos;
    }
    s.d2[pos] = d2;
    s.id[pos] = id;
    if (s.n < s.k) s.n++;
}

// Exact k nearest nodes of (x, y) (ties: lowest node id), skipping node `skip` -- what the reference asks of
// nn(kdtree, x) (src/mesh.jl:107) and knn(kdtree, x, k, true, skip) (src/mesh.jl:123). Ring search: after ring r every
// unvisited node is farther than the distance to the border of the visited block.
__device__ RT_SLOWPATH_INLINE void knn_query(const DevMesh &m, double x, double y, int skip, KBest &s) {
    s.n = 0;
    int bx = (int)floor((x - m.g0x) * m.ginv);
    int by = (int)floor((y - m.g0y) * m.ginv);
    bx = min(max(bx, 0), m.gx - 1);
    by = min(max(by, 0), m.gy - 1);
    const double slack = 1e-7 * m.gh;
    int rmax = max(m.gx, m.gy);
    for (int r = 0; r <= rmax; ++r) {
        int x0 = bx - r, x1 = bx + r, y0 = by - r, y1 = by + r;
        for (int iy = max(y0, 0); iy <= min(y1, m.gy - 1); ++iy) {
            bool edge_row = (iy == y0 || iy == y1);
            int step = edge_row ? 1 : (x1 - x0);
            if (step == 0) step = 1;
            for (int ix = x0; ix <= x1; ix += step) {
                if (ix < 0 || ix >= m.gx) continue;
                int b = iy * m.gx + ix;
                for (int q = m.grid_ptrs[b]; q < m.grid_ptrs[b + 1]; ++q) {
                    int id = m.grid_nodes[q];
                    if (id == skip) continue;
                    double2 p = m.xy[id];
                    double dx = x - p.x, dy = y - p.y;
                    kbest_insert(s, dx * dx + dy * dy, id);
                }
            }
        }
        bool covers = (x0 <= 0 && y0 <= 0 && x1 >= m.gx - 1 && y1 >= m.gy - 1);
        if (covers) break;
        if (s.n == s.k) {
            double bound = INFINITY;
            if (x0 > 0) bound = fmin(bound, x - (m.g0x + x0 * m.gh));
            if (x1 < m.gx - 1) bound = fmin(bound, (m.g0x + (x1 + 1) * m.gh) - x);
            if (y0 > 0) bound = fmin(bound, y - (m.g0y + y0 * m.gh));
            if (y1 < m.gy - 1) bound = fmin(bound, (m.g0y + (y1 + 1) * m.gh) - y);
            bound -= slack;
            if (bound > 0.0 && s.d2[s.k - 1] < bound * bound) break;
        }
    }
}

// point_in_triangle  src/mesh.jl:158-176 ; lambda = R \ r by the StaticArrays 3x3 closed form
__device__ __forceinline__ bool point_in_triangle(const DevMesh &m, int cell, double x, double y) {
    // vertex coordinates from the cell record (two adjacent 32-B sectors; the same values as xy[cell_nodes[3*cell + k]], which
    // cost two dependent gather levels)
    const CellRec &r = m.cells[cell];
    double x1 = r.vx[0], y1 = r.vy[0], x2 = r.vx[1], y2 = r.vy[1], x3 = r.vx[2], y3 = r.vy[2];
    double d = x1 * (y2 - y3) + y1 * (x3 - x2) + (x2 * y3 - y2 * x3);
    double l1 = ((y2 - y3) * x + (x3 - x2) * y + (x2 * y3 - x3 * y2)) / d;
    double l2 = ((y3 - y1) * x + (x1 - x3) * y + (x3 * y1 - x1 * y3)) / d;
    double l3 = ((y1 - y2) * x + (x2 - x1) * y + (x1 * y2 - x2 * y1)) / d;
    const double lo = 0.0 - kRtol, hi = 1.0 + kRtol;
    return (lo <= l1 && l1 <= hi) && (lo <= l2 && l2 <= hi) && (lo <= l3 && l3 <= hi);
}

// the same test on three explicit nodes (mixed meshes: no CellRec table)
__device__ __forceinline__ bool point_in_triangle_nodes(const DevMesh &m, int n1, int n2, int n3, double x, double y) {
    const double2 a = m.xy[n1], b = m.xy[n2], c = m.xy[n3];
    const double x1 = a.x, y1 = a.y, x2 = b.x, y2 = b.y, x3 = c.x, y3 = c.y;
    double d = x1 * (y2 - y3) + y1 * (x3 - x2) + (x2 * y3 - y2 * x3);
    double l1 = ((y2 - y3) * x + (x3 - x2) * y + (x2 * y3 - x3 * y2)) / d;
    double l2 = ((y3 - y1) * x + (x1 - x3) * y + (x3 * y1 - x1 * y3)) / d;
    double l3 = ((y1 - y2) * x + (x2 - x1) * y + (x1 * y2 - x2 * y1)) / d;
    const double lo = 0.0 - kRtol, hi = 1.0 + kRtol;
    return (lo <= l1 && l1 <= hi) && (lo <= l2 && l2 <= hi) && (lo <= l3 && l3 <= hi);
}

// point_in_element (src/mesh.jl:148-150) dispatched on the number of nodes: triangles as above; 4-node cells by
// point_in_quadrangle (src/mesh.jl:184-201): the four triangles (k, k+1, k+2) of the stored cycle
__device__ __noinline__ bool point_in_cell_generic(const DevMesh &m, int cell, double x, double y) {
    const int b = m.cell_ptrs[cell], nn = m.cell_ptrs[cell + 1] - b;
    const int *nid = m.cell_nodes + b;
    if (nn == 3) return point_in_triangle_nodes(m, nid[0], nid[1], nid[2], x, y);
    for (int i = 0; i < 4; ++i)
        if (point_in_triangle_nodes(m, nid[i], nid[(i + 1) & 3], nid[(i + 2) & 3], x, y)) return true;
    return false;
}

// MIXED is a compile-time switch: only the kernels that walk mixed meshes (k_walk<*, true>) contain the generic cell code, the
// triangle kernels are compiled exactly as before
template <bool MIXED = false>
__device__ __forceinline__ int scan_node_cells(const DevMesh &m, int node, double x, double y) {
    for (int q = m.nc_ptrs[node]; q < m.nc_ptrs[node + 1]; ++q) {
        int cell = m.nc_data[q];
        if (MIXED ? point_in_cell_generic(m, cell, x, y) : point_in_triangle(m, cell, x, y)) return cell;
    }
    return -1;
}

// find_element(mesh, x, k)  src/mesh.jl:103-146 ; returns 0-based cell or -1
template <bool MIXED = false>
__device__ RT_SLOWPATH_INLINE int find_element(const DevMesh &m, double x, double y, int k, unsigned long long *nq) {
    KBest s;
    s.k = 1;
    knn_query(m, x, y, -1, s);
    if (nq) nq[0]++;
    int nn = s.id[0];
    int c = scan_node_cells<MIXED>(m, nn, x, y);
    if (c >= 0) return c;
    s.k = min(k, kMaxK);  // (k <= kMaxK is checked by rt_segmentize)
    knn_query(m, x, y, nn, s);
    if (nq) nq[1]++;
    for (int i = 0; i < s.n; ++i) {
        c = scan_node_cells<MIXED>(m, s.id[i], x, y);
        if (c >= 0) return c;
    }
    return -1;
}

// inboundary(mesh, x, atol)  src/mesh.jl:91-95
__device__ __forceinline__ bool inboundary(const DevMesh &m, double x, double y, double atol) {
    double rtol = atol > 0.0 ? 0.0 : kRtol;
    return isapprox(x, m.bbmax[0], atol, rtol) || isapprox(x, m.bbmin[0], atol, rtol) ||
           isapprox(y, m.bbmax[1], atol, rtol) || isapprox(y, m.bbmin[1], atol, rtol);
}

// intersections(mesh, cell, track)  src/intersection.jl:34-119 (triangles: 3 edges, at most 3 hits).
// Returns 0, or 4 (RT_TRACK_UNDEF) when the 3-hit selection never assigns x_int1. e_p/e_q: local edges of p and q.
// mixed meshes: the reference's loop over the edges (i, i+1) of the stored node cycle of a 3- or 4-node cell, general_form of
// every edge evaluated on the spot like the reference does, at most four hits (src/intersection.jl:42-44), the farthest pair when
// there are three or four (:81-95).  Returns 0, or 4 (RT_TRACK_UNDEF) when that selection never assigns x_int1.
__device__ __noinline__ int intersections_generic(const DevMesh &m, int cell, const Line &trk, bool phi_lt_half_pi, P2 &p, P2 &q, int &e_p,
                                                  int &e_q) {
    const int b = m.cell_ptrs[cell], nn = m.cell_ptrs[cell + 1] - b;
    P2 ip[4];
    int ie[4];
    int n_int = 0;
    bool parallel_found = false;
    for (int i = 0; i < nn; ++i) {
        const int j = (i == nn - 1) ? 0 : i + 1;
        const double2 a = m.xy[m.cell_nodes[b + i]], c = m.xy[m.cell_nodes[b + j]];
        const P2 p1{a.x, a.y}, p2{c.x, c.y};
        const Line L = general_form(p1, p2);
        P2 X;
        if (intersection(trk, L, X)) {
            parallel_found = true;
            continue;
        }
        if (!point_in_segment(p1, p2, norm2(p1.x - p2.x, p1.y - p2.y), X)) continue;
        if (n_int < 4) {
            ip[n_int] = X;
            ie[n_int] = i;
        }
        n_int++;
    }
    e_p = e_q = -1;
    if (n_int == 3 || n_int == 4) {
        double l = 0.0;
        int s1 = -1, s2 = -1;
        for (int i = 2; i <= n_int; ++i)  // for i in 2:n_int, j in i:n_int: x1 = pts[i-1], x2 = pts[j]
            for (int j = i; j <= n_int; ++j) {
                const double li = norm2(ip[i - 2].x - ip[j - 1].x, ip[i - 2].y - ip[j - 1].y);
                if (li > l) {
                    s1 = i - 2;
                    s2 = j - 1;
                    l = li;
                }
            }
        if (s1 < 0) return 4;
        const bool first = order_first(phi_lt_half_pi, ip[s1], ip[s2]);
        p = first ? ip[s1] : ip[s2];
        q = first ? ip[s2] : ip[s1];
        e_p = first ? ie[s1] : ie[s2];
        e_q = first ? ie[s2] : ie[s1];
        return 0;
    }
    if (n_int == 2) {
        if (!parallel_found && isapprox_pt(ip[0], ip[1])) {
            p = ip[0];
            q = ip[1];
            e_p = ie[0];
            e_q = ie[1];
            return 0;
        }
        const bool first = order_first(phi_lt_half_pi, ip[0], ip[1]);
        p = first ? ip[0] : ip[1];
        q = first ? ip[1] : ip[0];
        e_p = first ? ie[0] : ie[1];
        e_q = first ? ie[1] : ie[0];
        return 0;
    }
    p.x = p.y = q.x = q.y = 0.0;
    return 0;
}

template <bool MIXED = false>
__device__ RT_SLOWPATH_INLINE int intersections(const DevMesh &m, int cell, const Line &trk, bool phi_lt_half_pi, P2 &p, P2 &q,
                                          int &e_p, int &e_q) {
    if (MIXED) return intersections_generic(m, cell, trk, phi_lt_half_pi, p, q, e_p, e_q);
    const CellRec &r = m.cells[cell];
    P2 ip[3];
    int ie[3];
    int n_int = 0;
    bool parallel_found = false;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        int j = (i == 2) ? 0 : i + 1;
        const EdgeRec e = m.edges[3 * cell + i];
        Line L;
        L.a = e.a;
        L.b = e.b;
        L.c = e.c;
        P2 X;
        bool par = intersection(trk, L, X);
        if (par) {
            parallel_found = true;
            continue;
        }
        P2 p1{r.vx[i], r.vy[i]}, p2{r.vx[j], r.vy[j]};
        if (!point_in_segment(p1, p2, e.len, X)) continue;
        ip[n_int] = X;
        ie[n_int] = i;
        n_int++;
    }
    e_p = e_q = -1;
    if (n_int == 3) {
        double l = 0.0;
        int s1 = -1, s2 = -1;
        // for i in 2:n, j in i:n: x1 = pts[i-1], x2 = pts[j]  -> pairs (1,2) (1,3) (2,3)
        const int pa[3] = {0, 0, 1}, pb[3] = {1, 2, 2};
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            double li = norm2(ip[pa[t]].x - ip[pb[t]].x, ip[pa[t]].y - ip[pb[t]].y);
            if (li > l) {
                s1 = pa[t];
                s2 = pb[t];
                l = li;
            }
        }
        if (s1 < 0) return 4;
        bool first = order_first(phi_lt_half_pi, ip[s1], ip[s2]);
        p = first ? ip[s1] : ip[s2];
        q = first ? ip[s2] : ip[s1];
        e_p = first ? ie[s1] : ie[s2];
        e_q = first ? ie[s2] : ie[s1];
        return 0;
    }
    if (n_int == 2) {
        if (!parallel_found && isapprox_pt(ip[0], ip[1])) {
            p = ip[0];
            q = ip[1];
            e_p = ie[0];
            e_q = ie[1];
            return 0;
        }
        bool first = order_first(phi_lt_half_pi, ip[0], ip[1]);
        p = first ? ip[0] : ip[1];
        q = first ? ip[1] : ip[0];
        e_p = first ? ie[0] : ie[1];
        e_q = first ? ie[1] : ie[0];
        return 0;
    }
    p.x = p.y = q.x = q.y = 0.0;
    return 0;
}

}  // namespace rt
