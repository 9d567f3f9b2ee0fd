// sweep.cuh -- what a transport sweep (NeutronTransport.jl, reference README.md:9,125-136) consumes besides the Segment
// records, produced and kept on the device (SURVEY 8f-1):
//   * azimuthal weights  init_weights!  (src/azimuthal_quad.jl:35-53)
//   * optical lengths    tau[s][g] = sigma_t[element(s)][g] * len(s)   -- the `tau::Vector{T}` field of every Segment
//     (src/segment.jl:27), which the reference leaves empty for the transport code to fill
#pragma once
#include "geom.cuh"

namespace rt {

// one thread per i in 1..N4 (0-based here); phi has N2 = 2*N4 entries; omega[i] = omega[N2-1-i]
__global__ void k_weights(int n2, const double *phi, double *omega) {
    const int n4 = n2 / 2;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // 0-based: reference i = this + 1
    if (i >= n4) return;
    double v;
    if (i == 0)  // isone(i), tested first (src/azimuthal_quad.jl:41)
        v = phi[1] - phi[0];
    else if (i == n4 - 1)
        v = kPi - phi[i] - phi[i - 1];
    else
        v = phi[i + 1] - phi[i - 1];
    v = v / (4.0 * kPi);
    omega[i] = v;
    omega[n2 - 1 - i] = v;
}

// segment-major (layout 0: tau[s*G + g], the concatenation of the reference's per-segment vectors) or group-major
// (layout 1: tau[g*S + s], unit-stride over segments for a sweep that runs one group at a time).
// BY_REGION: sigma_t is the small n_regions x n_groups table of a transport code's materials, indexed through the region map
// (rt_set_regions, 1-based); it stays in L1 / L2 where the per-cell table is one random HBM row per segment.  The product is the
// same IEEE multiplication, so tau is bit-equal to the per-cell call with the table expanded cell by cell.  (`region` comes last:
// the parameter offsets, and so the code, of the per-cell instantiation are those of the kernel before the switch.)
template <bool BY_REGION>
__global__ void k_tau(long long n_seg, int n_groups, const double *__restrict__ len, const int *__restrict__ element,
                      const double *__restrict__ sigma_t /* n_cells (n_regions) x n_groups */, int layout, double *__restrict__ tau,
                      const int *__restrict__ region) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n_seg * n_groups) return;
    long long s;
    int g;
    if (layout == 0) {
        s = i / n_groups;
        g = (int)(i - s * n_groups);
    } else {
        g = (int)(i / n_seg);
        s = i - (long long)g * n_seg;
    }
    int e = element[s] - 1;
    if constexpr (BY_REGION) e = region[e] - 1;
    tau[i] = sigma_t[(long long)e * n_groups + g] * len[s];
}

// ---- region map (rt_set_regions, rt_region_volumes) -----------------------------------------------------------------------
// One pass over the map: the first cell whose region is outside [1, n_regions] (atomicMin on its index; *first_bad starts at
// n_cells), and the (region - 1, cell) pairs whose stable sort by region gives the region -> cells order.
__global__ void k_region_check(int n_cells, int n_regions, const int *__restrict__ region, int *__restrict__ first_bad,
                               int *__restrict__ key, int *__restrict__ cell) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells) return;
    const int r = region[c];
    if (r < 1 || r > n_regions) atomicMin(first_bad, c);
    key[c] = r - 1;
    cell[c] = c;
}

// per-cell values in region order (order: the cell ids sorted stably by region), for k_exact_runs / k_exact_fold
__global__ void k_region_gather(int n_cells, const int *__restrict__ order, const double *__restrict__ v, double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_cells) return;
    out[i] = v[order[i]];
}

// element_volume(mesh, node_ids) = 1/2 * abs((x2 - x1) x (x3 - x1))  (src/trackgenerator.jl:402-411): the exact cell areas the
// reference computes into `volumes2` and then discards (its volume correction is a TODO, src/trackgenerator.jl:388-397).
// Gridap's cross of two 2-vectors: a[1]*b[2] - a[2]*b[1].
__global__ void k_element_volumes(int n_cells, const int *__restrict__ cell_nodes, const double2 *__restrict__ xy, double *__restrict__ area) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells) return;
    const double2 x1 = xy[cell_nodes[3 * c]], x2 = xy[cell_nodes[3 * c + 1]], x3 = xy[cell_nodes[3 * c + 2]];
    const double ax = x2.x - x1.x, ay = x2.y - x1.y, bx = x3.x - x1.x, by = x3.y - x1.y;
    area[c] = 0.5 * fabs(ax * by - ay * bx);
}

// The correction the reference announces ("correct volumes by changing segment lengths", src/trackgenerator.jl:388): every
// segment length of element e is scaled by area[e] / traced_volume[e], so that the traced volumes (src/trackgenerator.jl:371-386)
// of the corrected segments equal the exact areas.  Elements no track crosses (traced volume 0) keep factor 1.
__global__ void k_volume_factors(int n_cells, const double *__restrict__ area, const double *__restrict__ vol, double *__restrict__ factor) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells) return;
    const double v = vol[c];
    factor[c] = v > 0.0 ? area[c] / v : 1.0;
}
__global__ void k_scale_lengths(long long n_seg, const int *__restrict__ element, const double *__restrict__ factor, double *__restrict__ len) {
    const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    len[s] = len[s] * factor[element[s] - 1];
}

// ---- compact download of the Segment records (rt_segments_download_compact) ------------------------------------------------
// Inside a track the entry point of a segment IS the exit point of the one before it (the walk re-locates from q, and on generic
// transitions the two are the same bits, eval3.cuh), so `p` does not have to cross PCIe: the host rebuilds p[i] = q[i-1] and
// patches the few positions where that does not hold -- the first segment of every track and the neighbourhood of literal
// records.  This kernel lists those positions: (index, px, py) of every resident segment whose p differs, in any bit, from the q of
// its predecessor in the columns.  One thread per segment; the list is unordered (the host sorts the ~0.2 % it receives).
__global__ void k_p_exceptions(long long n_seg, const double *__restrict__ px, const double *__restrict__ py, const double *__restrict__ qx,
                               const double *__restrict__ qy, long long cap, unsigned long long *__restrict__ count, long long *__restrict__ idx,
                               double *__restrict__ epx, double *__restrict__ epy) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n_seg) return;
    const double x = px[i], y = py[i];
    bool differs = i == 0;
    if (!differs) differs = __double_as_longlong(x) != __double_as_longlong(qx[i - 1]) || __double_as_longlong(y) != __double_as_longlong(qy[i - 1]);
    if (differs) {
        const unsigned long long k = atomicAdd(count, 1ULL);
        if ((long long)k < cap) {
            idx[k] = i;
            epx[k] = x;
            epy[k] = y;
        }
    }
}

}  // namespace rt
