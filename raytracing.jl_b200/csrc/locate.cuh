// locate.cuh -- point location outside the walk: find_element(mesh, x, k) (src/mesh.jl:103-146) for a batch of points
// (rt_find_elements).  The answer is the walk's own find_element<MIXED> (mesh_dev.cuh): the first cell that passes the tolerant
// barycentric test (point_in_quadrangle on 4-node cells) around the nearest node, in Gridap's order, then around the k nearest
// other nodes.  locate_by_walk is NOT used: on shared edges and vertices it may name another of the cells that contain the point.
#pragma once
#include "mesh_dev.cuh"

namespace rt {

constexpr int kLocateThreads = 256;

// One thread per point.  element[i] = 1-based cell or -1 (no cell passes, like the reference).  *knn_points += the points of the
// block that entered the k-nearest-node branch (src/mesh.jl:123): a block count, one atomic per block.
template <bool MIXED>
__global__ void __launch_bounds__(kLocateThreads) k_find_elements(DevMesh m, long long n, const double2 *__restrict__ xy, int k,
                                                                  int *__restrict__ element, unsigned long long *knn_points) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    int knn = 0;
    if (i < n) {
        const double2 p = xy[i];
        unsigned long long nq[2] = {0, 0};  // nearest-node / k-nearest queries of this point
        const int c = find_element<MIXED>(m, p.x, p.y, k, nq);
        element[i] = c >= 0 ? c + 1 : -1;
        knn = nq[1] != 0;
    }
    const int block_knn = __syncthreads_count(knn);
    if (threadIdx.x == 0 && block_knn) atomicAdd(knn_points, (unsigned long long)block_knn);
}

}  // namespace rt
