/* The CPU oracle's find_element (orc_find_element, src/mesh.jl:103-146) for a batch of points in one call: tests pin the device's
 * rt_find_elements on it for up to millions of points, where one ctypes call per point would dominate.  Also counts the points that
 * enter the k-nearest-node branch (src/mesh.jl:123): those where no cell around the nearest node passes (src/mesh.jl:107-121). */
#include <stdint.h>

#include "../oracle/rt_oracle.h"

/* xy = x0,y0,x1,y1,... ; node_cell_ptrs / node_cell_data: the 1-based vertex -> cells table the oracle mesh was built with */
int64_t loc_find_elements(const orc_mesh *m, const int32_t *node_cell_ptrs, const int32_t *node_cell_data, int64_t n,
                          const double *xy, int k, int32_t *out) {
    int64_t n_knn = 0;
    for (int64_t i = 0; i < n; ++i) {
        const double x = xy[2 * i], y = xy[2 * i + 1];
        out[i] = orc_find_element(m, x, y, k);
        const int32_t nn = orc_nn(m, x, y);
        int found = 0;
        for (int32_t q = node_cell_ptrs[nn - 1]; q < node_cell_ptrs[nn] && !found; ++q)
            found = orc_point_in_element(m, node_cell_data[q - 1], x, y);
        n_knn += !found;
    }
    return n_knn;
}
