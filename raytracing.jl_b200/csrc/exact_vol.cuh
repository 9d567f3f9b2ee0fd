// exact_vol.cuh -- fill_volumes in the reference's order (RT_SEG_EXACT_VOLUMES).
// src/trackgenerator.jl:371-386 starts every volume at zero and adds delta_eff[azim] * len over the tracks in uid order and the
// segments of a track in walk order.  The fused path adds the same products with atomicAdd, so the last bits of a sum follow the
// order in which warps retire.  Here every segment of a batch writes one (element - 1, delta_eff * len) pair in segment order
// (k_exact_contrib), a stable radix sort groups the pairs by element without reordering an element's terms, k_exact_runs finds
// each element's run in the sorted pairs, and k_exact_fold continues one running sum per element through its run with plain `+`.
// Batches come in uid order, so folding them one after the other onto the same sums is the reference's loop.
#pragma once
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>

namespace rt {

constexpr int kExactThreads = 256;

// one warp per track of the batch (offsets are per track, and a track's azimuth is constant).  The product is rounded on its
// own: it is stored, and only the fold adds it (the build's -fmad=false keeps any a*b+c apart as well).
__global__ void __launch_bounds__(kExactThreads) k_exact_contrib(const long long *offsets, long long trk_begin, long long trk_end,
                                                                  long long offset_base, const int *azim, const double *delta_eff,
                                                                  const double *len, const int *elem, int *key, double *val) {
    const long long t = trk_begin + (blockIdx.x * (long long)blockDim.x + threadIdx.x) / 32;
    const int lane = threadIdx.x & 31;
    if (t >= trk_end) return;
    const long long o0 = offsets[t] - offset_base, o1 = offsets[t + 1] - offset_base;
    const double d = delta_eff[azim[t]];
    for (long long i = o0 + lane; i < o1; i += 32) {
        key[i] = elem[i] - 1;
        val[i] = d * len[i];  // volumes[i] += delta_s[a]*l, src/trackgenerator.jl:382
    }
}

// run bounds of every element in the sorted keys (start = end = 0 where an element has no pair: cleared before)
__global__ void __launch_bounds__(kExactThreads) k_exact_runs(const int *key, long long n, int n_cells, long long *start,
                                                               long long *end) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int k = key[i];
    if ((unsigned)k >= (unsigned)n_cells) return;
    if (i == 0 || key[i - 1] != k) start[k] = i;
    if (i == n - 1 || key[i + 1] != k) end[k] = i + 1;
}

// one thread per element: acc[e] continues through the element's run, in order
__global__ void __launch_bounds__(kExactThreads) k_exact_fold(int n_cells, const long long *start, const long long *end,
                                                               const double *val, double *acc) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_cells) return;
    double s = acc[e];
    for (long long i = start[e], i1 = end[e]; i < i1; ++i) s = s + val[i];
    acc[e] = s;
}

// The message of the rank-order chain of rt_volumes: n_cells running sums, then the number of ranks whose rt_segmentize failed,
// the number of ranks whose uid_begin was not their predecessor's uid_end, and the sender's uid_end.  One thread stamps this rank.
__global__ void k_chain_stamp(double *msg, int n_cells, int check_order, double uid_begin, double uid_end, double failed) {
    if (check_order && msg[n_cells + 2] != uid_begin) msg[n_cells + 1] += 1.0;
    msg[n_cells] += failed;
    msg[n_cells + 2] = uid_end;
}

}  // namespace rt
