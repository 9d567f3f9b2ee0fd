// topo.cuh -- sign-test walks of the half-edge graph.
//
// A Segment(p, q, l, element) depends only on (track, cell): intersections() uses the track's infinite line
// (src/intersection.jl:60).  So the serial part of _segmentize_track! (src/track.jl:106-178) is only the ORDER in which
// cells are accepted; the geometry of every accepted cell can be evaluated independently afterwards.
//
//   k_topo     count pass of the hybrid pipeline: walks the half-edge graph deciding each transition from the SIGNS of the
//                  signed distances of the cell's vertices from the track line (two multiply-adds per step, no division, no
//                  square root), under the same clearance test as the sequential fast path (walk.cuh); everything that test
//                  does not cover runs the literal walk of the reference, exactly as in walk.cuh.  (k_march, march.cuh, is the
//                  same walk for the single-walk pipeline: it also records every accepted cell.)
//   k_track_status per track: the reference's length check (src/track.jl:171-175) on the accumulated segment lengths.
#pragma once
#include "walk.cuh"

namespace rt {

constexpr int kTopoThreads = 128;
#ifndef RT_TOPO_MIN_BLOCKS
#define RT_TOPO_MIN_BLOCKS 8
#endif

// (the pool records are read back by k_eval3 within the same call: no eviction hint, they should stay in L2 if they fit)
__device__ __forceinline__ void stg256_plain_i(void *p, const int *v) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]),
                 "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

// exit point of cell `c` through its local edge k: the reference's intersection() with that edge's line
__device__ __forceinline__ P2 exit_point(const DevMesh &m, const Line &trk, int c, int k) {
    const EdgeRec e = m.edges[3 * c + k];
    P2 X;
    intersection(trk, Line{e.a, e.b, e.c}, X);
    return X;
}

// the count pass of the hybrid pipeline (see the top of this file)
__global__ void __launch_bounds__(kTopoThreads, RT_TOPO_MIN_BLOCKS) k_topo(const __grid_constant__ WalkParams P) {
    const unsigned FULL = 0xffffffffu;
    const DevMesh &m = P.m;
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
    // last pushed cell and the local edge it was left through (-1: unknown); (qx, qy) is its exit point when q_valid
    int cur = -1, cur_kout = -1, enc = -1;
    bool f = false, clean = false, q_valid = false;
    double s1 = 0, s2 = 0, qx = 0, qy = 0;
    float clearA = INFINITY;
    int stop_cell = -1, limit = P.max_iter, n_litpush = 0;
    const bool literal_only = (P.flags & 1u) != 0;
    bool active = false;
    const unsigned long long pol_keep = l2_policy_keep();
    constexpr double kKappa = 1.0 / RT_KAPPA_INV;  // smallest sine of a crossing angle the cheap filter accepts
    bool cheap_ok = false;                 // x-ordering of entry/exit is decided by the track direction, beyond rounding
    double ang_thr = 0.0;

    auto arm = [&](int e, int e_q) {
        const CellRec &r = m.cells[e];
        cur = e;
        cur_kout = e_q;
        clearA = fabsf(r.clear);
        double v0 = ta * r.vx[0] + tb * r.vy[0] + tc, v1 = ta * r.vx[1] + tb * r.vy[1] + tc, v2 = ta * r.vx[2] + tb * r.vy[2] + tc;
        double thr = g * (double)clearA;
        s1 = e_q == 0 ? v0 : (e_q == 1 ? v1 : v2);
        s2 = e_q == 0 ? v1 : (e_q == 1 ? v2 : v0);
        clean = (fabs(v0) >= thr) && (fabs(v1) >= thr) && (fabs(v2) >= thr) && ((s1 > 0) != (s2 > 0));
        enc = m.twin[3 * e + e_q];
        f = (enc & 1) != 0;
    };

    if (t < P.n_tracks && t >= P.trk_begin && t < P.trk_end) {
        int n = P.ch.nch[t];
        int seed = (j < n) ? (j == 0 ? -2 : P.ch.seed_cell[cidx]) : -1;
        active = (seed != -1);
        if (active) {
            az = P.t.azim[t];
            ta = P.t.a[t];
            tb = P.t.b[t];
            tc = P.t.c[t];
            right = P.ang.phi[az] < kPi / 2;  // isless(phi, pi/2), src/intersection.jl:153
            g = sqrt(ta * ta + tb * tb);
            ang_thr = kKappa * g * P.lmax;
            // |X.x - q.x| = l*|cos phi| >= l_min*|b|/g must exceed the rounding error of both points, ~ 8*eps*S/kappa each
            cheap_ok = P.lmin * (fabs(tb) / g) > 32.0 * 2.220446049250313e-16 * P.smax / kKappa;
            if (j == 0) {
                qx = P.t.px[t];  // the literal walk starts from advance_step(track.p), src/track.jl:114
                qy = P.t.py[t];
                q_valid = true;
                mode = MODE_SLOW;
            } else {
                arm(seed, P.ch.seed_kexit[cidx]);  // k_seed verified `clean`
                qx = P.ch.seed_qx[cidx];
                qy = P.ch.seed_qy[cidx];
                q_valid = true;
                mode = (literal_only || !clean) ? MODE_SLOW : MODE_FAST;
            }
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

    auto push = [&](int e) {
        nseg += 1;
        if (nseg >= limit) {  // while i < MAX_ITER (src/track.jl:119)
            endcode = END_CAP;
            mode = MODE_DONE;
        } else if (e == stop_cell) {
            endcode = END_HANDOFF;
            mode = MODE_DONE;
        }
    };

    while (__any_sync(FULL, mode != MODE_DONE)) {
        // ------------------------------------------------------------------ FAST phase: sign tests only
#pragma unroll 1
        for (int it = 0; it < 4 * kFastBatch; ++it) {
            if (!__any_sync(FULL, mode == MODE_FAST)) break;
            if (mode != MODE_FAST) continue;
            bool ok = false;
            if (enc >= 0) {
                double ax, ay, w0, w1;
                ldg256_keep(m.he + (enc >> 3), pol_keep, ax, ay, w0, w1);
                const float clearf = __int_as_float(__double2loint(w1));
                const float clearB = fabsf(clearf);
                const double sa = ta * ax + tb * ay + tc;
                const double thr = g * (double)fmaxf(clearA, clearB);
                if ((fabs(sa) >= thr) && (fabs(s1) >= thr) && (fabs(s2) >= thr)) {
                    const bool opp1 = (sa > 0) != (s1 > 0);  // the exit edge joins the apex with the end point across the line
                    const double ks = opp1 ? s1 : s2;        // ... which is the only vertex on its side of the track line
                    const bool exit1 = (opp1 == f);
                    const int nenc = exit1 ? __double2loint(w0) : __double2hiint(w0);
                    const int h = enc >> 3;
                    const int kin = (enc >> 1) & 3;
                    int kout = kin + (exit1 ? 1 : 2);
                    kout = kout >= 3 ? kout - 3 : kout;
                    const int cellB = h / 3;
                    // The geometric conditions of the fast path (exit edge not parallel, entry ordered first, chord > l_min)
                    // hold without evaluating the chord when the lone vertex is clear2 = l_min/sigma away from the line and
                    // both crossings are steeper than kappa (DESIGN.md, "cheap filter"); otherwise they are evaluated exactly.
                    const float clear2 = __int_as_float(__double2hiint(w1));
                    // (cells of the bounding-box band, clear stored negative, always take the exact evaluation)
                    bool accept = cheap_ok && (clearf >= 0.0f) && (fabs(ks) >= g * (double)clear2) && (fabs(ks) + fabs(sa) >= ang_thr) &&
                                  (fabs(s1) + fabs(s2) >= ang_thr);
                    if (!accept) {
                        const Line trk{ta, tb, tc};
                        const EdgeRec ei = m.edges[3 * cellB + kin], eo = m.edges[3 * cellB + kout];
                        P2 pi, X;
                        const bool par_i = intersection(trk, Line{ei.a, ei.b, ei.c}, pi);
                        const bool par_o = intersection(trk, Line{eo.a, eo.b, eo.c}, X);
                        const bool kin_lt_kout = (kin == 0) || (kin == 1 && exit1);
                        const bool in_first = right ? (kin_lt_kout ? (pi.x < X.x) : !(X.x < pi.x)) : (kin_lt_kout ? (pi.x > X.x) : !(X.x > pi.x));
                        const double l = norm2(pi.x - X.x, pi.y - X.y);
                        accept = !par_i && !par_o && in_first && l > P.lmin;
                        // band cells: the re-location points must not be `inboundary` (same test as walk.cuh)
                        if (accept && clearf < 0.0f) accept = bbox_dist(m, pi.x, pi.y) > 0.25 * l + 8.0 * P.tiny;
                    }
                    if (accept) {
                        cur = cellB;
                        cur_kout = kout;
                        q_valid = false;
                        s1 = ks;
                        s2 = sa;
                        f = (exit1 == ((nenc & 1) != 0));
                        enc = nenc;
                        clearA = clearB;
                        ok = true;
                        push(cur);
                    }
                }
            }
            if (!ok) mode = MODE_SLOW;
        }
        // ------------------------------------------------------------------ LITERAL phase (until one push)
        if (mode == MODE_SLOW) {
            if (!q_valid) {  // exit point of the last fast cell: needed now by advance_step(q, tiny, phi), src/track.jl:165
                P2 X = exit_point(m, Line{ta, tb, tc}, cur, cur_kout);
                qx = X.x;
                qy = X.y;
                q_valid = true;
            }
            LitIn in{ta, tb, tc, P.tiny * P.ang.cosp[az], P.tiny * P.ang.sinp[az], qx, qy, cur, right, j == 0 && nseg == 0};
            LitOut o;
            literal_until_push(P, in, o);
            if (P.counters) {
                atomicAdd(&P.counters[1], (unsigned long long)o.iters);
                atomicAdd(&P.counters[2], o.nq[0]);
                if (o.nq[1]) atomicAdd(&P.counters[3], o.nq[1]);
            }
            if (o.code == 0) {
                n_litpush++;
                push(o.e);
                cur = o.e;
                cur_kout = o.e_q;
                qx = o.qx;
                qy = o.qy;
                if (mode != MODE_DONE && !literal_only && o.e_q >= 0) {
                    arm(o.e, o.e_q);
                    if (clean) mode = MODE_FAST;
                }
            } else {
                endcode = o.code;
                status = o.status;
                mode = MODE_DONE;
            }
        }
    }

    if (t < P.n_tracks && j < P.ch.nch[t]) {
        P.ch.count[cidx] = active ? nseg : 0;
        P.ch.sum[cidx] = 0.0;
        P.ch.endcode[cidx] = active ? (endcode | (status << 8)) : (END_HANDOFF | (0 << 8));
    }
    if (P.counters) {
        unsigned long long v = active ? (unsigned long long)(nseg - n_litpush) : 0ull;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(FULL, v, o);
        if (lane == 0 && v) atomicAdd(&P.counters[0], v);
    }
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
