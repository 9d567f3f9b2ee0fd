// march.cuh -- k_march: the sign-test walk of the half-edge graph, with a REGISTER-RESIDENT hot loop.
//
// A Segment(p, q, l, element) depends only on (track, cell): intersections() uses the track's infinite line
// (src/intersection.jl:60).  So the serial part of _segmentize_track! (src/track.jl:106-178) is only the ORDER in which cells
// are accepted; the geometry of every accepted cell can be evaluated independently afterwards.  k_march walks each chunk
// deciding every transition from the SIGNS of the signed distances of the cell's vertices from the track line (two
// multiply-adds per step, no division, no square root), under the same clearance test as the sequential fast path (walk.cuh);
// everything that test does not cover runs the literal walk of the reference, exactly as in walk.cuh.  It counts the accepted
// cells of every chunk and, when it is given a record pool (single-walk pipeline), records each of them for k_eval3; without a
// pool (the count pass of the hybrid pipeline) it only counts.
//
// The code is laid out for the register allocator: with the literal path (point location, intersections(), 100+ live values)
// inlined next to the fast transition, ptxas runs out of the 64 registers that 8 resident blocks allow and keeps the walker's
// state in local memory -- 17 local loads/stores per fast transition (profiles/r1_q).  Here
//   * the hot loop touches only scalars that fit the register file: track line (a, b, c, g), signed distances of the entry
//     edge's end points (s1, s2), the encoded half-edge to enter next, clearances, counters;
//   * everything the slow path needs beyond that lives in a MarchState record whose address is passed to ONE out-of-line
//     function (march_slow); the hot scalars are stored to it before the call and reloaded after it, so nothing is live
//     across the call and the callee's register appetite cannot leak into the loop;
//   * the last accepted cell / exit edge are recovered from the last record instead of being carried.
#pragma once
#include "walk.cuh"

namespace rt {

// one warp per block, like k_eval3: a block's slot is free again the moment its unit is done (64 x 16, 64 x 18 at 56 registers,
// 128 x 9 measure the same within 0.5 %: profiles/r2_chunk_band.txt r4k; occupancy is not what limits the walk)
#ifndef RT_MARCH_THREADS
#define RT_MARCH_THREADS 32
#endif
constexpr int kMarchThreads = RT_MARCH_THREADS;
#ifndef RT_MARCH_WAIT
#define RT_MARCH_WAIT 6
#endif
constexpr int kMarchWait = RT_MARCH_WAIT;
#ifndef RT_MARCH_MIN_BLOCKS
#define RT_MARCH_MIN_BLOCKS 32
#endif

struct MarchState {
    // constants of the walker
    double ta, tb, tc, g, ang_thr;
    long long t, cidx;
    int j, az, limit, stop_cell;
    bool right, cheap_ok;
    // state of the fast path
    double s1, s2;
    int enc, last_rec;  // last_rec: record of the last accepted FAST cell, -1 when (cur, cur_kout, q) below are current
    float clearA;
    int f;
    int live;    // this lane owns a chunk slot of an existing track
    int active;  // ... whose seed is valid
    // state only the slow path uses
    double qx, qy;
    int cur, cur_kout;
    // bookkeeping
    int mode, nseg, pb, endcode, status, n_litpush;
    int recording;
    unsigned lit_iters, nn_q, knn_q;
    unsigned s_rec;  // shared-space address of this thread's column of the staging tile (stride kMarchThreads words)
};

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

// MODE_RETRY: the hot loop gave up on the transition through `enc`; march_slow re-examines it exactly before going literal
enum { MODE_RETRY = 3 };

__device__ __forceinline__ void sts32(unsigned addr, int v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ int lds32(unsigned addr) {
    int v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}

// one accepted segment: stage its record (8 records = one 32-byte sector per store), claim pool blocks, end conditions
__device__ __forceinline__ void march_push(const WalkParams &P, bool at_stop, int rec, int &nseg, int &pb, int &recording, int &mode,
                                           int &endcode, int limit, unsigned s_rec) {
    if (recording) {
        if (nseg > 0 && (nseg & (kRecBlock - 1)) == 0) {  // the current block is full: claim the next one
            const int nb = atomicAdd(P.pool_cursor, 1);
            if (nb >= P.pool_blocks) {
                recording = 0;  // pool exhausted (the host sees pool_cursor > pool_blocks and repeats the call)
            } else {
                P.pool_next[pb] = nb;
                pb = nb;
            }
        }
        if (recording) {
            const int k = nseg & 7;
            sts32(s_rec + 4u * kMarchThreads * k, rec);
            if (k == 7) {
                int v[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = lds32(s_rec + 4u * kMarchThreads * q);
                stg256_plain_i(P.pool + (long long)pb * kRecBlock + ((nseg & (kRecBlock - 1)) - 7), v);
            }
        }
    }
    nseg += 1;
    if (nseg >= limit) {  // while i < MAX_ITER (src/track.jl:119)
        endcode = END_CAP;
        mode = MODE_DONE;
    } else if (at_stop) {  // the cell the next valid chunk starts from: hand over
        endcode = END_HANDOFF;
        mode = MODE_DONE;
    }
}

__device__ __forceinline__ void march_arm(const DevMesh &m, MarchState &s, int e, int e_q, bool &clean) {
    const CellRec &r = m.cells[e];
    s.cur = e;
    s.cur_kout = e_q;
    s.last_rec = -1;
    s.clearA = fabsf(r.clear);
    const double v0 = s.ta * r.vx[0] + s.tb * r.vy[0] + s.tc, v1 = s.ta * r.vx[1] + s.tb * r.vy[1] + s.tc,
                 v2 = s.ta * r.vx[2] + s.tb * r.vy[2] + s.tc;
    const double thr = s.g * (double)s.clearA;
    s.s1 = e_q == 0 ? v0 : (e_q == 1 ? v1 : v2);
    s.s2 = e_q == 0 ? v1 : (e_q == 1 ? v2 : v0);
    clean = (fabs(v0) >= thr) && (fabs(v1) >= thr) && (fabs(v2) >= thr) && ((s.s1 > 0) != (s.s2 > 0));
    s.enc = m.twin[3 * e + e_q];
    s.f = s.enc & 1;
}

// exact form of the three geometric fast-path conditions (exit edge not parallel, entry ordered first, chord > l_min; band cells:
// re-location points not `inboundary`) for the transition into the cell of half-edge h -- the transitions the cheap filter of the
// hot loop cannot decide (0.6 % of them)
__device__ __forceinline__ bool march_exact(const WalkParams &P, double ta, double tb, double tc, int h, bool exit1, bool right, float clearf) {
    const DevMesh &m = P.m;
    const int cellB = h / 3;
    const int kin = h - 3 * cellB;
    int kout = kin + (exit1 ? 1 : 2);
    kout = kout >= 3 ? kout - 3 : kout;
    const Line trk{ta, tb, tc};
    const EdgeRec ei = m.edges[3 * cellB + kin], eo = m.edges[3 * cellB + kout];
    P2 pi, X;
    const bool par_i = intersection(trk, Line{ei.a, ei.b, ei.c}, pi);
    const bool par_o = intersection(trk, Line{eo.a, eo.b, eo.c}, X);
    const bool kin_lt_kout = (kin == 0) || (kin == 1 && exit1);
    const bool in_first = right ? (kin_lt_kout ? (pi.x < X.x) : !(X.x < pi.x)) : (kin_lt_kout ? (pi.x > X.x) : !(X.x > pi.x));
    const double l = norm2(pi.x - X.x, pi.y - X.y);
    bool accept = !par_i && !par_o && in_first && l > P.lmin;
    if (accept && clearf < 0.0f) accept = bbox_dist(m, pi.x, pi.y) > 0.25 * l + 8.0 * P.tiny;
    return accept;
}

// The slow side of the walk, out of line: (1) the transition the hot loop could not decide with the cheap filter is re-examined
// with the exact chord (march_exact); (2) if it is not a fast transition, the literal walk of the reference runs until
// it pushes one segment, and the fast path is re-armed from there.
__device__ __noinline__ void march_slow(const WalkParams &P, MarchState &s) {
    const DevMesh &m = P.m;
    const unsigned long long pol_keep = l2_policy_keep();
    const bool literal_only = (P.flags & 1u) != 0;
    if (s.mode == MODE_RETRY && s.enc >= 0) {
        double ax, ay, w0, w1;
        ldg256_keep(m.he + (s.enc >> 3), pol_keep, ax, ay, w0, w1);
        const float clearf = __int_as_float(__double2loint(w1));
        const float clearB = fabsf(clearf);
        const double sa = s.ta * ax + s.tb * ay + s.tc;
        const double thr = s.g * (double)fmaxf(s.clearA, clearB);
        if ((fabs(sa) >= thr) && (fabs(s.s1) >= thr) && (fabs(s.s2) >= thr)) {
            const bool opp1 = (sa > 0) != (s.s1 > 0);
            const double ks = opp1 ? s.s1 : s.s2;
            const bool exit1 = (opp1 == (s.f != 0));
            const int nenc = exit1 ? __double2loint(w0) : __double2hiint(w0);
            const int h = s.enc >> 3;
            const int cellB = h / 3;
            const bool accept = march_exact(P, s.ta, s.tb, s.tc, h, exit1, s.right, clearf);
            if (accept) {
                s.s1 = ks;
                s.s2 = sa;
                s.f = (exit1 == ((nenc & 1) != 0)) ? 1 : 0;
                s.enc = nenc;
                s.clearA = clearB;
                s.last_rec = (h << 2) | (exit1 ? 2 : 0);
                s.mode = MODE_FAST;
                march_push(P, cellB == s.stop_cell, s.last_rec, s.nseg, s.pb, s.recording, s.mode, s.endcode, s.limit, s.s_rec);
                return;
            }
        }
    }
    s.mode = MODE_SLOW;
    // ---- literal walk until one push: needs the exit point of the last accepted cell
    if (s.last_rec >= 0) {  // the last cell was accepted by the fast path: recover (cell, exit edge) from its record
        const int r = s.last_rec;
        const int h = r >> 2;
        const int cell = h / 3;
        const int kin = h - 3 * cell;
        int kout = kin + ((r & 2) ? 1 : 2);
        kout = kout >= 3 ? kout - 3 : kout;
        const P2 X = exit_point(m, Line{s.ta, s.tb, s.tc}, cell, kout);  // advance_step(q, tiny, phi) starts here, src/track.jl:165
        s.cur = cell;
        s.cur_kout = kout;
        s.qx = X.x;
        s.qy = X.y;
        s.last_rec = -1;
    }
    LitIn in{s.ta, s.tb, s.tc, P.tiny * P.ang.cosp[s.az], P.tiny * P.ang.sinp[s.az], s.qx, s.qy, s.cur, s.right, s.j == 0 && s.nseg == 0};
    LitOut o;
    literal_until_push(P, in, o);
    s.lit_iters += o.iters;
    s.nn_q += (unsigned)o.nq[0];
    s.knn_q += (unsigned)o.nq[1];
    if (o.code == 0) {
        s.n_litpush++;
        march_push(P, o.e == s.stop_cell, (o.e << 2) | 1, s.nseg, s.pb, s.recording, s.mode, s.endcode, s.limit, s.s_rec);
        s.cur = o.e;
        s.cur_kout = o.e_q;
        s.qx = o.qx;
        s.qy = o.qy;
        s.last_rec = -1;
        if (s.mode != MODE_DONE && !literal_only && o.e_q >= 0) {
            bool clean;
            march_arm(m, s, o.e, o.e_q, clean);
            if (clean) s.mode = MODE_FAST;
        }
    } else {
        s.endcode = o.code;
        s.status = o.status;
        s.mode = MODE_DONE;
    }
}

// prologue, out of line as well (it runs once per walker and shares nothing with the loop)
__device__ __noinline__ void march_init(const WalkParams &P, MarchState &s, int lane, long long unit) {
    const DevMesh &m = P.m;
    const int blk = P.ch.unit_block[unit];
    s.j = (int)(unit - P.ch.unit_base[blk]);
    s.t = 32LL * blk + lane;
    s.cidx = unit * 32 + lane;
    s.mode = MODE_DONE;
    s.nseg = 0;
    s.status = 0;
    s.endcode = END_TRACK;
    s.n_litpush = 0;
    s.lit_iters = s.nn_q = s.knn_q = 0;
    s.enc = -1;
    s.last_rec = -1;
    s.cur = -1;
    s.cur_kout = -1;
    s.stop_cell = -1;
    s.limit = P.max_iter;
    s.pb = (int)(s.cidx - P.pool_slot_base);
    s.recording = P.pool != nullptr;  // (the count pass of the hybrid pipeline records nothing)
    s.ta = s.tb = s.tc = s.g = s.ang_thr = s.s1 = s.s2 = s.qx = s.qy = 0.0;
    s.clearA = INFINITY;
    s.f = 0;
    s.right = true;
    s.cheap_ok = false;
    s.az = 0;
    s.live = s.active = 0;
    const long long t = s.t;
    if (t >= P.n_tracks) return;
    const int n = P.ch.nch[t];
    if (s.j >= n) return;
    s.live = 1;
    if (t < P.trk_begin || t >= P.trk_end) return;
    const int seed = s.j == 0 ? -2 : P.ch.seed_cell[s.cidx];
    if (seed == -1) return;  // void seed: the previous walker continues through this chunk (count 0, END_HANDOFF)
    s.active = 1;
    constexpr double kKappa = 1.0 / RT_KAPPA_INV;
    s.az = P.t.azim[t];
    s.ta = P.t.a[t];
    s.tb = P.t.b[t];
    s.tc = P.t.c[t];
    s.right = P.ang.phi[s.az] < kPi / 2;  // isless(phi, pi/2), src/intersection.jl:153
    s.g = sqrt(s.ta * s.ta + s.tb * s.tb);
    s.ang_thr = kKappa * s.g * P.lmax;
    s.cheap_ok = P.lmin * (fabs(s.tb) / s.g) > 32.0 * 2.220446049250313e-16 * P.smax / kKappa;
    const bool literal_only = (P.flags & 1u) != 0;
    if (s.j == 0) {
        s.qx = P.t.px[t];  // the literal walk starts from advance_step(track.p), src/track.jl:114
        s.qy = P.t.py[t];
        s.mode = MODE_SLOW;
    } else {
        bool clean;
        march_arm(m, s, seed, P.ch.seed_kexit[s.cidx], clean);  // k_seed verified `clean`
        s.qx = P.ch.seed_qx[s.cidx];
        s.qy = P.ch.seed_qy[s.cidx];
        s.mode = (literal_only || !clean) ? MODE_SLOW : MODE_FAST;
    }
    for (int jj = s.j + 1; jj < n; ++jj) {
        const int sc = P.ch.seed_cell[s.cidx + 32LL * (jj - s.j)];
        if (sc >= 0) {
            s.stop_cell = sc;
            break;
        }
    }
    if (s.j > 0 && s.stop_cell == s.cur) {  // next seed sits in the same cell: this chunk is empty
        s.endcode = END_HANDOFF;
        s.mode = MODE_DONE;
    }
    if (s.limit <= 0) {  // while i < MAX_ITER never runs
        s.endcode = END_CAP;
        s.mode = MODE_DONE;
    }
}

__global__ void __launch_bounds__(kMarchThreads, RT_MARCH_MIN_BLOCKS) k_march(const __grid_constant__ WalkParams P) {
    const unsigned FULL = 0xffffffffu;
    const DevMesh &m = P.m;
    __shared__ int s_rec[8 * kMarchThreads];  // 8 records per thread = one 32-byte sector
    const int lane = threadIdx.x & 31;
    const long long gw = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long slot = P.unit_begin + gw;
    if (slot >= P.unit_end) return;  // whole warp
    const long long unit = P.ch.order ? P.ch.order[slot] : slot;

    MarchState S;
    S.s_rec = (unsigned)__cvta_generic_to_shared(s_rec + threadIdx.x);
    march_init(P, S, lane, unit);
    const bool live = S.live != 0, active = S.active != 0;

    // ---- hot scalars
    // (also the loop invariants are re-read from S after every call of march_slow: a value that stays live across the call
    // would be kept in local memory by ptxas and re-loaded in every iteration of the loop)
    double ta = S.ta, tb = S.tb, tc = S.tc, g = S.g, ang_thr = S.ang_thr;
    bool cheap_ok = S.cheap_ok;
    int limit = S.limit, stop_cell = S.stop_cell;
    unsigned my_rec = S.s_rec;
    double s1 = S.s1, s2 = S.s2;
    int enc = S.enc, last_rec = S.last_rec, mode = S.mode, nseg = S.nseg, pb = S.pb, endcode = S.endcode;
    float clearA = S.clearA;
    int f = S.f, recording = S.recording;
    const unsigned long long pol_keep = l2_policy_keep();
#ifdef RT_MARCH_DIAG
    unsigned diag_tot = 0, diag_done = 0, diag_wait = 0;  // lane-slots of the fast loop: all / finished lanes / lanes waiting for the slow side
#endif

    // The record of the half-edge to enter next (apex, twins of the two possible exit edges, clearances) is REQUESTED AS SOON AS
    // THE EXIT EDGE IS KNOWN -- two multiply-adds and a sign test after the previous record arrived -- and lands while the rest of
    // the transition (clearance and cheap-filter tests, record staging, end conditions) executes: the walk is one dependent gather
    // per step, so every instruction between "record arrived" and "next record requested" is latency the next step pays for
    // (profiles/r1_w: 32 % of the walk's stall samples sat on this load, behind ~80 instructions of bookkeeping).
    double rax = 0.0, ray = 0.0, rw0 = 0.0, rw1 = 0.0;
    if (mode == MODE_FAST && enc >= 0) ldg256_keep(m.he + (enc >> 3), pol_keep, rax, ray, rw0, rw1);

    while (__any_sync(FULL, mode != MODE_DONE)) {
        // ------------------------------------------------------------------ FAST phase: sign tests only
#pragma unroll 1
        for (int it = 0; it < 4 * kFastBatch; ++it) {
            if (!__any_sync(FULL, mode == MODE_FAST)) break;
            // lanes that need the slow side wait for it; leave the fast phase once kMarchWait of them do (the slow phase
            // costs a few hundred instructions per entry, an idle lane costs a lane of every fast iteration)
            if ((it & 1) && __popc(__ballot_sync(FULL, mode == MODE_SLOW || mode == MODE_RETRY)) >= kMarchWait) break;
#ifdef RT_MARCH_DIAG
            diag_tot++;
            if (mode == MODE_DONE) diag_done++;
            else if (mode != MODE_FAST) diag_wait++;
#endif
            if (mode != MODE_FAST) continue;
            if (enc < 0) {  // the exit edge lies on the boundary: the literal walk ends the track
                mode = MODE_RETRY;
                continue;
            }
            const double sa = ta * rax + tb * ray + tc;
            const bool opp1 = (sa > 0) != (s1 > 0);  // the exit edge joins the apex with the end point across the line
            const bool exit1 = (opp1 == (f != 0));
            const int nenc = exit1 ? __double2loint(rw0) : __double2hiint(rw0);
            const float clearf = __int_as_float(__double2loint(rw1));
            const float clear2 = __int_as_float(__double2hiint(rw1));
            if (nenc >= 0) ldg256_keep(m.he + (nenc >> 3), pol_keep, rax, ray, rw0, rw1);  // (speculative: the tests below may still say no)
            const float clearB = fabsf(clearf);
            const double thr = g * (double)fmaxf(clearA, clearB);
            const double ks = opp1 ? s1 : s2;  // ... which is the only vertex on its side of the track line
            // clearance test + cheap filter (DESIGN.md): the geometric fast-path conditions hold without evaluating the chord;
            // transitions it cannot decide (and every cell of the bounding-box band) are re-examined exactly by march_slow -- not
            // here: any call or any larger body inside this loop makes ptxas keep the walker's state in local memory
            const bool accept = (fabs(sa) >= thr) & (fabs(s1) >= thr) & (fabs(s2) >= thr) & cheap_ok & (clearf >= 0.0f) &
                                (fabs(ks) >= g * (double)clear2) & (fabs(ks) + fabs(sa) >= ang_thr) & (fabs(s1) + fabs(s2) >= ang_thr);
            if (!accept) {
                mode = MODE_RETRY;  // (the record in flight belongs to a half-edge that is not entered: march_slow re-arms)
                continue;
            }
            const int h = enc >> 3;
            last_rec = (h << 2) | (exit1 ? 2 : 0);
            s1 = ks;
            s2 = sa;
            f = (exit1 == ((nenc & 1) != 0)) ? 1 : 0;
            enc = nenc;
            clearA = clearB;
            // (cell of h == stop_cell) without dividing: h in [3*stop_cell, 3*stop_cell + 2]; stop_cell = -1: never
            const bool at_stop = (unsigned)(h - 3 * stop_cell) < 3u;
            march_push(P, at_stop, last_rec, nseg, pb, recording, mode, endcode, limit, my_rec);
        }
        // ------------------------------------------------------------------ SLOW phase (out of line)
        if (mode == MODE_SLOW || mode == MODE_RETRY) {
            S.s1 = s1;
            S.s2 = s2;
            S.enc = enc;
            S.last_rec = last_rec;
            S.clearA = clearA;
            S.f = f;
            S.mode = mode;
            S.nseg = nseg;
            S.pb = pb;
            S.recording = recording;
            S.endcode = endcode;
            march_slow(P, S);
            ta = S.ta;
            tb = S.tb;
            tc = S.tc;
            g = S.g;
            ang_thr = S.ang_thr;
            cheap_ok = S.cheap_ok;
            limit = S.limit;
            stop_cell = S.stop_cell;
            my_rec = S.s_rec;
            s1 = S.s1;
            s2 = S.s2;
            enc = S.enc;
            last_rec = S.last_rec;
            clearA = S.clearA;
            f = S.f;
            mode = S.mode;
            nseg = S.nseg;
            pb = S.pb;
            recording = S.recording;
            endcode = S.endcode;
            // (assigned on every path: a value that stays live across the call above would be kept in local memory for the whole loop)
            rax = ray = rw0 = rw1 = 0.0;
            if (mode == MODE_FAST && enc >= 0) ldg256_keep(m.he + (enc >> 3), pol_keep, rax, ray, rw0, rw1);
        }
    }

    if (recording && (nseg & 7)) {  // the incomplete last sector of this chunk's records
        const int rem = nseg & 7;
        int *dst = P.pool + (long long)pb * kRecBlock + (((nseg - 1) & (kRecBlock - 1)) - (rem - 1));
        for (int kk = 0; kk < rem; ++kk) dst[kk] = lds32(my_rec + 4u * kMarchThreads * kk);
    }
    if (live) {
        P.ch.count[S.cidx] = active ? nseg : 0;
        P.ch.sum[S.cidx] = 0.0;
        P.ch.endcode[S.cidx] = active ? (endcode | (S.status << 8)) : (END_HANDOFF | (0 << 8));
    } else {
        P.ch.count[S.cidx] = 0;  // (a slot no track owns: the evaluation requests its count before it knows that)
    }
    if (P.counters) {
        unsigned long long v = active ? (unsigned long long)(nseg - S.n_litpush) : 0ull;
        unsigned long long li = S.lit_iters, q0 = S.nn_q, q1 = S.knn_q;
#ifdef RT_MARCH_DIAG
        li = diag_done;
        q0 = diag_wait;
        q1 = diag_tot;
#endif
        for (int o = 16; o > 0; o >>= 1) {
            v += __shfl_down_sync(FULL, v, o);
            li += __shfl_down_sync(FULL, li, o);
            q0 += __shfl_down_sync(FULL, q0, o);
            q1 += __shfl_down_sync(FULL, q1, o);
        }
        if (lane == 0) {
            if (v) atomicAdd(&P.counters[0], v);
            if (li) atomicAdd(&P.counters[1], li);
            if (q0) atomicAdd(&P.counters[2], q0);
            if (q1) atomicAdd(&P.counters[3], q1);
        }
    }
}

}  // namespace rt
