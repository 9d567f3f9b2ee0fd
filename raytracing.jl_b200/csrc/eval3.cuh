// eval3.cuh -- second half of the single-walk pipeline: ONE WARP PER CHUNK, ONE LANE PER SEGMENT.
//
// k_march (march.cuh) has walked every chunk once, counted its segments and left one 4-byte record per segment in the
// chunk's blocks of the record pool; k_fixup_tracks and the scan have fixed where the chunk's segments go.  This kernel turns
// the records into Segment(p, q, l, element) columns (src/segment.jl:23-33):
//
//   fast record    (h << 2) | (exit1 << 1)   h = entry half-edge 3*cell + k_in; the chord leaves through edge k_in+1 / k_in+2.
//                  q = intersection(track.ABC, general_form(exit edge))  (src/intersection.jl:127-138) with the edge's
//                  PRECOMPUTED general_form (EdgeRec, k_cell_records: src/intersection.jl:11-18 evaluated once per mesh, in the
//                  cell's stored orientation -- exactly the operands the reference recomputes for every track that crosses the
//                  cell); p = the previous segment's q (the shared edge gives the same line up to an exact sign flip, under
//                  which intersection() is invariant bit for bit), taken from the neighbouring lane by shuffle.
//   literal record (cell << 2) | 1           the reference's intersections() on that cell (src/intersection.jl:34-119), the
//                  same function the walk used when it accepted the cell (0.1 % of the segments); evaluated in a second loop
//                  so that its register appetite stays out of the main one.
//
// All lanes of a warp work on one track, so the track line is warp-uniform, the 32 records and the 32 x 6 output values of an
// iteration are contiguous (coalesced), and the per-track length sum needs one atomic per chunk.  Per segment the kernel
// gathers ONE 32-byte sector (the EdgeRec), executes ~45 FP64 instructions (one shared reciprocal, one square root) and
// writes 44 bytes: the HBM write stream of the Segment columns is its roofline.
#pragma once
#include "walk.cuh"

namespace rt {

// one warp per block: a block's slot is free again the moment its chunk is done (measured 1 % better than 4 warps per block,
// 3 % better than 8: profiles/r2_block_sizes.txt)
#ifndef RT_EVAL3_THREADS
#define RT_EVAL3_THREADS 32
#endif
constexpr int kEval3Threads = RT_EVAL3_THREADS;
#ifndef RT_EVAL3_MIN_BLOCKS
#define RT_EVAL3_MIN_BLOCKS 32
#endif
#ifndef RT_EVAL3_ALIGN
#define RT_EVAL3_ALIGN 8  // the first lane's output position is a multiple of this many segments (8 doubles = 64 bytes; see below)
#endif
#ifndef RT_EVAL3_PF_AHEAD
#define RT_EVAL3_PF_AHEAD 64  // L2 prefetch distance in units (= 32 warps each); 0: off
#endif

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// intersection(track, L) (src/intersection.jl:127-138) through the shared-reciprocal division; `redo` is set when a quotient did
// not pass ptxas' own acceptance test (zero or extreme numerators): the caller then repeats the formula with the plain operators
__device__ __forceinline__ bool eval3_cross(const Line &trk, const Line &L, P2 &out, bool &redo) {
    const double a = trk.b * L.a, b = L.b * trk.a;
    const double fa = fabs(a), fb = fabs(b);
    const bool par = fabs(a - b) <= kRtol * (fa > fb ? fa : fb);  // isapprox(a, b) for finite operands
    const Recip rd = recip_prepare(a - b);
    bool ok = rd.ok;
    out.x = div_try<false>(trk.c * L.b - L.c * trk.b, rd, ok);
    out.y = div_try<false>(trk.a * L.c - L.a * trk.c, rd, ok);
    redo = !ok;
    return par;
}

__global__ void __launch_bounds__(kEval3Threads, RT_EVAL3_MIN_BLOCKS) k_eval3(const __grid_constant__ WalkParams P) {
    const unsigned FULL = 0xffffffffu;
    const DevMesh &m = P.m;
    const int lane = threadIdx.x & 31;
    // warp -> chunk slot: 32 consecutive warps take the 32 chunks of one unit (the same chunk index of 32 adjacent tracks), units
    // in the spatial execution order of the walk
    const long long w = blockIdx.x * (long long)(kEval3Threads / 32) + (threadIdx.x >> 5);
    const long long slot = P.unit_begin + (w >> 5);
    if (slot >= P.unit_end) return;
    if (P.cancel && *P.cancel) return;  // (optimistic launch behind the walk: the batch turned out not to fit, scan.cuh ScanGuard)
    const int ls = (int)(w & 31);
    const long long unit = P.ch.order ? P.ch.order[slot] : slot;
    // Everything that only needs the chunk slot is requested at once, BEFORE the early exits (a warp lives for ~4 iterations,
    // so a chain of dependent header loads in front of them costs as much as the arithmetic): count, first records, prefix,
    // seed point next to the unit's block; then the track's data; then the per-angle data.
#if RT_EVAL3_PF_AHEAD > 0
    // The records and the slot data of the chunk that the warp RT_EVAL3_PF_AHEAD units behind this one will evaluate are pulled
    // into L2 now.  They are read exactly once, from DRAM, at the head of that warp's dependent load chain, and under the
    // evaluation's own 2.2 GB write stream a cold DRAM read costs several times its idle latency (the same kernel storing into an
    // L2-resident dummy region runs in 0.73 ms instead of 0.96).  Distances of 32 .. 128 units measure the same (-3.3 %), 512 and
    // more are evicted again before they are used (profiles/r2_eval_ablation.txt).
    {
        const long long slot_a = slot + RT_EVAL3_PF_AHEAD;
        if (slot_a < P.unit_end) {
            const long long unit_a = P.ch.order ? P.ch.order[slot_a] : slot_a;
            const long long cidx_a = unit_a * 32 + ls;
            const char *recs = (const char *)(P.pool + (cidx_a - P.pool_slot_base) * kRecBlock);
            if (lane < 4) prefetch_l2(recs + 128 * lane);
            else if (lane == 4) prefetch_l2(P.ch.count + cidx_a);
            else if (lane == 5) prefetch_l2(P.ch.prefix + cidx_a);
            else if (lane == 6) prefetch_l2(P.ch.seed_qx + cidx_a);
            else if (lane == 7) prefetch_l2(P.ch.seed_qy + cidx_a);
        }
    }
#endif
    const long long cidx = unit * 32 + ls;
    const int pb0 = (int)(cidx - P.pool_slot_base);
    int pb = pb0;
    const int cnt = P.ch.count[cidx];
    const int rec_first = P.pool[(long long)pb * kRecBlock + lane];
    const int prefix = P.ch.prefix[cidx];
    const double seedx = P.ch.seed_qx[cidx], seedy = P.ch.seed_qy[cidx];
    const int blk = P.ch.unit_block[unit];
    const long long t = 32LL * blk + ls;
    if (t >= P.n_tracks || t < P.trk_begin || t >= P.trk_end) return;
    const int nch = P.ch.nch[t];
    const long long ubase = P.ch.unit_base[blk];
    const int az = P.t.azim[t];
    const Line trk{P.t.a[t], P.t.b[t], P.t.c[t]};
    const long long off_t = P.offsets[t];
    const int j = (int)(unit - ubase);
    if (j >= nch) return;  // (count is only defined for the chunks the track has)
    if (cnt <= 0) return;
    int rec_cur = lane < cnt ? rec_first : 1;  // aligned record vector of this iteration (records 32 i .. 32 i + 31)
    int rec_prev = 1;                          // ... of the iteration before
    int rec;

    const unsigned long long pol_keep = l2_policy_keep();
    const bool right = P.ang.phi[az] < kPi / 2;  // isless(phi, pi/2), src/intersection.jl:153
    const double delta = P.vol ? P.ang.delta_eff[az] : 0.0;
    const long long base = off_t - P.offset_base + prefix;
    // entry point of the chunk's first segment when that is a fast record: the exit point of the seed cell (k_seed), which
    // the previous chunk's walker pushed last.  Afterwards: q of the previous iteration's lane 31 (kept in lane 0).
    double cqx = seedx, cqy = seedy;  // (only used when j > 0)
    int cfast = j > 0;
    double lsum = 0.0;
    bool bad = false, any_lit = false;
    const int rot = (lane + 31) & 31;

    // The lanes are shifted by sh = (first output position) mod RT_EVAL3_ALIGN so that every warp store starts on an aligned
    // boundary of its column: lane l of iteration i evaluates segment v = 32 i + l - sh.  An unaligned warp store of 32 x 8 bytes
    // touches 3 lines and 9 sectors; aligned to 16 segments (a 128-byte line) it touches 2 lines and 8 sectors, aligned to 8 or 4
    // segments 3 lines and 8 sectors -- and the SM -> L2 path, which the six column streams keep busy for 0.35 of the kernel's
    // duration, charges a request per line and a beat per sector (profiles/r2_eval_ablation.txt: -4.9 % for 16).  8 measures
    // another 1 % faster than 16 (profiles/r2_chunk_band.txt): half as many idle lanes in a chunk's first iteration buy more than
    // the third line costs.  The records stay loaded in aligned vectors (one 128-byte line each) and are rotated into place with
    // two shuffles.
    const int sh = (int)(base & (RT_EVAL3_ALIGN - 1));
    const int src_lane = (lane - sh) & 31;
    for (int i0 = 0; i0 < cnt + sh; i0 += 32) {
        const int v = i0 + lane - sh;
        int rec_next = 1;
        {
            const int i1 = i0 + 32;
            if (i1 < cnt && (i1 & (kRecBlock - 1)) == 0) pb = P.pool_next[pb];
            if (i1 + lane < cnt) rec_next = P.pool[(long long)pb * kRecBlock + ((i1 + lane) & (kRecBlock - 1))];
        }
        {
            const int a = __shfl_sync(FULL, rec_prev, src_lane), b = __shfl_sync(FULL, rec_cur, src_lane);
            rec = lane < sh ? a : b;
        }
        const bool fast = (rec & 1) == 0;  // (lanes outside the chunk carry rec = 1)
        const unsigned h = (unsigned)rec >> 2;
        const unsigned cell = fast ? h / 3u : h;
        const unsigned kin = h - 3u * cell;
        const bool exit1 = (rec & 2) != 0;
        P2 q{0.0, 0.0};
        bool par = false, redo = false;
        Line L{0.0, 0.0, 0.0};
        if (fast) {
            unsigned kout = kin + (exit1 ? 1u : 2u);
            kout = kout >= 3u ? kout - 3u : kout;
            double elen;
            ldg256_keep(m.edges + (3u * cell + kout), pol_keep, L.a, L.b, L.c, elen);
            par = eval3_cross(trk, L, q, redo);
        }
        if (redo) par = intersection(trk, L, q);  // plain IEEE operators (rare: a numerator is exactly zero)
        // hand-over of the exit points: lane i-1's q is my p; lane 0 takes the previous iteration's lane 31
        const double rx = __shfl_sync(FULL, q.x, rot), ry = __shfl_sync(FULL, q.y, rot);
        const int rfast = __shfl_sync(FULL, (int)fast, rot);
        const bool from_left = lane != 0 && v != 0;  // (the chunk's first segment takes the seed point, wherever its lane is)
        P2 p{from_left ? rx : cqx, from_left ? ry : cqy};
        const bool have = (from_left ? rfast : cfast) != 0;
        cqx = rx;
        cqy = ry;
        cfast = rfast;
        if (fast && !have) {  // the previous record is literal (or this is the first segment of the track): evaluate the entry edge
            double elen;
            ldg256_keep(m.edges + (3u * cell + kin), pol_keep, L.a, L.b, L.c, elen);
            intersection(trk, L, p);  // never parallel: the previous chord ended on this edge
        }
        if (fast) {
            const double dx = p.x - q.x, dy = p.y - q.y;
            const double l = sqrt(dx * dx + dy * dy);  // Segment(p, q): norm(p - q), src/segment.jl:32
            // (plain stores: an evict-first policy or st.cs on the output stream measures 1 % slower, write-through the same)
            const long long so = base + v;
            P.opx[so] = p.x;
            P.opy[so] = p.y;
            P.oqx[so] = q.x;
            P.oqy[so] = q.y;
            P.olen[so] = l;
            P.oelem[so] = (int)cell + 1;
            if (P.vol) atomicAdd(&P.vol[cell], delta * l);  // volumes[i] += delta_s[a]*l, src/trackgenerator.jl:382
            lsum += l;
            // the geometric conditions of the sequential fast path (walk.cuh); k_march's filters make them hold:
            // order_intersection_points (src/intersection.jl:151-159) must put the entry first (hits are stored in edge order)
            const bool kin_lt_kout = (kin == 0u) || (kin == 1u && exit1);
            const bool lt = right ? (p.x < q.x) : (p.x > q.x);
            const bool in_first = lt || (p.x == q.x && !kin_lt_kout);
            bad = bad || par || !in_first || !(l > P.lmin);
        } else if ((unsigned)v < (unsigned)cnt) {
            any_lit = true;
        }
        rec_prev = rec_cur;
        rec_cur = rec_next;
    }
    if (bad) atomicExch(P.verify_fail, 1);

    // ---- literal records (rare): the reference's intersections() on the cell
    if (__any_sync(FULL, any_lit)) {
        pb = pb0;
        for (int i0 = 0; i0 < cnt; i0 += 32) {
            if (i0 && (i0 & (kRecBlock - 1)) == 0) pb = P.pool_next[pb];
            const int v = i0 + lane;
            const int r = v < cnt ? P.pool[(long long)pb * kRecBlock + (v & (kRecBlock - 1))] : 0;
            if (r & 1) {
                const int cell = r >> 2;
                P2 p, q;
                int e_p, e_q;
                intersections(m, cell, trk, right, p, q, e_p, e_q);
                const double l = norm2(p.x - q.x, p.y - q.y);
                const long long so = base + v;
                P.opx[so] = p.x;
                P.opy[so] = p.y;
                P.oqx[so] = q.x;
                P.oqy[so] = q.y;
                P.olen[so] = l;
                P.oelem[so] = cell + 1;
                if (P.vol) atomicAdd(&P.vol[cell], delta * l);
                lsum += l;
            }
        }
    }
    if (P.tsum) {
        for (int o = 16; o > 0; o >>= 1) lsum += __shfl_down_sync(FULL, lsum, o);
        if (lane == 0) atomicAdd(&P.tsum[t], lsum);
    }
}

}  // namespace rt
