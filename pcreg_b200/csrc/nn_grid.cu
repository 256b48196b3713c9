// nn_grid.cu -- exact nearest neighbour on the uniform grid + occupancy pyramid (large models).
//
// Semantics identical to nn_brute.cu (knnsearch K=1, FP64, ties -> smallest original index); the
// reference's nearest analogue of a spatially pruned search is speedyDescriptors.m:44-60 (boxes with a
// halo) and getLocalPoints.m:8-15 (cube pre-filter).
//
// Up to three kernels per NN pass (one thread per query unless noted):
//   k_nn_list         (ICP passes >= 2) queries that own a CANDIDATE LIST -- every model point within
//                     R_list = r0 + skin of the position q0 the query had when the list was built -- scan it
//                     exactly.  A point outside the list is farther than R_list - |q - q0| from the moved
//                     query, so when the best list distance is below that the list answer is the exact
//                     nearest neighbour (ties included).  Everything else goes to the next kernel.
//                     Entries carry the level of their build-time distance, so candidates that cannot have
//                     become the nearest one are skipped without a gather; queries that are provably outside
//                     the trim / beyond the rejection threshold of this pass are not searched at all (lazy
//                     trimming, see the kernel).
//   k_nn_grid_direct  warm-started queries whose ball (radius = distance to the previous iteration's
//                     correspondence) spans at most GRID_ROW_SPAN level-0 cells in y and z: every (y,z) cell
//                     row the ball reaches is one contiguous run of points.  Persistent warps, one small state
//                     machine per lane, work drawn in 32-query chunks from a global cursor.  Everything else
//                     is appended to a work list (warp-aggregated atomics).
//                     BUILD variant: the scan is exhaustive within (best distance + gap) and the points within
//                     (best distance + skin) become the query's new candidate list.
//   k_nn_grid_rows    the same row scan for DENSE models (>= 6 points per occupied cell): one warp per query, the
//                     lanes take consecutive points of the ball's rows (coalesced runs), see the kernel.
//   k_nn_grid_walk_warp  the walk of DENSE models from the third pass on: one warp per query, breadth-first frontier in shared
//                     memory, leaves scanned like the rows of k_nn_grid_rows; hands overflowing queries to k_nn_grid_walk.
//   k_nn_grid_walk    branch-and-bound walk of the occupancy pyramid with a small explicit stack for the
//                     work list (far queries, and every query of the first iteration).  Keeping the two
//                     populations in separate launches keeps the lanes of a warp on similar work.
// Pruning tests run in FP32 in CELL UNITS with a conservative slop (a cell is skipped only when a
// guaranteed LOWER bound of its distance exceeds a guaranteed UPPER bound of the best distance); every
// visited point is evaluated in FP64 with the oracle's formula and operation order and competes on
// (d2, original index) -- the answer equals the FP64 brute-force answer bit for bit.
#include <math.h>
#include <float.h>
#include <stdlib.h>
#include <algorithm>

#include "pcreg_internal.h"
#include "pcreg_dev.cuh"
#include "pcreg_grid.cuh"

namespace pcreg {

// ---- kernel 1: row scan ----------------------------------------------------------------------------------
// Cells of one x-row are contiguous in memory, so for a fixed (y,z) the cells the ball can touch are ONE
// run of points [cell_start[row + xa], cell_start[row + xb + 1]).  A query whose bounding cube spans at
// most GRID_ROW_SPAN cells in y and z walks its rows.
//
// The cost per query varies by more than 10x (ball radius), so a fixed thread <-> query mapping leaves most
// lanes of a warp idle behind its slowest query.  Instead each WARP owns a contiguous range of queries and
// every lane runs a small state machine: one trip of the loop is either "process one point" or "advance one
// row"; a lane that finishes its query takes the next one of the warp's range.  Fetching (pose transform,
// warm-start bound) is batched: it runs only when >= GRID_FETCH_BATCH lanes are idle, so it executes with
// many active lanes too.
constexpr int GRID_ROW_SPAN = 12;
constexpr int GRID_FETCH_BATCH = 8;
constexpr int GRID_CHUNK = 32;
constexpr double GRID_WARP_ROWS_DENSITY = 6.0;      // model points per occupied cell from which the warp-per-query row scan is used

template <bool BUILD>
__global__ void __launch_bounds__(128, 8) k_nn_grid_direct(const __grid_constant__ GridArgs a) {
    const GridView& G = a.g;
    const int lane = threadIdx.x & 31;
    const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t total = a.in_list ? (int64_t)*a.in_count : a.nq;
    if (a.counters && blockIdx.x == 0 && threadIdx.x == 0) {
        atomicAdd(&a.counters[5], (unsigned long long)total);
        if (a.in_list) atomicAdd(&a.counters[3], (unsigned long long)(a.nq - total));      // the list scan answered the rest
    }
    // work is handed out in chunks of consecutive queries from a global cursor (the per-query cost varies by more
    // than 10x, fixed ranges per warp leave a long tail); `next`..`end` is the warp's current chunk
    int64_t next = 0, end = 0;
    bool more = true;
    (void)warp_id; (void)nwarps;
    const double inv_cell2 = G.inv_cell * G.inv_cell;
    const int dx0 = G.dims[0][0], dy0 = G.dims[0][1], dz0 = G.dims[0][2];
    unsigned long long n_pts = 0, n_cells = 0;

    Query Q;
    int64_t gq = -1;
    bool have = false;
    int x0 = 0, x1 = 0, y0 = 0, y1 = 0, z1 = 0, y = 0, z = 0;
    int32_t p = 0, e = 0;
    float dz2 = 0.f;
    // candidate-list construction (BUILD)
    bool bld = false;
    int lc = 0, ext_slot = -1;
    double thr2 = 0.0;
    float lo = 0.f;

    while (true) {
        // ---- batched fetch ----
        const unsigned idle = __ballot_sync(0xffffffffu, !have);
        const int nidle = __popc(idle);
        if (next >= end && more && nidle >= a.fetch_batch) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(a.cursor, (unsigned long long)a.chunk);
            base = __shfl_sync(0xffffffffu, base, 0);
            if ((int64_t)base >= total) more = false;
            else { next = (int64_t)base; end = min(total, next + a.chunk); }
        }
        if (next < end && (nidle >= a.fetch_batch || nidle == 32)) {
            bool defer = false;
            if (!have) {
                const int64_t cand = next + __popc(idle & ((1u << lane) - 1u));
                if (cand < end) {
                    gq = a.in_list ? (int64_t)a.in_list[cand] : cand;
                    float gap = 0.f;
                    if (BUILD) {
                        // a list pays only if the pose has (nearly) stopped moving
                        bld = !a.cl.delta || a.cl.delta[(unsigned)gq / (unsigned)a.ns] <= a.cl.build_max_delta;
                        gap = bld ? a.cl.gap_cells : 0.f;
                    }
                    setup_query(a, gq, Q, gap, a.prev[gq]);
                    if (Q.has_span && Q.ihy - Q.ily < a.row_span && Q.ihz - Q.ilz < a.row_span && Q.ihx - Q.ilx < 4 * a.row_span) {
                        x0 = max(Q.ilx, 0); x1 = min(Q.ihx, dx0 - 1);
                        y0 = max(Q.ily, 0); y1 = min(Q.ihy, dy0 - 1);
                        z = max(Q.ilz, 0); z1 = min(Q.ihz, dz0 - 1);
                        y = y0;
                        p = 0; e = 0;
                        if (x0 > x1 || y0 > y1 || z > z1) z = z1 + 1;       // nothing to scan: the warm start stands
                        const float t = axis_lb(Q.fz, (float)z, 1.f);
                        dz2 = t * t;
                        have = true;
                        if (BUILD) {
                            lc = 0; ext_slot = bld ? a.cl.ext[gq] : -1; thr2 = bld ? list_thr2(Q.best, a.cl.skin) : 0.0;
                            lo = __fsqrt_rd(__double2float_rd(Q.best)) - (float)a.cl.skin;      // every listed point is within [.., lo + 2 skin]
                        }
                    } else {
                        defer = true;
                    }
                }
            }
            next += nidle;
            worklist_append(a, defer, gq, lane);             // deferred queries go to the walk kernel
            continue;
        }
        if (nidle == 32 && !more) break;                     // nothing in flight and nothing left to fetch
        if (nidle == 32) continue;
        // ---- one trip: lanes out of points advance one row, then every lane with points processes one ----
        if (have && p >= e) {
            if (z > z1) {                                    // rows exhausted: done with this query
                a.idx[gq] = Q.bidx;
                if (a.d2) a.d2[gq] = Q.best;
                if (BUILD) list_commit(a.cl, G, gq, Q, bld, lc, ext_slot, lo);
                have = false;
            } else {                                         // ROW step
                float dy2 = axis_lb(Q.fy, (float)y, 1.f);
                dy2 *= dy2;
                const float lb = (dy2 + dz2) * (1.f - 6e-7f);
                if (lb <= Q.bestc) {
                    // cells of this row the ball can reach: |x - fx| <= sqrt(bestc - lb) (+ slop)
                    const float rx = __fsqrt_ru(Q.bestc - lb) * (1.f + 1e-6f) + 2.f * GRID_SLOP_ABS + GRID_SLOP_REL * fabsf(Q.fx);
                    const int xa = max(x0, (int)floorf(Q.fx - rx)), xb = min(x1, (int)floorf(Q.fx + rx));
                    if (xa <= xb) {
                        const int64_t c0 = ((int64_t)z * dy0 + y) * dx0;
                        p = G.cell_start[c0 + xa];
                        e = G.cell_start[c0 + xb + 1];
                        if (e > p) { ++n_cells; n_pts += (unsigned long long)(e - p); }
                    }
                }
                if (++y > y1) {
                    y = y0; ++z;
                    const float t = axis_lb(Q.fz, (float)z, 1.f);
                    dz2 = t * t;
                }
            }
        }
        if (have && p < e) {                                 // POINT step
            const GridPoint gp = G.pts[p];
            const double d = dist2_exact(gp.x, gp.y, gp.z, Q.qx, Q.qy, Q.qz);
            if (d < Q.best || (d == Q.best && gp.orig < Q.bidx)) {
                Q.best = d; Q.bidx = gp.orig;
                if (BUILD && bld) {
                    Q.bestc = best_ub_cells_gap(Q.best, G.inv_cell, a.cl.gap_cells);
                    thr2 = list_thr2(Q.best, a.cl.skin);
                } else {
                    Q.bestc = best_ub_cells(Q.best, inv_cell2);
                }
            }
            if (BUILD && bld && d <= thr2) list_append(a.cl, gq, lc, ext_slot, p, d, lo);
            ++p;
        }
    }
    flush_counters(a.counters, n_pts, n_cells, 0);
}

// ---- kernel 1b: row scan, one WARP per query (dense models) ------------------------------------------------
// Same rows, same points, same exact answer as the per-lane state machine above, but the 32 lanes of a warp work on
// ONE query at a time: the lanes take the (y,z) rows of the ball (bounds + cell_start pair per lane), a warp scan of
// the run lengths turns them into one flat range of points, and consecutive lanes take consecutive points of that
// range (the run of a point is found by a 5-step shuffle search in the scanned lengths), so the gathers of a trip
// are coalesced runs instead of 32 separate sectors.  Pays when a query visits hundreds of points (many points per
// occupied cell: C5); on sparse models (C3: ~20 points per query) the single dependent load chain per warp loses
// against the 32 independent chains of the state machine (measured, DESIGN.md 3.2) -- the launcher picks by density.
// Setup (pose transform, warm-start bound, cell span) stays lane-parallel: a warp draws 32 consecutive queries, every
// lane prepares one, then they are processed one after the other with their parameters broadcast by shuffles.  The
// pruning bound is the warm-start distance, re-tightened between rounds of 32 rows.
// BUILD: a point enters the list when d2 <= (sqrt(warp's best so far) + skin)^2 -- a superset of the final list,
// exactly like the sequential rule; entries are appended by ballot compaction.
#ifndef ROWS_U
#define ROWS_U 2        // rounds of 32 points whose gathers are in flight together
#endif
#ifndef ROWS_BPS
#define ROWS_BPS 8      // blocks per SM: the kernel is latency bound, occupancy beats the few spilled registers (measured on C5:
#endif                  // row-scan ms of a 21-pass run  U=1/5 blocks 102, 2/5 89, 4/5 83, 2/6 80, 2/7 86, 1/8 80, 2/8 68; per-lane kernel 125)
template <bool BUILD>
__global__ void __launch_bounds__(128, ROWS_BPS) k_nn_grid_rows(const __grid_constant__ GridArgs a) {
    const GridView& G = a.g;
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int64_t total = a.in_list ? (int64_t)*a.in_count : a.nq;
    if (a.counters && blockIdx.x == 0 && threadIdx.x == 0) {
        atomicAdd(&a.counters[5], (unsigned long long)total);
        if (a.in_list) atomicAdd(&a.counters[3], (unsigned long long)(a.nq - total));      // the list scan answered the rest
    }
    const double inv_cell2 = G.inv_cell * G.inv_cell;
    const int dx0 = G.dims[0][0], dy0 = G.dims[0][1], dz0 = G.dims[0][2];
    unsigned long long n_pts = 0, n_cells = 0;

    while (true) {
        unsigned long long cbase = 0;
        if (lane == 0) cbase = atomicAdd(a.cursor, 32ull);
        cbase = __shfl_sync(FULL, cbase, 0);
        if ((int64_t)cbase >= total) break;
        // ---- lane-parallel setup of 32 consecutive queries ----
        const int64_t cand = (int64_t)cbase + lane;
        Query Q;
        int64_t gq = -1;
        bool ready = false, defer = false, bld = false;
        int x0 = 0, x1 = -1, y0 = 0, y1 = -1, z0 = 0, z1 = -1, ext_slot = -1;
        float lo = 0.f;
        Q.qx = Q.qy = Q.qz = 0.0; Q.fx = Q.fy = Q.fz = 0.f; Q.best = INFINITY; Q.bidx = -1; Q.bestc = 0.f;
        if (cand < total) {
            gq = a.in_list ? (int64_t)a.in_list[cand] : cand;
            float gap = 0.f;
            if (BUILD) {
                bld = !a.cl.delta || a.cl.delta[(unsigned)gq / (unsigned)a.ns] <= a.cl.build_max_delta;   // a list pays only once the pose has nearly stopped
                gap = bld ? a.cl.gap_cells : 0.f;
            }
            setup_query(a, gq, Q, gap, a.prev[gq]);
            if (Q.has_span && Q.ihy - Q.ily < a.row_span && Q.ihz - Q.ilz < a.row_span && Q.ihx - Q.ilx < 4 * a.row_span) {
                x0 = max(Q.ilx, 0); x1 = min(Q.ihx, dx0 - 1);
                y0 = max(Q.ily, 0); y1 = min(Q.ihy, dy0 - 1);
                z0 = max(Q.ilz, 0); z1 = min(Q.ihz, dz0 - 1);
                ready = true;
                if (BUILD && bld) {
                    ext_slot = a.cl.ext[gq];
                    lo = __fsqrt_rd(__double2float_rd(Q.best)) - (float)a.cl.skin;          // every listed point is within [.., lo + 2 skin]
                }
            } else {
                defer = true;
            }
        }
        worklist_append(a, defer, gq, lane);                 // wide balls go to the walk kernel
        unsigned todo = __ballot_sync(FULL, ready);
        while (todo) {
            const int j = __ffs(todo) - 1;
            todo &= todo - 1;
            // ---- broadcast query j ----
            const double qx = __shfl_sync(FULL, Q.qx, j), qy = __shfl_sync(FULL, Q.qy, j), qz = __shfl_sync(FULL, Q.qz, j);
            const float fx = __shfl_sync(FULL, Q.fx, j), fy = __shfl_sync(FULL, Q.fy, j), fz = __shfl_sync(FULL, Q.fz, j);
            double best = __shfl_sync(FULL, Q.best, j);
            int32_t bidx = __shfl_sync(FULL, Q.bidx, j);
            float bestc = __shfl_sync(FULL, Q.bestc, j);
            const int ux0 = __shfl_sync(FULL, x0, j), ux1 = __shfl_sync(FULL, x1, j), uy0 = __shfl_sync(FULL, y0, j),
                      uy1 = __shfl_sync(FULL, y1, j), uz0 = __shfl_sync(FULL, z0, j), uz1 = __shfl_sync(FULL, z1, j);
            const int64_t ugq = __shfl_sync(FULL, gq, j);
            const bool ubld = BUILD && (__shfl_sync(FULL, (int)bld, j) != 0);
            int uext = BUILD ? __shfl_sync(FULL, ext_slot, j) : -1;
            const float ulo = BUILD ? __shfl_sync(FULL, lo, j) : 0.f;
            int lc = 0;
            const int nyr = uy1 - uy0 + 1;
            const int nrows = (ux0 > ux1 || uy0 > uy1 || uz0 > uz1) ? 0 : nyr * (uz1 - uz0 + 1);   // 0: nothing to scan, the warm start stands
            for (int rbase = 0; rbase < nrows; rbase += 32) {
                // ---- the rows of this round: one per lane ----
                const int r = rbase + lane;
                int32_t p = 0, len = 0;
                if (r < nrows) {
                    const int zz = uz0 + r / nyr, yy = uy0 + r % nyr;
                    const float tz = axis_lb(fz, (float)zz, 1.f), ty = axis_lb(fy, (float)yy, 1.f);
                    const float lb = (ty * ty + tz * tz) * (1.f - 6e-7f);
                    if (lb <= bestc) {
                        // cells of this row the ball can reach: |x - fx| <= sqrt(bestc - lb) (+ slop)
                        const float rx = __fsqrt_ru(bestc - lb) * (1.f + 1e-6f) + 2.f * GRID_SLOP_ABS + GRID_SLOP_REL * fabsf(fx);
                        const int xa = max(ux0, (int)floorf(fx - rx)), xb = min(ux1, (int)floorf(fx + rx));
                        if (xa <= xb) {
                            const int64_t c0 = ((int64_t)zz * dy0 + yy) * dx0;
                            p = G.cell_start[c0 + xa];
                            len = G.cell_start[c0 + xb + 1] - p;
                        }
                    }
                }
                if (len > 0) { ++n_cells; n_pts += (unsigned long long)len; }
                int incl = len;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(FULL, incl, o);
                    if (lane >= o) incl += t;
                }
                const int T = __shfl_sync(FULL, incl, 31);
                const int excl = incl - len;
                // ---- the points of those rows: consecutive lanes take consecutive points of the flat range ----
                for (int tb = 0; tb < T; tb += 32 * ROWS_U) {
                    // ROWS_U x 32 points per trip: all their gathers are issued before the first one is used
                    GridPoint gpu[ROWS_U];
                    int32_t posu[ROWS_U];
#pragma unroll
                    for (int u = 0; u < ROWS_U; ++u) {
                        const int t = tb + 32 * u + lane;
                        int s = 0;                               // first row whose inclusive count exceeds t
#pragma unroll
                        for (int step = 16; step >= 1; step >>= 1) {
                            const int v = __shfl_sync(FULL, incl, min(s + step - 1, 31));
                            if (v <= t) s += step;
                        }
                        s = min(s, 31);
                        const int32_t ps = __shfl_sync(FULL, p, s);
                        const int ex = __shfl_sync(FULL, excl, s);
                        posu[u] = (t < T) ? ps + (t - ex) : -1;
                        if (posu[u] >= 0) gpu[u] = G.pts[posu[u]];
                    }
#pragma unroll
                    for (int u = 0; u < ROWS_U; ++u) {
                        if (tb + 32 * u >= T) break;             // warp-uniform
                        const bool act = posu[u] >= 0;
                        const int32_t pos = posu[u];
                        double d = INFINITY;
                        if (act) {
                            const GridPoint gp = gpu[u];
                            d = dist2_exact(gp.x, gp.y, gp.z, qx, qy, qz);
                            if (d < best || (d == best && gp.orig < bidx)) { best = d; bidx = gp.orig; }
                        }
                        if (BUILD && ubld) {
                            // list threshold from the warp's best so far (an upper bound of the final one)
                            const unsigned mb = __reduce_min_sync(FULL, __float_as_uint(__double2float_ru(best)));
                            const double thr2 = list_thr2((double)__uint_as_float(mb), a.cl.skin);
                            const bool app = act && d <= thr2;
                            const unsigned am = __ballot_sync(FULL, app);
                            if (am) {
                                const int n = __popc(am);
                                if (lc + n > a.cl.cap && uext == -1) {       // first entry beyond the query's own row: take an extension slot
                                    unsigned sl = 0;
                                    if (lane == 0) sl = atomicAdd(a.cl.ext_count, 1u);
                                    sl = __shfl_sync(FULL, sl, 0);
                                    uext = sl < (unsigned)a.cl.ext_slots ? (int)sl : -2;                 // -2: pool exhausted
                                }
                                if (app) {
                                    const float sd = __fsqrt_rd(__double2float_rd(d));
                                    const int level = min(max((int)floorf((sd - ulo) * a.cl.inv_level) - 1, 0), 255);
                                    const int32_t entry = (int32_t)(((unsigned)pos << 8) | (unsigned)level);
                                    const int at = lc + __popc(am & lt_mask);
                                    if (at < a.cl.cap) {
                                        a.cl.list[ugq * a.cl.cap + at] = entry;
                                    } else {
                                        const int k = at - a.cl.cap;
                                        if (uext >= 0 && k < a.cl.ext_cap) a.cl.ext_list[(int64_t)uext * a.cl.ext_cap + k] = entry;
                                    }
                                }
                                lc += n;
                            }
                        }
                    }
                }
                if (rbase + 32 < nrows) {                        // tighten the pruning bound for the next round of rows
                    const float mb = __uint_as_float(__reduce_min_sync(FULL, __float_as_uint(__double2float_ru(best))));
                    bestc = ubld ? best_ub_cells_gap((double)mb, G.inv_cell, a.cl.gap_cells) : best_ub_cells((double)mb, inv_cell2);
                }
            }
            // ---- the warp's winner on (d2, original index) ----
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(FULL, best, o);
                const int32_t oi = __shfl_xor_sync(FULL, bidx, o);
                if (ob < best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
            }
            if (lane == j) {
                a.idx[gq] = bidx;
                if (a.d2) a.d2[gq] = best;
                if (BUILD) {
                    Q.best = best; Q.bidx = bidx;
                    list_commit(a.cl, G, gq, Q, bld, lc, uext, lo);
                }
            }
        }
    }
    flush_counters(a.counters, n_pts, n_cells, 0);
}

// ---- kernel 0: candidate-list scan -------------------------------------------------------------------------
// Bound by the gather rate of the model points (one L1 wavefront per lane and candidate), so most gathers are
// avoided: a candidate k was at distance d0_k from the build position q0, hence is at least d0_k - moved from the
// moved query, while the build-time neighbour is at most r0 + moved away.  Only candidates with
// d0_k <= r0 + 2 moved can win or tie; d0_k is stored on a 256-level scale in the low byte of the entry (rounded
// down), so the test is one integer compare and the skipped entries cost 4 streamed bytes each.
struct GP4 { double x, y, z; long long w; };     // one GridPoint as four 64-bit registers (orig in the low word of w)
__device__ __forceinline__ GP4 ldg_point(const GridPoint* p, bool use) {
    GP4 r;
    r.x = r.y = r.z = 1.0e300; r.w = 0x7fffffffll;       // an unused slot never wins
    if (use) asm volatile("ld.global.nc.v4.b64 {%0, %1, %2, %3}, [%4];" : "=d"(r.x), "=d"(r.y), "=d"(r.z), "=l"(r.w) : "l"(p));
    return r;
}
struct ListScan {
    const GridPoint* __restrict__ pts;
    double qx, qy, qz, best;
    int32_t bidx;
    int lmax;
    unsigned n_read, n_gather;
    __device__ __forceinline__ void take(const GP4& g) {
        const double d = dist2_exact(g.x, g.y, g.z, qx, qy, qz);
        const int32_t orig = (int32_t)(g.w & 0xffffffffll);
        if (d < best || (d == best && orig < bidx)) { best = d; bidx = orig; }
    }
    __device__ __forceinline__ void scan(const int32_t* __restrict__ L, int n) {
        const int4* __restrict__ L4 = reinterpret_cast<const int4*>(L);
        int4 nx = L4[0];
        for (int k = 0; k < n; k += 4) {
            const int4 e = nx;
            if (k + 4 < n) nx = L4[(k >> 2) + 1];
            const int m = n - k;                             // valid entries among the 4 (>= 1)
            const bool u0 = (e.x & 255) <= lmax, u1 = m > 1 && (e.y & 255) <= lmax, u2 = m > 2 && (e.z & 255) <= lmax,
                       u3 = m > 3 && (e.w & 255) <= lmax;
            const GP4 g0 = ldg_point(pts + ((unsigned)e.x >> 8), u0), g1 = ldg_point(pts + ((unsigned)e.y >> 8), u1);
            const GP4 g2 = ldg_point(pts + ((unsigned)e.z >> 8), u2), g3 = ldg_point(pts + ((unsigned)e.w >> 8), u3);
            if (u0) take(g0); if (u1) take(g1); if (u2) take(g2); if (u3) take(g3);
            n_read += (unsigned)min(m, 4);
            n_gather += (unsigned)u0 + (unsigned)u1 + (unsigned)u2 + (unsigned)u3;
        }
    }
};

__global__ void __launch_bounds__(128) k_nn_list(const __grid_constant__ GridArgs a) {
    const GridView& G = a.g;
    const int lane = threadIdx.x & 31;
    const int64_t gq = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool defer = false;
    unsigned n_read = 0, n_gather = 0;
    bool skipped = false;
    if (gq < a.nq && a.skip_thr) {
        // Lazy trimming: this query's residual was so far above the hypothesis' trim threshold that it cannot be among the
        // selected correspondences of this pass either (icp.cu).  Its correspondence is carried over and its residual
        // replaced by a lower bound (previous residual minus the largest possible motion), which keeps it out of the
        // selection and makes the same test valid in the next pass.
        const unsigned h = (unsigned)gq / (unsigned)a.ns;
        const double sd = sqrt(a.d2[gq]);
        if (sd * (1.0 - 1e-12) > a.skip_thr[h]) {
            const double nl = sd * (1.0 - 1e-12) - (double)a.cl.delta[h] * (1.0 + 1e-6);
            a.d2[gq] = nl * nl * (1.0 - 1e-12);
            a.idx[gq] = a.prev[gq];
            skipped = true;
        }
    }
    if (gq < a.nq && !skipped) {
        const int2 cs = a.cl.cnt[gq];
        const int cnt = cs.x;
        if (cnt <= 0) {
            defer = true;
        } else {
            const float4 hd = a.cl.hdr[gq];
            const unsigned h = (unsigned)gq / (unsigned)a.ns, i = (unsigned)gq - h * (unsigned)a.ns;
            ListScan S;
            S.pts = G.pts;
            quick_tf(a.T + (size_t)h * 16, a.sx[i], a.sy[i], a.sz[i], S.qx, S.qy, S.qz);
            S.best = INFINITY; S.bidx = -1; S.n_read = 0; S.n_gather = 0;
            // upper bound of |q - q0| (q0 = position when the list was built; both rounded to FP32 here)
            const float fx = __double2float_rn(S.qx - G.origin[0]), fy = __double2float_rn(S.qy - G.origin[1]), fz = __double2float_rn(S.qz - G.origin[2]);
            const float ex = fx - hd.x, ey = fy - hd.y, ez = fz - hd.z;
            float moved = __fsqrt_ru(__fmaf_ru(ex, ex, __fmaf_ru(ey, ey, __fmul_ru(ez, ez))));
            moved = moved * (1.f + 1e-6f) + 3e-7f * (fabsf(fx) + fabsf(fy) + fabsf(fz) + fabsf(hd.x) + fabsf(hd.y) + fabsf(hd.z)) + 1e-30f;
            const float skin = (float)a.cl.skin;
            // r0 = R_list - skin (upper bound); levels whose lower edge lies beyond r0 + 2 moved cannot matter
            const float reach = __fadd_ru(hd.w * (1.f + 1e-6f) - skin * (1.f - 1e-5f), 2.f * moved);
            const float lv = (reach - __int_as_float(cs.y)) * a.cl.inv_level;
            S.lmax = (lv >= 254.f) ? 255 : max((int)floorf(lv) + 1, 0);
            S.scan(a.cl.list + gq * a.cl.cap, min(cnt, a.cl.cap));
            if (cnt > a.cl.cap) S.scan(a.cl.ext_list + (int64_t)a.cl.ext[gq] * a.cl.ext_cap, cnt - a.cl.cap);
            // a model point outside the list is farther than R_list - moved from q: is the list's best closer?
            const float r1 = __fsqrt_ru(__double2float_ru(S.best));
            if (S.bidx >= 0 && __fadd_ru(r1, moved) * (1.f + 1e-6f) < hd.w) {
                a.idx[gq] = S.bidx;
                if (a.d2) a.d2[gq] = S.best;
            } else {
                defer = true;
            }
            n_read = S.n_read; n_gather = S.n_gather;
        }
    }
    worklist_append(a, defer, gq, lane);
    if (a.counters) flush_counters(a.counters, n_read, n_gather, skipped ? 1ull : 0ull, 6, 7, 10);
}

// ---- kernel 2: pyramid walk --------------------------------------------------------------------------------
// worklist != nullptr: the queries the direct kernel handed over (wide balls), warm-started by the caller's previous
// correspondences.  worklist == nullptr (first ICP pass, pcreg_nn_search): EVERY query, in chains of WALK_CHAIN
// consecutive queries per thread -- the source cloud is spatially sorted, so the answer of one query is a tight
// bound for the next and only the first query of a chain descends from the root.
constexpr int WALK_CHAIN = 3;

template <bool BUILD>
__global__ void __launch_bounds__(128) k_nn_grid_walk(const __grid_constant__ GridArgs a) {
    const GridView& G = a.g;
    const bool chained = (a.worklist == nullptr);
    const int64_t count = chained ? (a.nq + a.chain - 1) / a.chain : (int64_t)*a.work_count;
    if (a.counters && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&a.counters[4], (unsigned long long)(chained ? a.nq : count));
    unsigned long long n_pts = 0, n_cells = 0, n_nodes = 0;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < count; w += (int64_t)gridDim.x * blockDim.x) {
        const int nchain = chained ? (int)min((int64_t)a.chain, a.nq - w * a.chain) : 1;
        int32_t warm = -1;
        for (int j = 0; j < nchain; ++j) {
            const int64_t gq = chained ? w * a.chain + j : (int64_t)a.worklist[w];
            if (!chained) warm = a.prev ? a.prev[gq] : -1;
            bool bld = false;
            int lc = 0, ext_slot = -1;
            double thr2 = 0.0;
            float gap = 0.f;
            if (BUILD) {
                bld = !a.cl.delta || a.cl.delta[(unsigned)gq / (unsigned)a.ns] <= a.cl.build_max_delta;
                gap = bld ? a.cl.gap_cells : 0.f;
            }
            Query Q;
            setup_query(a, gq, Q, gap, warm);
            float lo = 0.f;
            if (BUILD && bld) {
                ext_slot = a.cl.ext[gq]; thr2 = list_thr2(Q.best, a.cl.skin);
                lo = __fsqrt_rd(__double2float_rd(Q.best)) - (float)a.cl.skin;
            }
            walk_search<BUILD>(a, gq, Q, bld, lc, ext_slot, thr2, lo, n_pts, n_cells, n_nodes);
            a.idx[gq] = Q.bidx;
            if (a.d2) a.d2[gq] = Q.best;
            if (BUILD) list_commit(a.cl, G, gq, Q, bld, lc, ext_slot, lo);
            else if (a.cl.cnt) a.cl.cnt[gq] = make_int2(-1, 0);
            warm = Q.bidx;
        }
    }
    flush_counters(a.counters, n_pts, n_cells, n_nodes, 8, 9);
}

// ---- kernel 2b: pyramid walk, one WARP per query (dense models, warm-started work list) ----------------------
// The per-lane walk above scans a dense model's leaves (13 points per occupied cell on C5) one point per lane and
// trip, at 8-9 active lanes.  Here the 32 lanes descend the pyramid together, level by level: the frontier of nodes whose
// box can still reach the ball lives in shared memory, one lane takes one (node, child) pair -- occupancy bit, box
// bound, ballot-compacted append to the next frontier -- and the level-0 frontier (leaf cells) is then handled like the
// rows of k_nn_grid_rows: a warp scan of the run lengths, consecutive lanes on consecutive points, two gather rounds in
// flight, the bound re-tightened between rounds of 32 leaves, ballot-compacted list entries (BUILD).  The bound is the
// warm start, so the breadth-first order costs no pruning power worth mentioning; a query whose frontier outgrows the
// buffer (or that has no bound) is handed to the per-lane walk through a second work list.  Exactness: identical
// pruning tests (box_lb vs the upper bound of the best distance, ties never pruned), every visited point in FP64,
// winner on (d2, original index).
constexpr int WW_CAP = 512;             // frontier entries per warp
constexpr int WW_WARPS = 4;
template <bool BUILD>
__global__ void __launch_bounds__(32 * WW_WARPS, 6) k_nn_grid_walk_warp(const __grid_constant__ GridArgs a) {
    __shared__ unsigned s_node[WW_WARPS][2][WW_CAP];     // z << 20 | y << 10 | x
    __shared__ float s_lb[WW_WARPS][2][WW_CAP];
    const GridView& G = a.g;
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int64_t count = (int64_t)*a.work_count;
    const double inv_cell2 = G.inv_cell * G.inv_cell;
    const int dx0 = G.dims[0][0], dy0 = G.dims[0][1];
    unsigned long long n_pts = 0, n_cells = 0, n_nodes = 0, n_done = 0;

    while (true) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(a.cursor, 1ull);
        w = __shfl_sync(FULL, w, 0);
        if ((int64_t)w >= count) break;
        // ---- setup, identical on every lane ----
        const int64_t gq = (int64_t)a.worklist[w];
        const int32_t warm = a.prev ? a.prev[gq] : -1;
        bool bld = false;
        float gap = 0.f;
        if (BUILD) {
            bld = !a.cl.delta || a.cl.delta[(unsigned)gq / (unsigned)a.ns] <= a.cl.build_max_delta;
            gap = bld ? a.cl.gap_cells : 0.f;
        }
        Query Q;
        setup_query(a, gq, Q, gap, warm);
        bool overflow = !Q.has_span;                         // no bound: the per-lane walk descends from the root
        const float fx = Q.fx, fy = Q.fy, fz = Q.fz;
        const double qx = Q.qx, qy = Q.qy, qz = Q.qz;
        double best = Q.best;
        int32_t bidx = Q.bidx;
        float bestc = Q.bestc;
        int cur = 0, n = 0, level = 0;
        if (!overflow) {
            // lowest level whose <= 2 x 2 x 2 nodes cover the ball's bounding cube (else the root)
            const int top = G.nlevels - 1;
            int l = 0;
            while (l < top && (((Q.ihx >> l) - (Q.ilx >> l)) > 1 || ((Q.ihy >> l) - (Q.ily >> l)) > 1 || ((Q.ihz >> l) - (Q.ilz >> l)) > 1)) ++l;
            level = l;
            bool ok = false;
            unsigned nd = 0;
            float lb = 0.f;
            if (l == top) {                                      // the root (1 x 1 x 1) wherever the ball lies
                if (lane == 0) { lb = box_lb(fx, fy, fz, 0, 0, 0, (float)(1 << l)); ok = lb <= bestc; nd = 0u; }
            } else if (lane < 8) {
                const int x = (Q.ilx >> l) + (lane & 1), y = (Q.ily >> l) + ((lane >> 1) & 1), z = (Q.ilz >> l) + (lane >> 2);
                const int dxl = G.dims[l][0], dyl = G.dims[l][1], dzl = G.dims[l][2];
                if (x <= (Q.ihx >> l) && y <= (Q.ihy >> l) && z <= (Q.ihz >> l) && x >= 0 && y >= 0 && z >= 0 && x < dxl && y < dyl && z < dzl &&
                    (l == 0 || G.mask[l][((int64_t)z * dyl + y) * dxl + x] != 0)) {
                    lb = box_lb(fx, fy, fz, x, y, z, (float)(1 << l));
                    ok = lb <= bestc;
                    nd = (unsigned)x | ((unsigned)y << 10) | ((unsigned)z << 20);
                }
            }
            const unsigned bm = __ballot_sync(FULL, ok);
            if (ok) { const int at = __popc(bm & lt_mask); s_node[warp][0][at] = nd; s_lb[warp][0][at] = lb; }
            n = __popc(bm);
            __syncwarp();
        }
        // ---- descend: frontier at `level` -> frontier at level - 1 ----
        while (!overflow && level >= 1) {
            const int dxl = G.dims[level][0], dyl = G.dims[level][1];
            const float edge = (float)(1 << (level - 1));       // child edge in cells
            const uint8_t* __restrict__ mk = G.mask[level];
            int nn = 0;
            for (int base = 0; base < 8 * n; base += 32) {
                const int it = base + lane;
                bool ok = false;
                unsigned child = 0;
                float lb = 0.f;
                if (it < 8 * n) {
                    const unsigned nd = s_node[warp][cur][it >> 3];
                    const int k = it & 7;
                    const int ix = (int)(nd & 1023u), iy = (int)((nd >> 10) & 1023u), iz = (int)(nd >> 20);
                    const unsigned m = mk[((int64_t)iz * dyl + iy) * dxl + ix];
                    if ((m >> k) & 1u) {
                        const int cx = 2 * ix + (k & 1), cy = 2 * iy + ((k >> 1) & 1), cz = 2 * iz + (k >> 2);
                        lb = box_lb(fx, fy, fz, cx, cy, cz, edge);
                        ok = lb <= bestc;
                        child = (unsigned)cx | ((unsigned)cy << 10) | ((unsigned)cz << 20);
                    }
                }
                const unsigned bm = __ballot_sync(FULL, ok);
                const int at = nn + __popc(bm & lt_mask);
                if (ok && at < a.ww_cap) { s_node[warp][cur ^ 1][at] = child; s_lb[warp][cur ^ 1][at] = lb; }
                nn += __popc(bm);
            }
            if (lane == 0) n_nodes += (unsigned long long)n;
            __syncwarp();
            if (nn > a.ww_cap) { overflow = true; break; }
            cur ^= 1; n = nn; --level;
        }
        if (overflow) {                                          // the per-lane walk takes it from here
            if (lane == 0) a.overflow[atomicAdd(a.overflow_count, 1u)] = (int32_t)gq;
            continue;
        }
        // ---- leaves: the frontier is a set of level-0 cells ----
        int lc = 0, uext = -1;
        float lo = 0.f;
        if (BUILD && bld) {
            uext = a.cl.ext[gq];
            lo = __fsqrt_rd(__double2float_rd(Q.best)) - (float)a.cl.skin;      // every listed point is within [.., lo + 2 skin]
        }
        for (int rbase = 0; rbase < n; rbase += 32) {
            const int r = rbase + lane;
            int32_t p = 0, len = 0;
            if (r < n && s_lb[warp][cur][r] <= bestc) {
                const unsigned nd = s_node[warp][cur][r];
                const int64_t c = ((int64_t)(nd >> 20) * dy0 + (int64_t)((nd >> 10) & 1023u)) * dx0 + (int64_t)(nd & 1023u);
                p = G.cell_start[c];
                len = G.cell_start[c + 1] - p;
                ++n_cells;
                n_pts += (unsigned long long)len;
            }
            int incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += t;
            }
            const int T = __shfl_sync(FULL, incl, 31);
            const int excl = incl - len;
            // (same point loop as k_nn_grid_rows)
            for (int tb = 0; tb < T; tb += 32 * ROWS_U) {
                GridPoint gpu[ROWS_U];
                int32_t posu[ROWS_U];
#pragma unroll
                for (int u = 0; u < ROWS_U; ++u) {
                    const int t = tb + 32 * u + lane;
                    int s = 0;                               // first leaf whose inclusive count exceeds t
#pragma unroll
                    for (int step = 16; step >= 1; step >>= 1) {
                        const int v = __shfl_sync(FULL, incl, min(s + step - 1, 31));
                        if (v <= t) s += step;
                    }
                    s = min(s, 31);
                    const int32_t ps = __shfl_sync(FULL, p, s);
                    const int ex = __shfl_sync(FULL, excl, s);
                    posu[u] = (t < T) ? ps + (t - ex) : -1;
                    if (posu[u] >= 0) gpu[u] = G.pts[posu[u]];
                }
#pragma unroll
                for (int u = 0; u < ROWS_U; ++u) {
                    if (tb + 32 * u >= T) break;             // warp-uniform
                    const bool act = posu[u] >= 0;
                    const int32_t pos = posu[u];
                    double d = INFINITY;
                    if (act) {
                        const GridPoint gp = gpu[u];
                        d = dist2_exact(gp.x, gp.y, gp.z, qx, qy, qz);
                        if (d < best || (d == best && gp.orig < bidx)) { best = d; bidx = gp.orig; }
                    }
                    if (BUILD && bld) {
                        const unsigned mb = __reduce_min_sync(FULL, __float_as_uint(__double2float_ru(best)));
                        const double thr2 = list_thr2((double)__uint_as_float(mb), a.cl.skin);
                        const bool app = act && d <= thr2;
                        const unsigned am = __ballot_sync(FULL, app);
                        if (am) {
                            const int na = __popc(am);
                            if (lc + na > a.cl.cap && uext == -1) {
                                unsigned sl = 0;
                                if (lane == 0) sl = atomicAdd(a.cl.ext_count, 1u);
                                sl = __shfl_sync(FULL, sl, 0);
                                uext = sl < (unsigned)a.cl.ext_slots ? (int)sl : -2;
                            }
                            if (app) {
                                const float sd = __fsqrt_rd(__double2float_rd(d));
                                const int lvl = min(max((int)floorf((sd - lo) * a.cl.inv_level) - 1, 0), 255);
                                const int32_t entry = (int32_t)(((unsigned)pos << 8) | (unsigned)lvl);
                                const int at = lc + __popc(am & lt_mask);
                                if (at < a.cl.cap) {
                                    a.cl.list[gq * a.cl.cap + at] = entry;
                                } else {
                                    const int k = at - a.cl.cap;
                                    if (uext >= 0 && k < a.cl.ext_cap) a.cl.ext_list[(int64_t)uext * a.cl.ext_cap + k] = entry;
                                }
                            }
                            lc += na;
                        }
                    }
                }
            }
            if (rbase + 32 < n) {                            // tighten the bound for the next round of leaves
                const float mb = __uint_as_float(__reduce_min_sync(FULL, __float_as_uint(__double2float_ru(best))));
                bestc = (BUILD && bld) ? best_ub_cells_gap((double)mb, G.inv_cell, a.cl.gap_cells) : best_ub_cells((double)mb, inv_cell2);
            }
        }
        if (lane == 0) n_nodes += (unsigned long long)n;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(FULL, best, o);
            const int32_t oi = __shfl_xor_sync(FULL, bidx, o);
            if (ob < best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
        }
        if (lane == 0) {
            a.idx[gq] = bidx;
            if (a.d2) a.d2[gq] = best;
            Q.best = best; Q.bidx = bidx;
            if (BUILD) list_commit(a.cl, G, gq, Q, bld, lc, uext, lo);
            else if (a.cl.cnt) a.cl.cnt[gq] = make_int2(-1, 0);
            ++n_done;
        }
        __syncwarp();
    }
    if (a.counters) {
        flush_counters(a.counters, n_pts, n_cells, n_nodes, 8, 9);
        if (lane == 0 && n_done) atomicAdd(&a.counters[4], n_done);
    }
}

void nn_grid_launch(const pcreg_model* m, const double* d_sx, const double* d_sy, const double* d_sz, int64_t ns,
                    const double* d_T, int64_t nhyp, const int32_t* d_prev, int32_t* d_idx, double* d_d2,
                    unsigned long long* d_counters, GridScratch& sc, const CandView* cl, bool scan_lists, const double* d_skip_thr,
                    cudaStream_t st, const int32_t* d_stop_iter) {
    PCREG_REQUIRE(m->has_grid, "grid NN requested but the model was created without build_grid");
    GridArgs a{};
    a.g = m->grid; a.md = m->md.p;
    a.sx = d_sx; a.sy = d_sy; a.sz = d_sz; a.ns = ns; a.T = d_T; a.nq = nhyp * ns;
    a.prev = d_prev; a.idx = d_idx; a.d2 = d_d2; a.counters = d_counters;
    if (cl) a.cl = *cl;
    a.skip_thr = (cl && scan_lists && d_prev) ? d_skip_thr : nullptr;
    static const int row_span_env = [] { const char* e = getenv("PCREG_ROW_SPAN"); return e ? atoi(e) : 0; }();
    a.row_span = row_span_env > 0 ? row_span_env : GRID_ROW_SPAN;
    static const int fb_env = [] { const char* e = getenv("PCREG_FETCH_BATCH"); return e ? atoi(e) : 0; }();
    static const int ch_env = [] { const char* e = getenv("PCREG_CHUNK"); return e ? atoi(e) : 0; }();
    static const int chain_env = [] { const char* e = getenv("PCREG_WALK_CHAIN"); return e ? atoi(e) : 0; }();
    a.chain = chain_env > 0 ? chain_env : WALK_CHAIN;
    a.fetch_batch = std::min(32, fb_env > 0 ? fb_env : GRID_FETCH_BATCH); a.chunk = std::max(1, ch_env > 0 ? ch_env : GRID_CHUNK);
    PCREG_REQUIRE(a.nq > 0, "nn_grid: no queries");
    PCREG_REQUIRE(a.nq < 2147483647LL, "nn_grid: too many queries in one launch");
    PCREG_REQUIRE(!cl || (int64_t)cl->cap * a.nq < ((int64_t)1 << 40), "nn_grid: candidate lists too large");
    PCREG_REQUIRE(!cl || m->n <= ((int64_t)1 << 24), "nn_grid: candidate lists address at most 2^24 model points");
    auto mark = [&](int kind) {
        if (!sc.timing) return;
        cudaEvent_t ev = pooled_event((*sc.ev_cursor)++);
        PCREG_CUDA(cudaEventRecord(ev, st));
        sc.timing->push_back(GridScratch::Mark{kind, ev});
    };
    const int64_t blocks = (a.nq + 127) / 128;
    static const int wcap_env = [] { const char* e = getenv("PCREG_WALK_CAP"); return e ? atoi(e) : 0; }();
    const int64_t wcap = (int64_t)ctx().sm_count * (wcap_env > 0 ? wcap_env : 256);
    const int walk_blocks = (int)std::min<int64_t>(blocks, wcap);
    if (m->has_vox && !cl) {
        // Voronoi voxel map (nn_vox.cu): one list scan per query; the few queries whose voxel has no list (or that lie outside
        // the padded box) are walked, warm-started by the previous correspondence when there is one.
        a.vox = m->vox;
        a.stop_iter = d_stop_iter;
        if (sc.worklist.n < (size_t)a.nq) sc.worklist.alloc((size_t)a.nq);
        if (sc.count.n < 2) sc.count.alloc(2);
        PCREG_CUDA(cudaMemsetAsync(sc.count.p, 0, 2 * sizeof(unsigned int), st));
        a.worklist = sc.worklist.p; a.work_count = sc.count.p;
        mark(0);
        nn_vox_launch(m, a, st);
        mark(2);
        k_nn_grid_walk<false><<<(int)std::min<int64_t>(blocks, (int64_t)ctx().sm_count * 16), 128, 0, st>>>(a);
        PCREG_LAUNCHED();
        mark(3);
        return;
    }
    if (d_prev) {
        if (sc.worklist.n < (size_t)a.nq) sc.worklist.alloc((size_t)a.nq);
        if (sc.count.n < 2) sc.count.alloc(2);
        PCREG_CUDA(cudaMemsetAsync(sc.count.p, 0, 2 * sizeof(unsigned int), st));
        const int direct_blocks = (int)std::min<int64_t>(blocks, (int64_t)ctx().sm_count * 16);
        if (cl && scan_lists) {
            if (sc.worklist0.n < (size_t)a.nq) sc.worklist0.alloc((size_t)a.nq);
            a.worklist = sc.worklist0.p; a.work_count = sc.count.p + 1;
            mark(0);
            k_nn_list<<<(unsigned)blocks, 128, 0, st>>>(a);
            PCREG_LAUNCHED();
            a.in_list = sc.worklist0.p; a.in_count = sc.count.p + 1;
        }
        a.worklist = sc.worklist.p; a.work_count = sc.count.p;
        if (sc.cursor.n < 1) sc.cursor.alloc(1);
        PCREG_CUDA(cudaMemsetAsync(sc.cursor.p, 0, sizeof(unsigned long long), st));
        a.cursor = sc.cursor.p;
        mark(1);
        // dense models (many points per occupied cell, hundreds of points per query): one warp per query with coalesced
        // runs; sparse models: the per-lane state machine.  PCREG_ROWSCAN=lane|warp forces one of them.
        const char* rows_e = getenv("PCREG_ROWSCAN");            // read per launch: the tests flip it inside one process
        const int rows_env = !rows_e ? 0 : (rows_e[0] == 'w' ? 2 : (rows_e[0] == 'l' ? 1 : 0));
        const bool warp_rows = rows_env ? rows_env == 2 : (double)m->n >= GRID_WARP_ROWS_DENSITY * (double)std::max<int64_t>(m->g_occupied, 1);
        if (warp_rows) {
            if (cl) k_nn_grid_rows<true><<<direct_blocks, 128, 0, st>>>(a);
            else    k_nn_grid_rows<false><<<direct_blocks, 128, 0, st>>>(a);
        } else {
            if (cl) k_nn_grid_direct<true><<<direct_blocks, 128, 0, st>>>(a);
            else    k_nn_grid_direct<false><<<direct_blocks, 128, 0, st>>>(a);
        }
        PCREG_LAUNCHED();
        a.in_list = nullptr; a.in_count = nullptr;
        mark(2);
        // dense models: warp-per-query walk first, the per-lane walk then takes what that one hands on.  PCREG_WALK=lane|warp forces.
        const char* walk_e = getenv("PCREG_WALK");
        const int walk_env = !walk_e ? 0 : (walk_e[0] == 'w' ? 2 : (walk_e[0] == 'l' ? 1 : 0));
        // (from the third NN pass on -- scan_lists is "pass >= 2": right after the first pose update the warm-start bound is loose and the
        // breadth-first frontier visits 1.6x the points of the nearest-first per-lane walk; measured on C5: 8.0 vs 4.9 ms in that pass)
        const bool warp_walk = walk_env ? walk_env == 2
                                        : (scan_lists && (double)m->n >= GRID_WARP_ROWS_DENSITY * (double)std::max<int64_t>(m->g_occupied, 1));
        if (warp_walk) {
            if (sc.worklist0.n < (size_t)a.nq) sc.worklist0.alloc((size_t)a.nq);
            PCREG_CUDA(cudaMemsetAsync(sc.cursor.p, 0, sizeof(unsigned long long), st));     // the row scan is done with both
            PCREG_CUDA(cudaMemsetAsync(sc.count.p + 1, 0, sizeof(unsigned int), st));
            a.overflow = sc.worklist0.p; a.overflow_count = sc.count.p + 1;
            const char* cap_e = getenv("PCREG_WW_CAP");
            a.ww_cap = cap_e ? std::min(std::max(atoi(cap_e), 8), WW_CAP) : WW_CAP;          // >= 8: the start frontier always fits
            const int ww_blocks = (int)std::min<int64_t>((a.nq + WW_WARPS - 1) / WW_WARPS, (int64_t)ctx().sm_count * 12);
            if (cl) k_nn_grid_walk_warp<true><<<ww_blocks, 32 * WW_WARPS, 0, st>>>(a);
            else    k_nn_grid_walk_warp<false><<<ww_blocks, 32 * WW_WARPS, 0, st>>>(a);
            PCREG_LAUNCHED();
            a.worklist = sc.worklist0.p; a.work_count = sc.count.p + 1;
        }
        if (cl) k_nn_grid_walk<true><<<walk_blocks, 128, 0, st>>>(a);
        else    k_nn_grid_walk<false><<<walk_blocks, 128, 0, st>>>(a);
        PCREG_LAUNCHED();
        mark(3);
    } else {
        a.worklist = nullptr; a.work_count = nullptr;
        const int64_t chains = (a.nq + a.chain - 1) / a.chain;
        const int chain_blocks = (int)std::min<int64_t>((chains + 127) / 128, wcap);
        mark(2);
        k_nn_grid_walk<false><<<chain_blocks, 128, 0, st>>>(a);
        PCREG_LAUNCHED();
        mark(3);
    }
}

}  // namespace pcreg
