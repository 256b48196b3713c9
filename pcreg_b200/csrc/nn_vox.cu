// nn_vox.cu -- Voronoi voxel map: exact nearest neighbour as ONE short contiguous list scan per query.
//
// Semantics identical to nn_brute.cu / nn_grid.cu (knnsearch K=1, FP64, ties -> smallest original index; the
// reference's only literal cloud->cloud 1-NN loop is ColorCodeModel.m:15-18, its spatial pruning analogue the
// cube pre-filter of getLocalPoints.m:8-15 and the halo boxes of speedyDescriptors.m:44-60).
//
// Idea.  The pyramid walk and the row scan of nn_grid.cu spend ~2000 warp instructions per query deciding WHICH
// points to look at; HBM is idle.  B200 has 180 GB of it, so the decision is made once per model instead: the padded
// bounding box is cut into voxels of about one point spacing, and every voxel V stores N(V), a conservative superset
// of { p : p is a nearest neighbour of some location x in V }.  The nearest neighbour of a query in V is in N(V) by
// construction -- ties included -- so a query is: voxel index -> (first, count) -> scan `count` contiguous 16-byte
// entries in FP32 -> decide among the entries inside the FP32 error band in FP64 with the oracle's formula.
//
// Build (vox_build, once per model, on the device).  p can be a nearest neighbour somewhere in the box V (centre c,
// half edge e) only if it is at least as close as ANY other model point p0 somewhere in V:
//      min_{x in V} |x-p|^2 - |x-p0|^2  =  |a|^2 - |a0|^2 - 2 e ||a - a0||_1  <=  0,      a = p - c, a0 = p0 - c
// (the difference is linear in x, so the minimum sits in a corner).  Nine pivots p0 are used -- the list members
// nearest to the centre and to the eight corners -- and p is kept only if it passes all nine tests.  Lists are
// refined top-down: N(child) is filtered out of N(parent), which is correct because N(child) is a subset of
// N(parent) and the pivots are model points.  All build arithmetic is FP32 with margins that only ever ADD
// candidates.  Lists longer than a per-level cap are dropped (medial-axis regions, where thousands of points are
// almost equidistant): queries in such voxels, or outside the padded box, go to the pyramid walk of nn_grid.cu.
//
// Query (k_nn_vox): FP32 scan of d32 = |a_k - x|^2 with x = fl32(q - c).  Error bound (u = 2^-24, h0 = half
// diagonal of a voxel, D the true distance):  |d32 - D^2| <= 9u D^2 + 2u h0^2  (rounding of a_k, x, the difference
// and the three-term sum), so every entry that could be the true minimum or tie it satisfies
// d32 <= min32 (1 + 3e-6) + 1e-6 h0^2.  Those (normally one) are evaluated exactly in FP64 on the original
// coordinates and compete on (d2, original index).
#include <math.h>
#include <float.h>
#include <stdlib.h>
#include <stdio.h>
#include <time.h>
#include <algorithm>
#include <array>
#include <vector>

#include "pcreg_internal.h"
#include "pcreg_dev.cuh"
#include "pcreg_grid.cuh"
#include "pcreg_vox.cuh"

namespace pcreg {

constexpr uint32_t VOX_DROPPED = 0xffffffffu;   // intermediate levels: list dropped (too long / pool full); descendants inherit
constexpr int VOX_CHUNK = 512;                  // pool entries a warp reserves per atomic
constexpr int VOX_TOP_DIM = 16;                 // the top level (lists filtered out of ALL points) has at most this many voxels per axis
constexpr int VOX_BASE_CAP = 64;                // longest list kept at the finest level (x4 per level above)

struct VoxLevelArgs {
    const GridPoint* pts; uint32_t npts;
    const uint2* p_hdr; const int32_t* p_ids;   // parent level (brick order)
    int32_t pd[3], pt[3];                       // parent dims / tiles
    uint2* c_hdr; int32_t cd[3], ct[3];         // child level
    int32_t* c_ids; float4* c_ent;              // child lists: point positions (intermediate level) or entries (finest level)
    unsigned long long* pool_cursor; unsigned long long pool_cap;
    unsigned long long* work_cursor;            // next unassigned parent slot
    double origin[3]; double cs;                // child voxel edge
    uint32_t maxlen;
    float band;                                 // > 0: voxels farther than this from the model get no list (band-limited map of a dense model)
    unsigned long long* stats;                  // [0] listed voxels, [1] entries, [2] dropped: too long, [3] dropped: no room, [4] longest list,
                                                // [5] dropped: outside the band
};

struct Pivots { float x[9], y[9], z[9], n[9]; };

// keep p (a = p - c) unless one of the pivots is strictly closer everywhere in the (inflated) voxel
__device__ __forceinline__ bool vox_keep(float ax, float ay, float az, const Pivots& pv, float e2, float tol_abs) {
    const float na = fmaf(az, az, fmaf(ay, ay, ax * ax));
    bool keep = true;
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        const float l1 = fabsf(ax - pv.x[j]) + fabsf(ay - pv.y[j]) + fabsf(az - pv.z[j]);
        keep = keep && ((na - pv.n[j]) <= fmaf(e2, l1, fmaf(1e-5f, na + pv.n[j], tol_abs)));
    }
    return keep;
}
// per-lane running arg-min of the squared distance to the centre (j = 0) and to the eight corners of the voxel;
// key = distance bits << 32 | id (distances are shifted by a common constant, so only their order matters)
__device__ __forceinline__ void pivot_update(float ax, float ay, float az, float e, uint32_t id, unsigned long long (&best)[9]) {
    const float na = fmaf(az, az, fmaf(ay, ay, ax * ax));
    const float e2 = 2.f * e, off = 3.f * e * e;                       // |a - r|^2 = |a|^2 - 2 a.r + 3 e^2 >= 0
    const float sxy0 = ax + ay, sxy1 = ax - ay;
    float d[9];
    d[0] = na;
    d[1] = fmaf(-e2, sxy0 + az, na) + off;  d[2] = fmaf(-e2, sxy0 - az, na) + off;      // (+,+,+) (+,+,-)
    d[3] = fmaf(-e2, sxy1 + az, na) + off;  d[4] = fmaf(-e2, sxy1 - az, na) + off;      // (+,-,+) (+,-,-)
    d[5] = fmaf(e2, sxy1 - az, na) + off;   d[6] = fmaf(e2, sxy1 + az, na) + off;       // (-,+,+) (-,+,-)
    d[7] = fmaf(e2, sxy0 - az, na) + off;   d[8] = fmaf(e2, sxy0 + az, na) + off;       // (-,-,+) (-,-,-)
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        const unsigned long long key = ((unsigned long long)__float_as_uint(fmaxf(d[j], 0.f)) << 32) | (unsigned long long)id;
        best[j] = key < best[j] ? key : best[j];
    }
}
__device__ __forceinline__ void load_pivots(const GridPoint* __restrict__ pts, const unsigned long long (&best)[9], double cx, double cy,
                                            double cz, Pivots& pv) {
#pragma unroll
    for (int j = 0; j < 9; ++j) {
        const uint32_t id = (uint32_t)(best[j] & 0xffffffffull);
        const double px = pts[id].x, py = pts[id].y, pz = pts[id].z;
        pv.x[j] = __double2float_rn(px - cx); pv.y[j] = __double2float_rn(py - cy); pv.z[j] = __double2float_rn(pz - cz);
        pv.n[j] = fmaf(pv.z[j], pv.z[j], fmaf(pv.y[j], pv.y[j], pv.x[j] * pv.x[j]));
    }
}

// ---- coarse levels: one BLOCK per voxel ----------------------------------------------------------------------------------
// Candidates = ALL points (top level, HAS_PARENT = false: streamed, coalesced) or the parent's list (levels whose lists are
// still thousands of points long: a warp per parent would take seconds there).
template <bool HAS_PARENT>
__global__ void __launch_bounds__(256) k_vox_block(const __grid_constant__ VoxLevelArgs a) {
    __shared__ unsigned long long s_best[8][9];
    __shared__ unsigned long long s_piv[9];
    __shared__ unsigned int s_cnt, s_off, s_ok;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int cx, cy, cz;
    brick_decode((int64_t)blockIdx.x, a.ct, cx, cy, cz);
    if (cx >= a.cd[0] || cy >= a.cd[1] || cz >= a.cd[2]) return;            // padding slot of the brick layout
    const int64_t ci = brick_index(cx, cy, cz, a.ct);
    uint32_t n_c = a.npts;
    const int32_t* __restrict__ ids = nullptr;
    if (HAS_PARENT) {
        const uint2 ph = a.p_hdr[brick_index(cx >> 1, cy >> 1, cz >> 1, a.pt)];
        if (ph.y == VOX_DROPPED || ph.y == 0u) {                            // block-uniform
            if (tid == 0) a.c_hdr[ci] = make_uint2(0u, VOX_DROPPED);
            return;
        }
        n_c = ph.y;
        ids = a.p_ids + ph.x;
    }
    auto cand = [&](uint32_t t, uint32_t& id, double& x, double& y, double& z) {
        id = HAS_PARENT ? (uint32_t)ids[t] : t;
        x = a.pts[id].x; y = a.pts[id].y; z = a.pts[id].z;
    };
    const double ccx = vox_centre(a.origin[0], cx, a.cs), ccy = vox_centre(a.origin[1], cy, a.cs), ccz = vox_centre(a.origin[2], cz, a.cs);
    const float e = (float)(0.5 * a.cs * (1.0 + 1e-4));
    const float tol_abs = 1e-6f * e * e;
    // pass 1: pivots
    unsigned long long best[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) best[j] = ~0ull;
    for (uint32_t t = tid; t < n_c; t += 256) {
        uint32_t id; double px, py, pz;
        cand(t, id, px, py, pz);
        pivot_update(__double2float_rn(px - ccx), __double2float_rn(py - ccy), __double2float_rn(pz - ccz), e, id, best);
    }
#pragma unroll
    for (int j = 0; j < 9; ++j) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long ob = __shfl_xor_sync(0xffffffffu, best[j], o); best[j] = ob < best[j] ? ob : best[j]; }
        if (lane == 0) s_best[warp][j] = best[j];
    }
    if (tid == 0) { s_cnt = 0; s_ok = 0; }
    __syncthreads();
    if (tid < 9) {
        unsigned long long b = ~0ull;
        for (int w = 0; w < 8; ++w) b = s_best[w][tid] < b ? s_best[w][tid] : b;
        s_piv[tid] = b;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 9; ++j) best[j] = s_piv[j];
    Pivots pv;
    load_pivots(a.pts, best, ccx, ccy, ccz, pv);
    // pivot 0 is the model point nearest to the voxel centre: a voxel that lies wholly farther than `band` from the model is
    // left without a list (its queries are walked) -- block-uniform
    if (a.band > 0.f && sqrtf(pv.n[0]) - 1.7320509f * e > a.band) {
        if (tid == 0) { a.c_hdr[ci] = make_uint2(0u, VOX_DROPPED); atomicAdd(&a.stats[5], 1ull); }
        return;
    }
    // pass 2: count
    unsigned int cnt = 0;
    for (uint32_t t = tid; t < n_c; t += 256) {
        uint32_t id; double px, py, pz;
        cand(t, id, px, py, pz);
        cnt += vox_keep(__double2float_rn(px - ccx), __double2float_rn(py - ccy), __double2float_rn(pz - ccz), pv, 2.f * e, tol_abs) ? 1u : 0u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0 && cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    if (tid == 0) {
        const unsigned int total = s_cnt;
        if (total > a.maxlen) {
            a.c_hdr[ci] = make_uint2(0u, VOX_DROPPED);
            atomicAdd(&a.stats[2], 1ull);
        } else {
            const unsigned long long off = atomicAdd(a.pool_cursor, (unsigned long long)total);
            if (off + total > a.pool_cap) {
                a.c_hdr[ci] = make_uint2(0u, VOX_DROPPED);
                atomicAdd(&a.stats[3], 1ull);
            } else {
                a.c_hdr[ci] = make_uint2((unsigned int)off, total);
                s_off = (unsigned int)off; s_ok = 1;
                atomicAdd(&a.stats[0], 1ull); atomicAdd(&a.stats[1], (unsigned long long)total); atomicMax(&a.stats[4], (unsigned long long)total);
            }
        }
        s_cnt = 0;
    }
    __syncthreads();
    if (!s_ok) return;
    // pass 3: write (order within the list is irrelevant)
    const unsigned int off = s_off;
    for (uint32_t t0 = 0; t0 < n_c; t0 += 256) {
        const uint32_t t = t0 + tid;
        bool keep = false;
        uint32_t id = 0;
        if (t < n_c) {
            double px, py, pz;
            cand(t, id, px, py, pz);
            keep = vox_keep(__double2float_rn(px - ccx), __double2float_rn(py - ccy), __double2float_rn(pz - ccz), pv, 2.f * e, tol_abs);
        }
        const unsigned bm = __ballot_sync(0xffffffffu, keep);
        if (bm) {
            unsigned int base = 0;
            if (lane == 0) base = atomicAdd(&s_cnt, (unsigned)__popc(bm));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (keep) a.c_ids[off + base + __popc(bm & ((1u << lane) - 1u))] = (int32_t)id;
        }
    }
}

// ---- refinement: one WARP per parent voxel, the lists of its (up to) eight children filtered out of the parent's ------------
template <bool FINAL>
__global__ void __launch_bounds__(256) k_vox_refine(const __grid_constant__ VoxLevelArgs a) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const int64_t nslots = (int64_t)a.pt[0] * a.pt[1] * a.pt[2] * 64;
    unsigned long long w_off = 0, w_end = 0;                               // pool range reserved by this warp
    unsigned long long st_listed = 0, st_entries = 0, st_long = 0, st_room = 0, st_max = 0, st_far = 0;
    const float e = (float)(0.5 * a.cs * (1.0 + 1e-4));
    const float tol_abs = 1e-6f * e * e;

    while (true) {
        unsigned long long wbase = 0;
        if (lane == 0) wbase = atomicAdd(a.work_cursor, 32ull);
        wbase = __shfl_sync(FULL, wbase, 0);
        if ((int64_t)wbase >= nslots) break;
        const int64_t wend = min((int64_t)wbase + 32, nslots);
        for (int64_t slot = (int64_t)wbase; slot < wend; ++slot) {
            int px, py, pz;
            brick_decode(slot, a.pt, px, py, pz);
            if (px >= a.pd[0] || py >= a.pd[1] || pz >= a.pd[2]) continue;
            const uint2 ph = a.p_hdr[slot];
            const bool dropped = ph.y == VOX_DROPPED;
            const uint32_t n_p = dropped ? 0u : ph.y;
            const int32_t* __restrict__ ids = a.p_ids + ph.x;
            // the first 64 points of the parent's list stay in registers for all eight children
            uint32_t id0 = 0, id1 = 0;
            double x0 = 0, y0 = 0, z0 = 0, x1 = 0, y1 = 0, z1 = 0;
            if ((uint32_t)lane < n_p) { id0 = (uint32_t)ids[lane]; x0 = a.pts[id0].x; y0 = a.pts[id0].y; z0 = a.pts[id0].z; }
            if ((uint32_t)lane + 32u < n_p) { id1 = (uint32_t)ids[lane + 32]; x1 = a.pts[id1].x; y1 = a.pts[id1].y; z1 = a.pts[id1].z; }
            auto fetch = [&](uint32_t it, uint32_t& id, double& x, double& y, double& z) {
                if (it == 0) { id = id0; x = x0; y = y0; z = z0; }
                else if (it == 1) { id = id1; x = x1; y = y1; z = z1; }
                else { id = (uint32_t)ids[it * 32 + lane]; x = a.pts[id].x; y = a.pts[id].y; z = a.pts[id].z; }
            };
            for (int k = 0; k < 8; ++k) {
                const int cx = 2 * px + (k & 1), cy = 2 * py + ((k >> 1) & 1), cz = 2 * pz + (k >> 2);
                if (cx >= a.cd[0] || cy >= a.cd[1] || cz >= a.cd[2]) continue;
                const int64_t ci = brick_index(cx, cy, cz, a.ct);
                if (dropped || n_p == 0) {
                    if (lane == 0) a.c_hdr[ci] = make_uint2(0u, FINAL ? 0u : VOX_DROPPED);
                    continue;
                }
                const double ccx = vox_centre(a.origin[0], cx, a.cs), ccy = vox_centre(a.origin[1], cy, a.cs), ccz = vox_centre(a.origin[2], cz, a.cs);
                // sweep 1: pivots
                unsigned long long best[9];
#pragma unroll
                for (int j = 0; j < 9; ++j) best[j] = ~0ull;
                const uint32_t nit = (n_p + 31u) >> 5;
                for (uint32_t it = 0; it < nit; ++it) {
                    if (it * 32 + lane < n_p) {
                        uint32_t id; double x, y, z;
                        fetch(it, id, x, y, z);
                        pivot_update(__double2float_rn(x - ccx), __double2float_rn(y - ccy), __double2float_rn(z - ccz), e, id, best);
                    }
                }
#pragma unroll
                for (int j = 0; j < 9; ++j) {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) { const unsigned long long ob = __shfl_xor_sync(FULL, best[j], o); best[j] = ob < best[j] ? ob : best[j]; }
                }
                Pivots pv;
                load_pivots(a.pts, best, ccx, ccy, ccz, pv);
                if (a.band > 0.f && sqrtf(pv.n[0]) - 1.7320509f * e > a.band) {       // wholly outside the band (see k_vox_top)
                    if (lane == 0) a.c_hdr[ci] = make_uint2(0u, FINAL ? 0u : VOX_DROPPED);
                    ++st_far;
                    continue;
                }
                // sweep 2: count (the keep flags of the first 32 rounds are remembered)
                uint32_t cnt = 0, flags = 0;
                for (uint32_t it = 0; it < nit; ++it) {
                    bool keep = false;
                    if (it * 32 + lane < n_p) {
                        uint32_t id; double x, y, z;
                        fetch(it, id, x, y, z);
                        keep = vox_keep(__double2float_rn(x - ccx), __double2float_rn(y - ccy), __double2float_rn(z - ccz), pv, 2.f * e, tol_abs);
                    }
                    if (it < 32 && keep) flags |= 1u << it;
                    cnt += (uint32_t)__popc(__ballot_sync(FULL, keep));
                }
                if (cnt > a.maxlen) {
                    if (lane == 0) a.c_hdr[ci] = make_uint2(0u, FINAL ? 0u : VOX_DROPPED);
                    ++st_long;
                    continue;
                }
                // finest level: lists start on even entries and are padded to an even length with a far sentinel, so that the
                // scan reads PAIRS of entries with one 256-bit load (pcreg_vox.cuh)
                const uint32_t cnt_al = FINAL ? ((cnt + 1u) & ~1u) : cnt;
                if (w_off + cnt_al > w_end) {                            // reserve more pool space (one atomic per VOX_CHUNK entries)
                    const unsigned long long need = cnt_al > (uint32_t)VOX_CHUNK ? (unsigned long long)cnt_al : (unsigned long long)VOX_CHUNK;
                    unsigned long long o = 0;
                    if (lane == 0) o = atomicAdd(a.pool_cursor, need);
                    w_off = __shfl_sync(FULL, o, 0);
                    w_end = w_off + need;
                }
                if (w_end > a.pool_cap) {                                // pool exhausted: no list (the walk answers these queries)
                    if (lane == 0) a.c_hdr[ci] = make_uint2(0u, FINAL ? 0u : VOX_DROPPED);
                    ++st_room;
                    continue;
                }
                const unsigned long long off = w_off;
                w_off += cnt_al;
                if (FINAL && (cnt & 1u) && lane == 0) a.c_ent[off + cnt] = make_float4(1.0e18f, 1.0e18f, 1.0e18f, __int_as_float(0));
                // sweep 3: write
                uint32_t pos = 0;
                for (uint32_t it = 0; it < nit; ++it) {
                    bool keep = false;
                    uint32_t id = 0; double x = 0, y = 0, z = 0;
                    const bool in = it * 32 + lane < n_p;
                    if (it < 32) {
                        keep = (flags >> it) & 1u;
                        if (keep) fetch(it, id, x, y, z);
                    } else if (in) {
                        fetch(it, id, x, y, z);
                        keep = vox_keep(__double2float_rn(x - ccx), __double2float_rn(y - ccy), __double2float_rn(z - ccz), pv, 2.f * e, tol_abs);
                    }
                    const unsigned bm = __ballot_sync(FULL, keep);
                    if (keep) {
                        const unsigned long long at = off + pos + (unsigned)__popc(bm & lt);
                        if (FINAL) a.c_ent[at] = make_float4(__double2float_rn(x - ccx), __double2float_rn(y - ccy), __double2float_rn(z - ccz), __int_as_float((int)id));
                        else       a.c_ids[at] = (int32_t)id;
                    }
                    pos += (uint32_t)__popc(bm);
                }
                if (lane == 0) a.c_hdr[ci] = make_uint2((unsigned int)off, cnt);
                ++st_listed; st_entries += cnt; st_max = cnt > st_max ? cnt : st_max;
            }
        }
    }
    if (lane == 0) {
        if (st_listed) atomicAdd(&a.stats[0], st_listed);
        if (st_entries) atomicAdd(&a.stats[1], st_entries);
        if (st_long) atomicAdd(&a.stats[2], st_long);
        if (st_room) atomicAdd(&a.stats[3], st_room);
        if (st_max) atomicMax(&a.stats[4], st_max);
        if (st_far) atomicAdd(&a.stats[5], st_far);
    }
}

// ---- query --------------------------------------------------------------------------------------------------------------
// One thread per query.  counters (profiling): [3] queries answered here, [6] entries read, [7] points gathered for the
// FP64 decision; queries without a list are appended to the work list of the pyramid walk.  The queries of a hypothesis the
// tolerance stop has stopped (a.stop_iter[h] >= 0) are neither answered nor handed to the walk: they carry their previous
// correspondence forward (a stop happens at an update, so every pass after one has a.prev), which keeps every
// correspondence buffer a valid warm start for the final pass; their d2 stays stale (nothing reads it before the final pass).
__global__ void __launch_bounds__(256) k_nn_vox(const __grid_constant__ GridArgs a) {
    const VoxView& V = a.vox;
    const int lane = threadIdx.x & 31;
    const int64_t gq = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool defer = false;
    unsigned long long n_read = 0, n_gather = 0, n_done = 0;
    const unsigned h = (unsigned)gq / (unsigned)a.ns, i = (unsigned)gq - h * (unsigned)a.ns;
    if (gq < a.nq && a.stop_iter && a.prev && a.stop_iter[h] >= 0) {
        a.idx[gq] = a.prev[gq];
    } else if (gq < a.nq) {
        double qx, qy, qz;
        quick_tf(a.T + (size_t)h * 16, a.sx[i], a.sy[i], a.sz[i], qx, qy, qz);
        uint2 hd;
        float x, y, z;
        if (vox_lookup(V, qx, qy, qz, hd, x, y, z)) {
            int32_t bidx; double best; unsigned ng;
            vox_scan<4, false>(V, a.g.pts, hd, x, y, z, qx, qy, qz, bidx, best, ng);
            a.idx[gq] = bidx;
            if (a.d2) a.d2[gq] = best;
            n_read = hd.y; n_gather = ng; n_done = 1;
        } else {
            defer = true;
        }
    }
    worklist_append(a, defer, gq, lane);
    if (a.counters) flush_counters(a.counters, n_read, n_gather, n_done, 6, 7, 3);
}

void nn_vox_launch(const pcreg_model* m, const GridArgs& a, cudaStream_t st) {
    (void)m;
    const int64_t blocks = (a.nq + 255) / 256;
    k_nn_vox<<<(unsigned)blocks, 256, 0, st>>>(a);
    PCREG_LAUNCHED();
}

// ---- build (host driver) ---------------------------------------------------------------------------------------------------
static double env_double(const char* name, double dflt) { const char* e = getenv(name); return e ? atof(e) : dflt; }

void vox_build(pcreg_model* m, const pcreg_model_opts& o, cudaStream_t st) {
    m->has_vox = false;
    if (!m->has_grid || o.voxel_map < 0) return;
    if (const char* e = getenv("PCREG_VOX")) { if (e[0] == '0' && o.voxel_map != 1) return; }
    Context& c = ctx();
    const int64_t n = m->n;
    double ext[3], maxext = 0.0;
    for (int a = 0; a < 3; ++a) { ext[a] = m->bbox_hi[a] - m->bbox_lo[a]; maxext = std::max(maxext, ext[a]); }
    if (!(maxext > 0.0)) return;                                      // a single location: nothing to index
    // point spacing: the occupied cells of the grid approximate the sampled surface (or volume) at cell resolution
    const double cell = m->grid.cell;
    const double occ = (double)std::max<int64_t>(m->g_occupied, 1);
    const double delta = sqrt(occ * cell * cell / (double)n);
    const double scale = o.voxel_scale > 0.0 ? o.voxel_scale : env_double("PCREG_VOX_SCALE", 1.25);
    double s = scale * delta;
    if (!(s > 0.0) || !std::isfinite(s)) return;
    double margin = o.voxel_margin > 0.0 ? o.voxel_margin : (o.voxel_margin < 0.0 ? 0.0 : env_double("PCREG_VOX_MARGIN", 0.04) * maxext);
    size_t budget_bytes = c.total_mem / 8;                            // entries of the finest level (band-limited maps: 1/5 of the memory)
    // voxels of a full-resolution map: 2^28 (a 2 M-point model: 240 M voxels of 1.25 spacings, 442 M entries, 11.7 GB, built in
    // 0.85 s -- against the 2.5-spacing map that a cap of 2^27 forces on it, the C4 polish takes 264 instead of 380 ms per
    // 16 384 poses); ~42 B per voxel measured (8 B header + 2.1 entries), 64 budgeted
    const double max_vox = (double)(o.max_voxels > 0 ? o.max_voxels
                                    : std::min<int64_t>((int64_t)env_double("PCREG_VOX_MAX", 268435456.0), (int64_t)(budget_bytes / 64)));
    int32_t dims[3];
    auto size_for = [&](double edge) {
        double tot = 1.0;
        for (int a = 0; a < 3; ++a) { const double d = ceil((ext[a] + 2.0 * margin) / edge); dims[a] = (int32_t)std::max(1.0, std::min(d, 2.0e9)); tot *= std::max(1.0, d); }
        return tot;
    };
    double nv = size_for(s);
    double band = 0.0;                                                // 0: every voxel of the padded box gets a list
    int base_cap = (int)std::max(8.0, env_double("PCREG_VOX_CAP", (double)VOX_BASE_CAP));
    if (nv > max_vox && o.voxel_map != 1 && o.max_voxels <= 0) {
        // Dense model (C5: 16 M points, 0.04 mm spacing): a map over the whole box does not fit.  ICP queries live near the
        // surface, so only the voxels within `band` of the model get lists (about max_vox of them); the header array stays
        // dense (8 B per voxel), queries beyond the band are walked.  Voxels of 2.5 spacings: lists of ~30 entries.
        // Padding of 8 % instead of 4: the source points that wide starts throw outside the box are walked one by one on a model
        // this dense (C5: 0.08 % of the queries were 12 % of the step; 334 -> 311 ms for 2 GB more header array).
        const double margin_full = margin;
        if (o.voxel_margin == 0.0 && !getenv("PCREG_VOX_MARGIN")) margin = 0.08 * maxext;
        const double s_band = std::max(s, env_double("PCREG_VOX_DENSE_SCALE", 2.5) * delta);
        const double hdr_budget = (double)c.total_mem / 16.0 / 8.0;            // voxels whose headers fit in 1/16 of the memory
        double sb = s_band;
        double nvb = size_for(sb);
        while (nvb > hdr_budget && sb < 6.0 * delta) { sb *= 1.05; nvb = size_for(sb); }
        const double area = occ * cell * cell;
        const double max_near = env_double("PCREG_VOX_NEAR", 536870912.0);       // listed voxels (2^29: C5 -> band ~12 mm)
        const double b = max_near * sb * sb * sb / (2.0 * area);                // slab of +- band around the surface holds ~max_near voxels
        if (nvb <= hdr_budget && b >= 4.0 * sb) {
            s = sb; nv = nvb; band = std::min(b, maxext);
            base_cap = std::max(base_cap, 192);
            budget_bytes = c.total_mem / 5;
        } else {
            margin = margin_full;
            nv = size_for(s);
        }
    }
    if (band == 0.0 && env_double("PCREG_VOX_BAND", 0.0) > 0.0) band = env_double("PCREG_VOX_BAND", 0.0);      // tests: force a band
    else if (band == 0.0) {
        while (nv > max_vox) { s *= std::max(1.02, cbrt(nv / max_vox)); nv = size_for(s); }
        // too dense for the budget: the lists would hold hundreds of points -- leave such models to the grid kernels
        if (s > 3.5 * delta && o.voxel_map != 1) return;
    }
    std::vector<std::array<int32_t, 3>> ld;
    ld.push_back({dims[0], dims[1], dims[2]});
    // the top level filters ALL points per voxel (cost: voxels x points): fewer, larger top voxels for large models
    const int top_dim = n > 2000000 ? VOX_TOP_DIM / 2 : VOX_TOP_DIM;
    while (std::max({ld.back()[0], ld.back()[1], ld.back()[2]}) > top_dim)
        ld.push_back({(ld.back()[0] + 1) / 2, (ld.back()[1] + 1) / 2, (ld.back()[2] + 1) / 2});
    const int top = (int)ld.size() - 1;
    if (top == 0) {                                                   // tiny map: give the top-level kernel a level of its own
        ld.push_back({(dims[0] + 1) / 2, (dims[1] + 1) / 2, (dims[2] + 1) / 2});
    }
    const int L = (int)ld.size();

    cudaEvent_t e0 = pooled_event(0), e1 = pooled_event(1);
    PCREG_CUDA(cudaEventRecord(e0, st));
    DevBuf<unsigned long long> ctrl(8);                               // [0] pool cursor, [1] work cursor, [2..7] stats
    auto tiles_of = [](const std::array<int32_t, 3>& d, int32_t* t) { for (int a = 0; a < 3; ++a) t[a] = (d[a] + 3) / 4; };
    auto slots_of = [&](const std::array<int32_t, 3>& d) { int32_t t[3]; tiles_of(d, t); return (size_t)t[0] * t[1] * t[2] * 64; };
    auto maxlen_of = [&](int l) { double v = (double)base_cap * pow(4.0, (double)l); return (uint32_t)std::min<double>(std::min<double>(v, (double)n), 4.0e9); };

    static const bool dbg = [] { const char* e = getenv("PCREG_DEBUG_HOST"); return e && e[0] == '1'; }();
    auto dbg_now = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return 1e3 * ts.tv_sec + 1e-6 * ts.tv_nsec; };
    double t_level = dbg ? (cudaStreamSynchronize(st), dbg_now()) : 0.0;
    DevBuf<uint2> p_hdr, c_hdr;
    DevBuf<int32_t> p_ids, c_ids;
    DevBuf<float4> ent;
    unsigned long long used = 0, listed_parent = 0, h_ctrl[8];
    const double origin[3] = {m->bbox_lo[0] - margin, m->bbox_lo[1] - margin, m->bbox_lo[2] - margin};
    for (int l = L - 1; l >= 0; --l) {
        const bool is_top = (l == L - 1), fin = (l == 0);
        VoxLevelArgs a{};
        a.pts = m->g_pts.p; a.npts = (uint32_t)n;
        a.cs = s * (double)(1u << l);
        for (int k = 0; k < 3; ++k) { a.cd[k] = ld[l][k]; a.origin[k] = origin[k]; }
        tiles_of(ld[l], a.ct);
        c_hdr.alloc(slots_of(ld[l]));
        PCREG_CUDA(cudaMemsetAsync(c_hdr.p, 0, c_hdr.bytes(), st));
        PCREG_CUDA(cudaMemsetAsync(ctrl.p, 0, ctrl.bytes(), st));
        unsigned long long cap;
        const unsigned long long nvox_l = (unsigned long long)ld[l][0] * ld[l][1] * ld[l][2];
        if (is_top) cap = std::min<unsigned long long>(nvox_l * std::min<unsigned long long>((unsigned long long)n, maxlen_of(l)),
                                                       std::max<unsigned long long>(64ull * (unsigned long long)n, 1ull << 26));
        else        cap = 8ull * used + 65536ull * (unsigned long long)VOX_CHUNK;     // a child's list is a subset of its parent's: 8 x is the worst case (+ chunk tails)
        if (fin && !is_top) cap += 8ull * listed_parent;                                  // + the pad entry of odd lists
        if (fin) cap = std::min<unsigned long long>(cap, (unsigned long long)(budget_bytes / sizeof(float4)));
        cap = std::min<unsigned long long>(std::max<unsigned long long>(cap, 1024ull), 0xfffffff0ull);
        if (fin) ent.alloc((size_t)cap); else c_ids.alloc((size_t)cap);
        a.c_hdr = c_hdr.p; a.c_ids = fin ? nullptr : c_ids.p; a.c_ent = fin ? ent.p : nullptr;
        a.pool_cursor = ctrl.p; a.pool_cap = cap; a.work_cursor = ctrl.p + 1; a.stats = ctrl.p + 2;
        a.maxlen = maxlen_of(l);
        a.band = (float)band;
        if (!is_top) {
            a.p_hdr = p_hdr.p; a.p_ids = p_ids.p;
            for (int k = 0; k < 3; ++k) a.pd[k] = ld[l + 1][k];
            tiles_of(ld[l + 1], a.pt);
        }
        if (is_top) {
            PCREG_REQUIRE(!fin, "vox_build: the top level cannot be the finest one");
            k_vox_block<false><<<(unsigned)slots_of(ld[l]), 256, 0, st>>>(a);
        } else if (!fin && listed_parent > 0 && used / listed_parent > 768 && slots_of(ld[l]) < ((size_t)1 << 22)) {
            // long parent lists (coarse levels): a block per child voxel
            k_vox_block<true><<<(unsigned)slots_of(ld[l]), 256, 0, st>>>(a);
        } else {
            const int blocks = (int)std::min<size_t>((slots_of(ld[l + 1]) + 255) / 256 + 1, (size_t)c.sm_count * 8);
            if (fin) k_vox_refine<true><<<blocks, 256, 0, st>>>(a);
            else     k_vox_refine<false><<<blocks, 256, 0, st>>>(a);
        }
        PCREG_LAUNCHED();
        PCREG_CUDA(cudaMemcpyAsync(h_ctrl, ctrl.p, sizeof h_ctrl, cudaMemcpyDeviceToHost, st));
        PCREG_CUDA(cudaStreamSynchronize(st));
        used = std::min<unsigned long long>(h_ctrl[0], cap);
        listed_parent = h_ctrl[2];
        if (dbg) {
            const double t = dbg_now();
            fprintf(stderr, "[pcreg vox] level %d (%d x %d x %d, edge %.4g): %.1f ms, %llu listed, %llu entries, %llu too long, %llu no room, %llu far, longest %llu\n",
                    l, ld[l][0], ld[l][1], ld[l][2], a.cs, t - t_level, h_ctrl[2], h_ctrl[3], h_ctrl[4], h_ctrl[5], h_ctrl[7], h_ctrl[6]);
            t_level = t;
        }
        if (fin) {
            m->v_listed = (int64_t)h_ctrl[2]; m->v_entries = (int64_t)h_ctrl[3];
            m->v_too_long = (int64_t)h_ctrl[4]; m->v_no_room = (int64_t)h_ctrl[5]; m->v_max_len = (int64_t)h_ctrl[6];
            m->v_far = (int64_t)h_ctrl[7]; m->v_band = band;
            m->v_voxels = (int64_t)nvox_l;
        }
        p_hdr = std::move(c_hdr);
        p_ids = std::move(c_ids);
    }
    // keep what is used: the pool was sized for the worst case
    if ((size_t)used + 1024 < ent.n / 10 * 7) {
        DevBuf<float4> exact((size_t)used + 16);
        PCREG_CUDA(cudaMemcpyAsync(exact.p, ent.p, (size_t)used * sizeof(float4), cudaMemcpyDeviceToDevice, st));
        PCREG_CUDA(cudaStreamSynchronize(st));
        ent = std::move(exact);
    }
    PCREG_CUDA(cudaEventRecord(e1, st));
    PCREG_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    PCREG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    m->v_build_ms = (double)ms;
    m->v_hdr = std::move(p_hdr);
    m->v_ent = std::move(ent);
    VoxView& V = m->vox;
    V.ent = m->v_ent.p; V.hdr = m->v_hdr.p;
    for (int k = 0; k < 3; ++k) { V.dims[k] = ld[0][k]; V.origin[k] = origin[k]; }
    tiles_of(ld[0], V.tiles);
    V.s = s; V.inv_s = 1.0 / s;
    V.band_abs = (float)(0.8e-6 * s * s);
    m->has_vox = true;
}

}  // namespace pcreg

using namespace pcreg;

extern "C" int pcreg_model_voxel_info(const pcreg_model* m, int32_t dims[3], double* voxel_size, int64_t stats[10]) {
    if (!m) { set_error("pcreg_model_voxel_info: null model"); return PCREG_ERR_ARG; }
    if (!m->has_vox) {
        if (dims) dims[0] = dims[1] = dims[2] = 0;
        if (voxel_size) *voxel_size = 0.0;
        if (stats) for (int k = 0; k < 10; ++k) stats[k] = 0;
        return PCREG_OK;
    }
    if (dims) for (int k = 0; k < 3; ++k) dims[k] = m->vox.dims[k];
    if (voxel_size) *voxel_size = m->vox.s;
    if (stats) {
        stats[0] = m->v_voxels; stats[1] = m->v_listed; stats[2] = m->v_entries; stats[3] = m->v_too_long;
        stats[4] = m->v_no_room; stats[5] = m->v_max_len; stats[6] = (int64_t)(m->v_build_ms * 1000.0);
        stats[7] = (int64_t)(m->v_ent.bytes() + m->v_hdr.bytes());
        stats[8] = m->v_far; stats[9] = (int64_t)(m->v_band * 1.0e6);
    }
    return PCREG_OK;
}
