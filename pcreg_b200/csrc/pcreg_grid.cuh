// pcreg_grid.cuh -- kernel argument block and warp helpers shared by the grid NN kernels (nn_grid.cu) and the
// voxel-map list scan (nn_vox.cu).
#pragma once
#include <math.h>
#include <float.h>
#include "pcreg_internal.h"
#include "pcreg_dev.cuh"

namespace pcreg {

struct GridArgs {
    GridView g;
    const ModelPointD* md;
    const double* sx; const double* sy; const double* sz; int64_t ns;
    const double* T; int64_t nq;
    const int32_t* prev;
    int32_t* idx; double* d2;
    VoxView vox;                    // Voronoi voxel map of the model (nn_vox.cu; vox.hdr == nullptr: none)
    CandView cl;                    // candidate lists of the chunk (cl.cnt == nullptr: disabled)
    const double* skip_thr;         // [nhyp] or null: list kernel skips queries whose previous residual exceeds it (lazy trimming)
    const int32_t* stop_iter;       // [nhyp] or null: the voxel-map kernel skips the queries of hypotheses with stop_iter >= 0
    const int32_t* in_list;         // direct kernel: the queries to process (nullptr: all nq)
    const unsigned int* in_count;   //                and how many
    int32_t* worklist;              // [nq] query ids handed to the next kernel (list -> direct -> walk)
    unsigned int* work_count;       // number of entries in worklist
    unsigned long long* cursor;     // direct kernel: next unassigned position of its input (zeroed before the launch)
    int32_t* overflow;              // warp walk: queries it hands on to the per-lane walk (frontier too large, no bound)
    unsigned int* overflow_count;
    int ww_cap;                     // warp walk: frontier entries it may use (<= WW_CAP; the tests force overflows with a small one)
    int fetch_batch, chunk;         // (tuning)
    int chain;                      // first-pass walk: consecutive queries per thread
    int row_span;                   // direct kernel: widest (y,z) cell span it row-scans itself
    unsigned long long* counters;   // profiling only (may be null): [0] points / [1] rows visited by the row scan, [2] pyramid
                                    // nodes popped, [3] queries answered from their list, [4] queries walked, [5] queries
                                    // row-scanned, [6] list entries read, [7] list points gathered, [8] points / [9] leaf cells
                                    // visited by the walk
};

// Arguments of the fused per-hypothesis ICP kernel (icp_fused.cu): everything one block needs for all passes.
struct FusedArgs {
    GridArgs g;                 // g.g (grid + points), g.md, g.vox: what the NN step reads (the other members are unused)
    const double* sx; const double* sy; const double* sz; const double* w_src; int32_t ns;
    double pivot[3];
    double* T;                  // [nhyp][16] row-major poses, in / out
    int32_t* frozen;            // [nhyp] in / out
    double* rmse; int32_t* n_used;          // [nhyp] out (final pass)
    double* rmse_hist; int hist_stride;     // optional [nhyp][iters + 1]
    int32_t* idx_out;           // optional [nhyp][ns] final correspondences, ORIGINAL source order
    const int32_t* perm;        // [ns] original index of (sorted) source position r, or null
    const int32_t* tie_order;   // [ns] (sorted) position of original index (stable tie rule of the trim), or null
    int mode; double k_frac, R_w, thDist2; int reflection_fix; int iters;
    unsigned long long* counters;           // profiling (may be null): [4] queries walked, [6] list entries read, [7] points gathered
    IcpStopRule stop;                       // tolerance stop (the k_icp_fused<*, true> instantiations only)
    int32_t* n_iter; int32_t* converged;    // [nhyp] optional outputs of the tolerance stop
    const ModelPointD* nrm;                 // model normals (original order): the point-to-plane metric; null: point-to-point
    // plane-to-plane metric (null: the other two): unit source normals in the order of sx / sy / sz, and the covariance epsilon
    const double* snx; const double* sny; const double* snz; double gicp_eps;
    // pose extrapolation (the k_icp_fused<*, 2, 0> instantiations only): the rule, the source centroid of each window ([nwin][3]; one
    // window without WIN) and the optional [nhyp] count of extrapolated updates
    IcpExtrapRule ex; const double* ex_cen; int32_t* n_extrap;
    IcpCovOut cov;                          // the covariance pass (the k_icp_fused<*, 0, 3> instantiations; cov.cov null otherwise)
};
// Windowed calls (pcreg_icp_batch_windows; the k_icp_fused<*, *, *, true> instantiations): the source arrays, w_src, the source
// normals, perm and tie_order are the concatenation of nwin windows (column stride of sx / sy / sz: the total row count), and
// ns is the largest window's row count.  Window w owns rows win_src[w] .. win_src[w + 1] - 1 and hypotheses win_hyp[w] ..
// win_hyp[w + 1] - 1; its perm / tie_order entries are relative to its first row, and its [H_w][ns_w] block of idx_out starts at
// win_idx[w].
struct FusedWinArgs : FusedArgs {
    const int64_t* win_src; const int64_t* win_hyp; const int64_t* win_idx;   // device, [nwin + 1], [nwin + 1], [nwin]
    int32_t nwin;
};
size_t icp_fused_smem(int64_t ns, int mode);
// stop: 0 no tolerance stop, 1 the stop, 2 the stop with pose extrapolation (point-to-point only)
bool icp_fused_eligible(const pcreg_model* m, int64_t ns, int64_t nhyp, const pcreg_icp_opts& o, int stop, int metric);
void icp_fused_launch(FusedArgs& a, int64_t nhyp, int stop, cudaStream_t st);
// windowed calls: the instantiation they launch fits the largest window (ns_max) in shared memory on the model's voxel map
bool icp_fused_windows_fit(const pcreg_model* m, int64_t ns_max, const pcreg_icp_opts& o, int stop, int metric);
void icp_fused_windows_launch(const FusedWinArgs& a, int64_t nhyp, int stop, cudaStream_t st);

__device__ __forceinline__ void flush_counters(unsigned long long* counters, unsigned long long n_pts,
                                               unsigned long long n_cells, unsigned long long n_nodes, int i_pts = 0, int i_cells = 1,
                                               int i_nodes = 2) {
    if (!counters) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_pts += __shfl_xor_sync(0xffffffffu, n_pts, o);
        n_cells += __shfl_xor_sync(0xffffffffu, n_cells, o);
        n_nodes += __shfl_xor_sync(0xffffffffu, n_nodes, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (n_pts) atomicAdd(&counters[i_pts], n_pts);
        if (n_cells) atomicAdd(&counters[i_cells], n_cells);
        if (n_nodes) atomicAdd(&counters[i_nodes], n_nodes);
    }
}

// warp-aggregated append of query ids to the next kernel's work list
__device__ __forceinline__ void worklist_append(const GridArgs& a, bool defer, int64_t gq, int lane) {
    const unsigned dm = __ballot_sync(0xffffffffu, defer);
    if (dm) {
        const int leader = __ffs(dm) - 1;
        unsigned base = 0;
        if (lane == leader) base = atomicAdd(a.work_count, (unsigned)__popc(dm));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (defer) a.worklist[base + __popc(dm & ((1u << lane) - 1u))] = (int32_t)gq;
    }
}

constexpr int GRID_STACK = 80;
// depth-first walk: starts from the root (1 entry, GRID_MAX_LEVELS - 1 levels to descend) or from <= 8 nodes below it;
// every expanded node replaces itself by at most 8 children (net +7 per level)
static_assert(1 + 7 * (GRID_MAX_LEVELS - 1) <= GRID_STACK && 8 + 7 * (GRID_MAX_LEVELS - 2) <= GRID_STACK,
              "k_nn_grid_walk: explicit stack too small for GRID_MAX_LEVELS");
constexpr float GRID_SLOP_ABS = 1.3e-4f;   // cell units: FP32 rounding of the query (<= 1024 cells) + of the difference
constexpr float GRID_SLOP_REL = 2.5e-7f;

// stack entry: [63:34] lower bound (positive float, lowest mantissa bit dropped = rounded down),
//              [33:30] level, [29:20] z, [19:10] y, [9:0] x
__device__ __forceinline__ unsigned long long pack_entry(float lb, int level, int x, int y, int z) {
    return ((unsigned long long)(__float_as_uint(lb) >> 1) << 34) | ((unsigned long long)(unsigned)level << 30) |
           ((unsigned long long)(unsigned)z << 20) | ((unsigned long long)(unsigned)y << 10) | (unsigned long long)(unsigned)x;
}

// conservative (never too large) distance along one axis, in cell units, from q to the slab [lo, lo+edge]
__device__ __forceinline__ float axis_lb(float q, float lo, float edge) {
    const float d = fmaxf(lo - q, q - (lo + edge));
    return fmaxf(fmaf(-GRID_SLOP_REL, fabsf(d), d) - GRID_SLOP_ABS, 0.f);
}
// conservative squared distance, in cell units, from the query to the box [x, x+1] * edge (corners exact in FP32)
__device__ __forceinline__ float box_lb(float qx, float qy, float qz, int x, int y, int z, float edge) {
    const float dx = axis_lb(qx, (float)x * edge, edge), dy = axis_lb(qy, (float)y * edge, edge), dz = axis_lb(qz, (float)z * edge, edge);
    return (dx * dx + dy * dy + dz * dz) * (1.f - 6e-7f);
}
// guaranteed upper bound of best (squared distance) in squared cell units, as a float.  Beyond the float range it is
// +infinity, not FLT_MAX: the box bounds of a query some 1e19 cells away overflow to +infinity as well, and a finite bound
// would prune every box -- the query would end without an answer.  With +infinity nothing is pruned (every box is visited).
__device__ __forceinline__ float best_ub_cells(double best, double inv_cell2) {
    const double b = best * inv_cell2;
    return (b < 3.0e38) ? __double2float_ru(b) * (1.f + 6e-7f) : INFINITY;
}
// same for the ball of radius (sqrt(best) + gap): everything inside it gets visited
__device__ __forceinline__ float best_ub_cells_gap(double best, double inv_cell, float gap_cells) {
    const double r = sqrt(best) * inv_cell + (double)gap_cells;
    const double b = r * r;
    return (b < 3.0e38) ? __double2float_ru(b) * (1.f + 6e-7f) : INFINITY;
}

struct Query {
    double qx, qy, qz;      // FP64 query (oracle order)
    float fx, fy, fz;       // in cell units, FP32 (pruning only)
    double best; int32_t bidx; float bestc;
    int ilx, ihx, ily, ihy, ilz, ihz;   // level-0 cell span of the ball's bounding cube (valid when has_span)
    bool has_span;
};

// Q.qx/qy/qz set by the caller: cell-unit copy, warm-start bound, cell span of the ball
__device__ __forceinline__ void setup_query_at(const GridView& G, const ModelPointD* __restrict__ md, Query& Q, float gap_cells, int32_t warm);
__device__ __forceinline__ void setup_query(const GridArgs& a, int64_t gq, Query& Q, float gap_cells, int32_t warm) {
    const unsigned h = (unsigned)gq / (unsigned)a.ns, i = (unsigned)gq - h * (unsigned)a.ns;      // nq < 2^31 (launcher)
    quick_tf(a.T + (size_t)h * 16, a.sx[i], a.sy[i], a.sz[i], Q.qx, Q.qy, Q.qz);
    setup_query_at(a.g, a.md, Q, gap_cells, warm);
}
__device__ __forceinline__ void setup_query_at(const GridView& G, const ModelPointD* __restrict__ md, Query& Q, float gap_cells, int32_t warm) {
    Q.fx = __double2float_rn((Q.qx - G.origin[0]) * G.inv_cell);
    Q.fy = __double2float_rn((Q.qy - G.origin[1]) * G.inv_cell);
    Q.fz = __double2float_rn((Q.qz - G.origin[2]) * G.inv_cell);
    Q.best = INFINITY;
    Q.bidx = -1;
    if (warm >= 0) {                 // any model point bounds the answer: the caller's previous correspondence, or a neighbour's
        const ModelPointD mp = md[warm];
        Q.best = dist2_exact(mp.x, mp.y, mp.z, Q.qx, Q.qy, Q.qz);
        Q.bidx = warm;
    }
    Q.bestc = (gap_cells > 0.f) ? best_ub_cells_gap(Q.best, G.inv_cell, gap_cells) : best_ub_cells(Q.best, G.inv_cell * G.inv_cell);
    Q.has_span = false;
    if (Q.bidx >= 0 && Q.bestc < 1.0e12f) {
        // ball radius in cells (upper bound) -> integer cell span
        const float rc = __fsqrt_ru(Q.bestc) + 2.0f * GRID_SLOP_ABS + GRID_SLOP_REL * (fabsf(Q.fx) + fabsf(Q.fy) + fabsf(Q.fz));
        const float big = 1.0e6f;
        Q.ilx = (int)floorf(fmaxf(fminf(Q.fx - rc, big), -big)); Q.ihx = (int)floorf(fmaxf(fminf(Q.fx + rc, big), -big));
        Q.ily = (int)floorf(fmaxf(fminf(Q.fy - rc, big), -big)); Q.ihy = (int)floorf(fmaxf(fminf(Q.fy + rc, big), -big));
        Q.ilz = (int)floorf(fmaxf(fminf(Q.fz - rc, big), -big)); Q.ihz = (int)floorf(fmaxf(fminf(Q.fz + rc, big), -big));
        Q.has_span = true;
    }
}

__device__ __forceinline__ void scan_points(const GridView& G, int32_t s0, int32_t s1, Query& Q, double inv_cell2) {
    bool improved = false;
    for (int32_t p = s0; p < s1; ++p) {
        const GridPoint gp = G.pts[p];
        const double d = dist2_exact(gp.x, gp.y, gp.z, Q.qx, Q.qy, Q.qz);
        if (d < Q.best || (d == Q.best && gp.orig < Q.bidx)) { Q.best = d; Q.bidx = gp.orig; improved = true; }
    }
    if (improved) Q.bestc = best_ub_cells(Q.best, inv_cell2);
}

// (sqrt(best) + skin)^2, never too small: the points with d2 <= this value enter the candidate list
__device__ __forceinline__ double list_thr2(double best, double skin) {
    const double t = sqrt(best) + skin;
    return t * t * (1.0 + 1e-12);
}
// append grid position p to the list under construction: the first cl.cap entries live in the query's own
// row, longer lists (wide balls) continue in an extension slot taken from a shared pool on first need
// entry = position << 8 | level, level = where sqrt(d2) falls in [lo, lo + 2 skin] on a 256-step scale, rounded DOWN by
// a whole step (the scan skips an entry only if even the lower edge of its level is out of reach)
__device__ __forceinline__ void list_append(const CandView& cl, int64_t gq, int& lc, int& ext_slot, int32_t pos, double d, float lo) {
    const float sd = __fsqrt_rd(__double2float_rd(d));
    const int level = min(max((int)floorf((sd - lo) * cl.inv_level) - 1, 0), 255);
    const int32_t p = (int32_t)(((unsigned)pos << 8) | (unsigned)level);
    if (lc < cl.cap) {
        cl.list[gq * cl.cap + lc] = p;
    } else {
        if (ext_slot == -1) {
            const unsigned s = atomicAdd(cl.ext_count, 1u);
            ext_slot = s < (unsigned)cl.ext_slots ? (int)s : -2;          // -2: pool exhausted
        }
        const int k = lc - cl.cap;
        if (ext_slot >= 0 && k < cl.ext_cap) cl.ext_list[(int64_t)ext_slot * cl.ext_cap + k] = p;
    }
    ++lc;
}
// close the list of a finished search: header + count, or "no list"
__device__ __forceinline__ void list_commit(const CandView& cl, const GridView& G, int64_t gq, const Query& Q, bool bld, int lc, int ext_slot, float lo) {
    if (ext_slot >= 0) cl.ext[gq] = ext_slot;
    if (bld && lc > 0 && (lc <= cl.cap || (ext_slot >= 0 && lc <= cl.cap + cl.ext_cap))) {
        // every model point within R_list of this position is in the list
        const double rl = (sqrt(Q.best) + cl.skin) * (1.0 - 1e-7);
        cl.hdr[gq] = make_float4(__double2float_rn(Q.qx - G.origin[0]), __double2float_rn(Q.qy - G.origin[1]),
                                 __double2float_rn(Q.qz - G.origin[2]), __double2float_rd(rl));
        cl.cnt[gq] = make_int2(lc, __float_as_int(lo));
    } else {
        cl.cnt[gq] = make_int2(-1, 0);
    }
}

// Branch-and-bound walk of the occupancy pyramid for ONE query whose Query record is set up (position, warm-start bound,
// cell span): nearest octant first, explicit stack, every visited point evaluated exactly.  BUILD: also records the
// candidate list of the query (nn_grid.cu).  Used by k_nn_grid_walk and, for the few queries the Voronoi voxel map
// cannot answer, by the fused ICP kernel (icp_fused.cu).
template <bool BUILD>
__device__ __forceinline__ void walk_search(const GridArgs& a, int64_t gq, Query& Q, bool bld, int& lc, int& ext_slot, double& thr2, float lo,
                                            unsigned long long& n_pts, unsigned long long& n_cells, unsigned long long& n_nodes) {
    const GridView& G = a.g;
    const double inv_cell2 = G.inv_cell * G.inv_cell;
    const float fx = Q.fx, fy = Q.fy, fz = Q.fz;
    unsigned long long stack[GRID_STACK];
    int sp = 0;
    const int top = G.nlevels - 1;
    bool from_root = true;
    if (Q.has_span) {
        // lowest level whose <= 2 x 2 x 2 nodes cover the ball's bounding cube
        int l = 0;
        while (l < top && (((Q.ihx >> l) - (Q.ilx >> l)) > 1 || ((Q.ihy >> l) - (Q.ily >> l)) > 1 || ((Q.ihz >> l) - (Q.ilz >> l)) > 1)) ++l;
        if (((Q.ihx >> l) - (Q.ilx >> l)) <= 1 && ((Q.ihy >> l) - (Q.ily >> l)) <= 1 && ((Q.ihz >> l) - (Q.ilz >> l)) <= 1) {
            from_root = false;
            const float edge = (float)(1 << l);
            const int dxl = G.dims[l][0], dyl = G.dims[l][1], dzl = G.dims[l][2];
            for (int z = Q.ilz >> l; z <= (Q.ihz >> l); ++z) {
                if (z < 0 || z >= dzl) continue;
                for (int y = Q.ily >> l; y <= (Q.ihy >> l); ++y) {
                    if (y < 0 || y >= dyl) continue;
                    for (int x = Q.ilx >> l; x <= (Q.ihx >> l); ++x) {
                        if (x < 0 || x >= dxl) continue;
                        if (l > 0 && G.mask[l][((int64_t)z * dyl + y) * dxl + x] == 0) continue;
                        const float lb = box_lb(fx, fy, fz, x, y, z, edge);
                        if (lb <= Q.bestc) stack[sp++] = pack_entry(lb, l, x, y, z);
                    }
                }
            }
        }
    }
    if (from_root) stack[sp++] = pack_entry(0.f, top, 0, 0, 0);

    while (sp > 0) {
        const unsigned long long e = stack[--sp];
        const float lbf = __uint_as_float((unsigned)(e >> 34) << 1);
        if (lbf > Q.bestc) continue;
        const unsigned lo32 = (unsigned)e;
        const int level = (int)((e >> 30) & 0xF);
        const int ix = (int)(lo32 & 1023u), iy = (int)((lo32 >> 10) & 1023u), iz = (int)((lo32 >> 20) & 1023u);
        ++n_nodes;
        if (level == 0) {
            // exact FP64 scan of the leaf's points
            const int64_t c = ((int64_t)iz * G.dims[0][1] + iy) * G.dims[0][0] + ix;
            const int32_t s0 = G.cell_start[c], s1 = G.cell_start[c + 1];
            ++n_cells;
            n_pts += (unsigned long long)(s1 - s0);
            bool improved = false;
            for (int32_t p = s0; p < s1; ++p) {
                const GridPoint gp = G.pts[p];
                const double d = dist2_exact(gp.x, gp.y, gp.z, Q.qx, Q.qy, Q.qz);
                if (d < Q.best || (d == Q.best && gp.orig < Q.bidx)) {
                    Q.best = d; Q.bidx = gp.orig; improved = true;
                    if (BUILD && bld) thr2 = list_thr2(Q.best, a.cl.skin);
                }
                if (BUILD && bld && d <= thr2) list_append(a.cl, gq, lc, ext_slot, p, d, lo);
            }
            if (improved) Q.bestc = (BUILD && bld) ? best_ub_cells_gap(Q.best, G.inv_cell, a.cl.gap_cells) : best_ub_cells(Q.best, inv_cell2);
            continue;
        }
        const int64_t c = ((int64_t)iz * G.dims[level][1] + iy) * G.dims[level][0] + ix;
        unsigned m = G.mask[level][c];
        const float edge = (float)(1 << (level - 1));              // child edge in cells
        // per-axis squared bounds of the two half slabs; a child's bound is one pick per axis
        const float bx = (float)(2 * ix) * edge, by = (float)(2 * iy) * edge, bz = (float)(2 * iz) * edge;
        float ax0 = axis_lb(fx, bx, edge), ax1 = axis_lb(fx, bx + edge, edge);
        float ay0 = axis_lb(fy, by, edge), ay1 = axis_lb(fy, by + edge, edge);
        float az0 = axis_lb(fz, bz, edge), az1 = axis_lb(fz, bz + edge, edge);
        ax0 *= ax0; ax1 *= ax1; ay0 *= ay0; ay1 *= ay1; az0 *= az0; az1 *= az1;
        const unsigned oct = (fx >= bx + edge ? 1u : 0u) | (fy >= by + edge ? 2u : 0u) | (fz >= bz + edge ? 4u : 0u);
        // permute the mask so that bit t <-> child (t ^ oct); then high bits = far octants
        if (oct & 1u) m = ((m & 0xAAu) >> 1) | ((m & 0x55u) << 1);
        if (oct & 2u) m = ((m & 0xCCu) >> 2) | ((m & 0x33u) << 2);
        if (oct & 4u) m = ((m & 0xF0u) >> 4) | ((m & 0x0Fu) << 4);
        while (m) {
            const int t = 31 - __clz(m);                           // far first, so the near octant is popped first
            m &= ~(1u << t);
            const int k = t ^ (int)oct;
            const float lb = ((((k & 1) ? ax1 : ax0) + ((k & 2) ? ay1 : ay0)) + ((k & 4) ? az1 : az0)) * (1.f - 6e-7f);
            if (lb <= Q.bestc) {
                if (sp >= GRID_STACK) __trap();            // unreachable (static_assert below): never drop a node silently
                stack[sp++] = pack_entry(lb, level - 1, 2 * ix + (k & 1), 2 * iy + ((k >> 1) & 1), 2 * iz + (k >> 2));
            }
        }
    }
}

}  // namespace pcreg
