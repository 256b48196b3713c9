// icp_fused.cu -- the whole ICP of one hypothesis in ONE thread block: every pass (exact NN -> select / weight -> 17 FP64 sums
// -> Kabsch SVD -> pose compose) runs inside a single kernel launch, the hypotheses of a batch being independent
// (the reference runs them under parfor: slideMatchingWindow_v2.m:178, completeExperiment.m:265).
//
// Why.  With the Voronoi voxel map (nn_vox.cu) an NN pass costs ~0.6 ms for 20 M queries; the per-pass kernels then spend as
// much again writing correspondences / residuals / trim keys to HBM and reading them back, and a small batch (strong scaling:
// a few hundred hypotheses per GPU) is bound by the 60-odd launches.  Here the correspondences and the trim keys of a hypothesis live in
// SHARED memory (4 + 8 bytes per source point), the pose in shared memory, and nothing but the voxel lists, the source cloud
// and the gathered model points is read from global memory; there is one launch per batch and no host synchronisation.
//
// Same arithmetic as the per-pass path (pcreg_icp.cuh, pcreg_vox.cuh, pcreg_select.cuh are shared; thread t sums the
// correspondences t, t + UPD_THREADS, ... in both), so poses, RMSE history and correspondences are bit-identical to it and to the
// brute-force path (tests/test_gpu_icp.py).  Composition as in icp.cu: quickTF.m:5-7, ransac.m:49, AlignPoints_KNN.m:20-26,
// AlignPoints_weighted.m:16-18, estimateTransform.m:41-71.
// A query whose voxel has no list (or that lies outside the padded box) is walked through the occupancy pyramid by its own
// thread (walk_search, pcreg_grid.cuh), warm-started by its previous correspondence.
#include <math.h>
#include <float.h>
#include <stdlib.h>
#include <algorithm>
#include <type_traits>

#include "pcreg_internal.h"
#include "pcreg_dev.cuh"
#include "pcreg_grid.cuh"
#include "pcreg_vox.cuh"
#include "pcreg_select.cuh"
#include "pcreg_icp.cuh"

namespace pcreg {

#ifndef FUSED_SKIP_UNSELECTED
#define FUSED_SKIP_UNSELECTED 1 // trimmed mode: the sums pass does not gather the model points of unselected correspondences (C3: 35.8 -> 35.2 ms)
#endif
#ifndef FUSED_INLINE_SUMS
#define FUSED_INLINE_SUMS 0     // 1: modes without a trim accumulate the 17 sums inside the NN loop (no sums pass, no second gather).
#endif                          // Measured SLOWER (C4 polish, 16 384 poses: 592 vs 465 ms): the 34 accumulator registers push the NN loop
                                // into spills.  Kept as a switch.

// Returned by value: reference outputs would make the NN loop's winners address-taken, stored to and reloaded from local memory
// on every trip.
struct WalkHit { int32_t bidx; double best; };
__device__ __noinline__ WalkHit fused_walk(const GridArgs& a, double qx, double qy, double qz, int32_t warm) {
    Query Q;
    Q.qx = qx; Q.qy = qy; Q.qz = qz;
    setup_query_at(a.g, a.md, Q, 0.f, warm);
    int lc = 0, ext_slot = -1;
    double thr2 = 0.0;
    unsigned long long n1 = 0, n2 = 0, n3 = 0;
    walk_search<false>(a, 0, Q, false, lc, ext_slot, thr2, 0.f, n1, n2, n3);
    return WalkHit{Q.bidx, Q.best};
}
template <int METRIC>
__device__ __noinline__ bool fused_pose_update(const double (&s)[icp_nsums<METRIC>], long long n_used, const double* pivot, bool reflection_fix,
                                               double* Ts /*shared, row-major 4x4, updated in place*/) {
    double Tc[16], Tn[16];
    for (int k = 0; k < 16; ++k) Tc[k] = Ts[k];
    if (!icp_pose_update_m<METRIC>(s, n_used, pivot, reflection_fix, Tc, Tn)) return false;
    for (int k = 0; k < 16; ++k) Ts[k] = Tn[k];
    return true;
}
// Tolerance stop: the update of pass `it` (update it + 1) and the stop rule.  0: degenerate, pose left alone; 1: pose updated;
// 2: pose updated and the rule says stop.
template <int METRIC>
__device__ __noinline__ int fused_pose_update_stop(const double (&s)[icp_nsums<METRIC>], long long n_used, const double* pivot, bool reflection_fix,
                                                   const IcpStopRule& rule, int it, double* ring /*shared*/, double* Ts /*shared*/) {
    double Tc[16], Tn[16];
    for (int k = 0; k < 16; ++k) Tc[k] = Ts[k];
    if (!icp_pose_update_m<METRIC>(s, n_used, pivot, reflection_fix, Tc, Tn)) return 0;
    for (int k = 0; k < 16; ++k) Ts[k] = Tn[k];
    return icp_stop_update(rule, Tc, Tn, it + 1, ring) ? 2 : 1;
}
// The same with pose extrapolation between the Kabsch update and the stop rule (point-to-point; ex_state: shared, thread 0's).
__device__ __noinline__ int fused_pose_update_extrap(const double (&s)[KABSCH_NSUMS], long long n_used, const double* pivot, bool reflection_fix,
                                                     const IcpStopRule& rule, const IcpExtrapRule& ex, const double* cen, int it,
                                                     double* ring, double* ex_state, double* Ts) {
    double Tc[16], Tn[16];
    for (int k = 0; k < 16; ++k) Tc[k] = Ts[k];
    if (!icp_pose_update(s, n_used, pivot, reflection_fix, Tc, Tn)) return 0;
    icp_extrap_update(ex, s, pivot, cen, Tc, Tn, it + 1, ex_state);
    for (int k = 0; k < 16; ++k) Ts[k] = Tn[k];
    return icp_stop_update(rule, Tc, Tn, it + 1, ring) ? 2 : 1;
}

// The source rows of a block's hypothesis: rows r0 .. r0 + ns - 1 of the source arrays, its idx_out block at idx_base (windowed calls).
struct FusedWindow { int64_t r0, idx_base; int ns, w; };
template <bool WIN, class Args>
__device__ __forceinline__ FusedWindow fused_window(const Args& a, int64_t h) {
    if constexpr (WIN) {
        int lo = 0, hi = a.nwin - 1;            // the last window w with win_hyp[w] <= h (windows without hypotheses are skipped)
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (a.win_hyp[mid] <= h) lo = mid; else hi = mid - 1; }
        const int64_t r0 = a.win_src[lo];
        const int ns = (int)(a.win_src[lo + 1] - r0);
        return FusedWindow{r0, a.win_idx[lo] + (h - a.win_hyp[lo]) * (int64_t)ns, ns, lo};
    } else {
        return FusedWindow{0, 0, a.ns, 0};
    }
}

// KNN = the trimmed mode (its selection scratch -- 18 KB of shared memory -- exists only in that instantiation).
// STOP = the tolerance stop (pcreg_icp_batch_stop): a stop -- by the rule or by a degenerate update -- makes the block's next
// pass its final scoring pass, after which the block exits.  The STOP = 0 instantiations are the loop without it; STOP = 2 (METRIC 0
// only) adds the pose extrapolation (pcreg_icp_batch_extrap) before the stop rule.
// METRIC = 0 point-to-point; 1 point-to-plane (pcreg_icp_batch_metric): 29 sums in a pass of their own, model normals gathered
// there; 2 plane-to-plane (pcreg_icp_batch_gicp): the same, and the source normal of each correspondence rotated by the pose.
// METRIC = 3 (STOP = 0 only): the covariance pass of pcreg_icp_covariance -- iters = 0, the single pass accumulates as metric 1 with
// sum w b^2 in place of g, and the block writes a.cov (icp_cov_write) instead of updating the pose.
// WIN = a windowed call (pcreg_icp_batch_windows, FusedWinArgs): a prologue finds the block's window; from there on the block runs
// exactly as in a call on that window alone (its rows, ns, perm / tie_order entries and idx_out block).
template <bool KNN, int STOP, int METRIC, bool WIN = false>
__global__ void __launch_bounds__(UPD_THREADS, FUSED_MIN_BLOCKS) k_icp_fused(const __grid_constant__ std::conditional_t<WIN, FusedWinArgs, FusedArgs> a) {
    constexpr int NS = icp_nsums<METRIC>;
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ double Ts[16];
    __shared__ double red[(NS + 1) * 32];
    __shared__ HistSelShared hsel;
    __shared__ int s_frozen;
    __shared__ int s_stop;                                  // STOP: the next pass is the final one
    __shared__ double s_ring[2 * ICP_STOP_WINDOW_MAX + (STOP == 2 ? EXTRAP_STATE : 0)];   // STOP: thread 0's window of update
                                                                                          // motions; STOP = 2: then its extrapolation state

    const FusedWindow W = fused_window<WIN>(a, blockIdx.x);
    const int ns = W.ns;
    int32_t* __restrict__ idx_s = (int32_t*)dyn;
    unsigned long long* __restrict__ keys_s = (unsigned long long*)(dyn + (((size_t)ns * 4 + 15) / 16) * 16);    // KNN mode only
    const int64_t h = blockIdx.x;
    const int tid = threadIdx.x;
    const VoxView& V = a.g.vox;
    const GridPoint* __restrict__ pts = a.g.g.pts;
    const bool reject = a.thDist2 > 0.0;
    constexpr bool knn = KNN;
    constexpr bool two_pass = KNN || METRIC != ICP_M_POINT || !FUSED_INLINE_SUMS;      // sums in a pass of their own (needed after a trim selection)
    const double px = a.pivot[0], py = a.pivot[1], pz = a.pivot[2];
    unsigned long long c_read = 0, c_gather = 0, c_walk = 0;
    long long t_nn = 0, t_sel = 0, t_sum = 0, t_svd = 0, t_mark = 0;       // phase clocks of thread 0 (profiling only)
    const bool timing = a.counters != nullptr && tid == 0;

    if (tid < 16) Ts[tid] = a.T[h * 16 + tid];
    if (tid == 0) { s_frozen = a.frozen[h]; if (STOP) s_stop = 0; }
    if (STOP == 2 && tid < EXTRAP_STATE) s_ring[2 * ICP_STOP_WINDOW_MAX + tid] = 0.0;
    if (KNN) for (int b = tid; b < SEL_BINS; b += UPD_THREADS) hsel.hist[b] = 0;     // block_hist_finish leaves it zero after
    __syncthreads();
    // trimmed mode: the K-th residual key of the last pass (0: none yet, or nothing selected); the next pass centres its
    // histogram window on it
    unsigned long long vK = 0ull;
    bool all_eq = false;

    for (int it = 0; it <= a.iters; ++it) {
        const bool last = it == a.iters || (STOP && s_stop);     // block-uniform: s_stop was written before the last barrier
        // ---- exact nearest neighbours of the hypothesis' ns queries (two per trip: their header / entry loads overlap) ----
        double s[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) s[k] = 0.0;
        long long n_used = 0;
        // trim histogram, filled where the keys are produced: a range-free monotone bin map (exact at any scale; the window
        // only decides how many keys share the boundary bin)
        const SelBinsShift bins = SelBinsShift::around(vK);
        auto weight_of = [&](int i, int32_t j, double d) -> double {
            const bool keep = j >= 0 && (!reject || d < a.thDist2);
            double w = 0.0;
            if (knn) w = (j >= 0 && key_selected(keys_s[i], vK, all_eq)) ? 1.0 : 0.0;
            else if (a.mode == PCREG_ICP_PLAIN) w = keep ? 1.0 : 0.0;
            else if (keep) w = fmax(__dsub_rn(a.R_w, __dsqrt_rn(d)), 0.0);
            if (a.w_src) w = __dmul_rn(w, a.w_src[W.r0 + i]);
            return w;
        };
        if (timing) t_mark = clock64();
        for (int i0 = tid; i0 < ns; i0 += 2 * UPD_THREADS) {
            const int i1 = i0 + UPD_THREADS;
            const bool has1 = i1 < ns;
            const int i1c = has1 ? i1 : i0;
            double q0x, q0y, q0z, q1x, q1y, q1z;
            quick_tf(Ts, a.sx[W.r0 + i0], a.sy[W.r0 + i0], a.sz[W.r0 + i0], q0x, q0y, q0z);
            quick_tf(Ts, a.sx[W.r0 + i1c], a.sy[W.r0 + i1c], a.sz[W.r0 + i1c], q1x, q1y, q1z);
            uint2 hd0 = make_uint2(0u, 0u), hd1 = make_uint2(0u, 0u);
            float x0, y0, z0, x1, y1, z1;
            const bool ok0 = vox_lookup(V, q0x, q0y, q0z, hd0, x0, y0, z0);
            const bool ok1 = has1 && vox_lookup(V, q1x, q1y, q1z, hd1, x1, y1, z1);
            int32_t b0 = -1, b1 = -1;
            double d0 = INFINITY, d1 = INFINITY;
            unsigned ng = 0;
            double w0c[3], w1c[3];                               // the winners' coordinates (modes without a trim: sums right here)
            if (ok0) { vox_scan<8, true>(V, pts, hd0, x0, y0, z0, q0x, q0y, q0z, b0, d0, ng, two_pass ? nullptr : w0c); c_read += hd0.y; c_gather += ng; }
            else     { const WalkHit r = fused_walk(a.g, q0x, q0y, q0z, it > 0 ? idx_s[i0] : -1); b0 = r.bidx; d0 = r.best; ++c_walk; }
            if (has1) {
                if (ok1) { vox_scan<8, true>(V, pts, hd1, x1, y1, z1, q1x, q1y, q1z, b1, d1, ng, two_pass ? nullptr : w1c); c_read += hd1.y; c_gather += ng; }
                else     { const WalkHit r = fused_walk(a.g, q1x, q1y, q1z, it > 0 ? idx_s[i1] : -1); b1 = r.bidx; d1 = r.best; ++c_walk; }
            }
            idx_s[i0] = b0;
            if (has1) idx_s[i1] = b1;
            if constexpr (!two_pass) {
                ModelPointD m;
                if (ok0) { m.x = w0c[0]; m.y = w0c[1]; m.z = w0c[2]; m.pad = 0.0; } else m = a.g.md[b0 >= 0 ? b0 : 0];
                const double w0 = weight_of(i0, b0, d0);
                if (w0 > 0.0) ++n_used;
                icp_accumulate(s, w0, d0, q0x, q0y, q0z, m, px, py, pz);
                if (has1) {
                    if (ok1) { m.x = w1c[0]; m.y = w1c[1]; m.z = w1c[2]; m.pad = 0.0; } else m = a.g.md[b1 >= 0 ? b1 : 0];
                    const double w1 = weight_of(i1, b1, d1);
                    if (w1 > 0.0) ++n_used;
                    icp_accumulate(s, w1, d1, q1x, q1y, q1z, m, px, py, pz);
                }
            }
            if (knn) {
                const bool keep0 = b0 >= 0 && (!reject || d0 < a.thDist2);
                const unsigned long long key0 = keep0 ? dbits(__dsqrt_rn(d0)) : KEY_NOSEL;
                keys_s[i0] = key0;
                if (keep0) atomicAdd(&hsel.hist[bins(key0)], 1);
                if (has1) {
                    const bool keep1 = b1 >= 0 && (!reject || d1 < a.thDist2);
                    const unsigned long long key1 = keep1 ? dbits(__dsqrt_rn(d1)) : KEY_NOSEL;
                    keys_s[i1] = key1;
                    if (keep1) atomicAdd(&hsel.hist[bins(key1)], 1);
                }
            }
        }
        __syncthreads();
        if (timing) { const long long t = clock64(); t_nn += t - t_mark; t_mark = t; }
        // ---- trim: the round(k_frac * kept) smallest residuals, stable tie rule (AlignPoints_KNN.m:20-26) ----
        // (the histogram's total is the number of kept residuals)
        if (knn) {
            const auto k_of_kept = [&](long long nkept) {
                const long long K = (long long)floor(a.k_frac * (double)nkept + 0.5);     // MATLAB round (AlignPoints_KNN.m:21)
                return K > nkept ? nkept : K;
            };
            block_hist_finish(keys_s, ns, bins, k_of_kept, hsel, vK, all_eq, WIN ? a.tie_order + W.r0 : a.tie_order);
        }
        if (timing) { const long long t = clock64(); t_sel += t - t_mark; t_mark = t; }
        // ---- weights + the 17 sums (thread t: correspondences t, t + UPD_THREADS, ... in this order, as k_icp_update) ----
        if (two_pass) {
            for (int i = tid; i < ns; i += UPD_THREADS) {
                const int32_t j = idx_s[i];
#if FUSED_SKIP_UNSELECTED
                // trimmed mode: a correspondence outside the selection has weight zero and would add exact zeros to every sum --
                // its model point is not gathered at all
                if (knn && !(j >= 0 && key_selected(keys_s[i], vK, all_eq))) continue;
#endif
                double qx, qy, qz;
                quick_tf(Ts, a.sx[W.r0 + i], a.sy[W.r0 + i], a.sz[W.r0 + i], qx, qy, qz);
                const ModelPointD m = a.g.md[j >= 0 ? j : 0];
                const double d = j >= 0 ? dist2_exact(m.x, m.y, m.z, qx, qy, qz) : (double)INFINITY;      // the NN step's d2, bit for bit
                const double w = weight_of(i, j, d);
                if (w > 0.0) ++n_used;
                if constexpr (METRIC == ICP_M_GICP)
                    icp_accumulate_gicp(s, w, d, qx, qy, qz, m, a.nrm[j >= 0 ? j : 0], a.snx[W.r0 + i], a.sny[W.r0 + i], a.snz[W.r0 + i], Ts, a.gicp_eps, px, py, pz);
                else if constexpr (METRIC == ICP_M_PLANE) icp_accumulate_plane(s, w, d, qx, qy, qz, m, a.nrm[j >= 0 ? j : 0], px, py, pz);
                else if constexpr (METRIC == ICP_M_COV) icp_accumulate_cov(s, w, d, qx, qy, qz, m, a.nrm[j >= 0 ? j : 0], px, py, pz);
                else icp_accumulate(s, w, d, qx, qy, qz, m, px, py, pz);
            }
        }
        n_used = block_sum_count<NS>(s, n_used, red);
        if (timing) { const long long t = clock64(); t_sum += t - t_mark; t_mark = t; }
        if (tid == 0) {
            const double sw = s[0];
            const double rmse = (sw > 0.0) ? sqrt(s[NS - 1] / sw) : nan("");
            if (a.rmse_hist) {
                if (STOP && last) { for (int c = it; c <= a.iters; ++c) a.rmse_hist[h * a.hist_stride + c] = rmse; }
                else a.rmse_hist[h * a.hist_stride + it] = rmse;
            }
            if (last) { a.rmse[h] = rmse; a.n_used[h] = (int32_t)n_used; }
            if (STOP && last) {
                // a degenerate update at pass p applied p updates and ends the loop with pass p + 1
                if (a.n_iter) a.n_iter[h] = it - s_frozen;
                if (a.converged) a.converged[h] = s_stop && !s_frozen;
            }
            if (METRIC != ICP_M_COV && !last && !s_frozen) {
                if (!STOP) {
                    if (!fused_pose_update<METRIC>(s, n_used, a.pivot, a.reflection_fix != 0, Ts)) s_frozen = 1;
                } else if constexpr (STOP == 2) {
                    const int r = fused_pose_update_extrap(s, n_used, a.pivot, a.reflection_fix != 0, a.stop, a.ex, a.ex_cen + 3 * W.w, it,
                                                           s_ring, s_ring + 2 * ICP_STOP_WINDOW_MAX, Ts);
                    if (r == 0) s_frozen = 1;
                    if (r != 1) s_stop = 1;
                } else {
                    const int r = fused_pose_update_stop<METRIC>(s, n_used, a.pivot, a.reflection_fix != 0, a.stop, it, s_ring, Ts);
                    if (r == 0) s_frozen = 1;
                    if (r != 1) s_stop = 1;
                }
            }
        }
        if constexpr (METRIC == ICP_M_COV) if (last) icp_cov_write(a.cov, s, n_used, a.pivot, h, red);
        if (timing) { const long long t = clock64(); t_svd += t - t_mark; t_mark = t; }
        __syncthreads();
        if (STOP && last) break;
    }
    if (tid < 16) a.T[h * 16 + tid] = Ts[tid];
    if (tid == 0) a.frozen[h] = s_frozen;
    if (STOP == 2 && tid == 0 && a.n_extrap) a.n_extrap[h] = (int32_t)s_ring[2 * ICP_STOP_WINDOW_MAX + 18];
    if (a.idx_out) {
        int32_t* __restrict__ out = a.idx_out + (WIN ? W.idx_base : h * (int64_t)ns);
        for (int r = tid; r < ns; r += UPD_THREADS) out[a.perm ? a.perm[W.r0 + r] : r] = idx_s[r];
    }
    if (a.counters) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c_read += __shfl_xor_sync(0xffffffffu, c_read, o);
            c_gather += __shfl_xor_sync(0xffffffffu, c_gather, o);
            c_walk += __shfl_xor_sync(0xffffffffu, c_walk, o);
        }
        if (tid == 0) {
            atomicAdd(&a.counters[11], (unsigned long long)t_nn); atomicAdd(&a.counters[12], (unsigned long long)t_sel);
            atomicAdd(&a.counters[13], (unsigned long long)t_sum); atomicAdd(&a.counters[14], (unsigned long long)t_svd);
        }
        if ((tid & 31) == 0) {
            if (c_read) atomicAdd(&a.counters[6], c_read);
            if (c_gather) atomicAdd(&a.counters[7], c_gather);
            if (c_walk) atomicAdd(&a.counters[4], c_walk);
        }
    }
}

size_t icp_fused_smem(int64_t ns, int mode) {
    return (((size_t)ns * 4 + 15) / 16) * 16 + (mode == PCREG_ICP_KNN ? (size_t)ns * 8 : 0);
}

template <int METRIC, bool WIN = false>
static const void* fused_kernel(bool knn, int stop) {
    if constexpr (METRIC == ICP_M_COV) {            // no stop
        return knn ? (const void*)k_icp_fused<true, 0, METRIC, WIN> : (const void*)k_icp_fused<false, 0, METRIC, WIN>;
    } else {
        if constexpr (METRIC == ICP_M_POINT)
            if (stop == 2) return knn ? (const void*)k_icp_fused<true, 2, METRIC, WIN> : (const void*)k_icp_fused<false, 2, METRIC, WIN>;
        return knn ? (stop ? (const void*)k_icp_fused<true, 1, METRIC, WIN> : (const void*)k_icp_fused<true, 0, METRIC, WIN>)
                   : (stop ? (const void*)k_icp_fused<false, 1, METRIC, WIN> : (const void*)k_icp_fused<false, 0, METRIC, WIN>);
    }
}

static bool fused_fits(const void* fn, int64_t ns, int mode) {
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, fn) != cudaSuccess) { cudaGetLastError(); return false; }
    return icp_fused_smem(ns, mode) + fa.sharedSizeBytes + 1024 <= ctx().smem_optin;
}

// Point-to-point calls without extrapolation keep the check they always had (the static shared memory of k_icp_fused<true, 0, 0>);
// the others check the instantiation they launch (the other metrics' reduction buffer is 29 instead of 17 doubles x 32, the
// extrapolation adds its state).
bool icp_fused_eligible(const pcreg_model* m, int64_t ns, int64_t nhyp, const pcreg_icp_opts& o, int stop, int metric) {
    if (!m->has_vox || o.nn != PCREG_NN_GRID) return false;
    if (const char* e = getenv("PCREG_FUSED")) { if (e[0] == '0') return false; if (e[0] == '1') nhyp = (int64_t)1 << 40; }
    // one block per hypothesis: a batch smaller than the SM count leaves SMs idle, the per-pass kernels (all SMs on every
    // pass) are faster there (C2, one hypothesis: 13.9 ms fused vs the per-pass path; PCREG_FUSED=1 forces the fused kernel)
    if (nhyp < ctx().sm_count) return false;
    if (ns >= ((int64_t)1 << 30)) return false;
    const bool knn = o.mode == PCREG_ICP_KNN;
    const void* fn = metric == ICP_M_POINT ? (stop == 2 ? fused_kernel<ICP_M_POINT>(knn, 2) : (const void*)k_icp_fused<true, 0, ICP_M_POINT>)
                   : metric == ICP_M_PLANE ? fused_kernel<ICP_M_PLANE>(knn, stop)
                   : metric == ICP_M_GICP ? fused_kernel<ICP_M_GICP>(knn, stop) : fused_kernel<ICP_M_COV>(knn, 0);
    return fused_fits(fn, ns, o.mode);
}

bool icp_fused_windows_fit(const pcreg_model* m, int64_t ns_max, const pcreg_icp_opts& o, int stop, int metric) {
    if (!m->has_vox || o.nn != PCREG_NN_GRID || ns_max >= ((int64_t)1 << 30)) return false;
    const bool knn = o.mode == PCREG_ICP_KNN;
    const void* fn = metric == ICP_M_POINT ? fused_kernel<ICP_M_POINT, true>(knn, stop)
                   : metric == ICP_M_PLANE ? fused_kernel<ICP_M_PLANE, true>(knn, stop)
                   : metric == ICP_M_GICP ? fused_kernel<ICP_M_GICP, true>(knn, stop) : fused_kernel<ICP_M_COV, true>(knn, 0);
    return fused_fits(fn, ns_max, o.mode);
}

template <bool KNN, int STOP, int METRIC, bool WIN, class Args>
static void fused_launch_one(const Args& a, int64_t nhyp, size_t dyn, cudaStream_t st) {
    PCREG_CUDA(cudaFuncSetAttribute(k_icp_fused<KNN, STOP, METRIC, WIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    k_icp_fused<KNN, STOP, METRIC, WIN><<<(unsigned)nhyp, UPD_THREADS, dyn, st>>>(a);
}

template <int METRIC, bool WIN, class Args>
static void fused_launch_metric(const Args& a, int64_t nhyp, int stop, size_t dyn, cudaStream_t st) {
    const bool knn = a.mode == PCREG_ICP_KNN;
    if constexpr (METRIC == ICP_M_COV) {               // no stop
        if (knn) fused_launch_one<true, 0, METRIC, WIN>(a, nhyp, dyn, st);
        else     fused_launch_one<false, 0, METRIC, WIN>(a, nhyp, dyn, st);
    } else {
        if constexpr (METRIC == ICP_M_POINT) {
            if (stop == 2) {
                if (knn) fused_launch_one<true, 2, METRIC, WIN>(a, nhyp, dyn, st);
                else     fused_launch_one<false, 2, METRIC, WIN>(a, nhyp, dyn, st);
                return;
            }
        }
        if (knn && !stop)       fused_launch_one<true, 0, METRIC, WIN>(a, nhyp, dyn, st);
        else if (!knn && !stop) fused_launch_one<false, 0, METRIC, WIN>(a, nhyp, dyn, st);
        else if (knn)           fused_launch_one<true, 1, METRIC, WIN>(a, nhyp, dyn, st);
        else                    fused_launch_one<false, 1, METRIC, WIN>(a, nhyp, dyn, st);
    }
}

template <bool WIN, class Args>
static void fused_launch(const Args& a, int64_t nhyp, int stop, cudaStream_t st) {
    const size_t dyn = icp_fused_smem(a.ns, a.mode);
    if (a.cov.cov)  fused_launch_metric<ICP_M_COV, WIN>(a, nhyp, stop, dyn, st);
    else if (a.snx) fused_launch_metric<ICP_M_GICP, WIN>(a, nhyp, stop, dyn, st);
    else if (a.nrm) fused_launch_metric<ICP_M_PLANE, WIN>(a, nhyp, stop, dyn, st);
    else            fused_launch_metric<ICP_M_POINT, WIN>(a, nhyp, stop, dyn, st);
    PCREG_LAUNCHED();
}

void icp_fused_launch(FusedArgs& a, int64_t nhyp, int stop, cudaStream_t st) { fused_launch<false>(a, nhyp, stop, st); }
void icp_fused_windows_launch(const FusedWinArgs& a, int64_t nhyp, int stop, cudaStream_t st) { fused_launch<true>(a, nhyp, stop, st); }

}  // namespace pcreg
