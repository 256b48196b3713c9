// icp.cu -- the batched ICP loop: (NN) -> select / weight -> 17 FP64 sums -> Kabsch SVD -> pose
// compose, for a batch of independent hypotheses, plus the C-ABI entry points pcreg_icp_batch{,_stop,_metric,_gicp}{,_dev}
// and pcreg_nn_search.
//
// Composition restated from the reference's primitives (SURVEY.md section 8c, oracle/icp.py):
//   pose apply    quickTF.m:5-7
//   rejection     squared-distance compare (ransac.m:49: dist < thDist keeps)
//   trimming      keep round(k_frac * n) smallest residuals, stable sort  (AlignPoints_KNN.m:20-26)
//   weights       w = max(R_w - r, 0)                                      (AlignPoints_weighted.m:16-18)
//   rigid fit     estimateTransform.m:41-71 as estimateTransform(pts1 = model_j, pts2 = q)
//   compose       T <- T * dT (row-vector convention)
//   winner        first-index arg-min of rmse (ransac.m:69-73 tie rule mirrored)
#include <math.h>
#include <float.h>
#include <stdio.h>
#include <cmath>
#include <stdlib.h>
#include <time.h>
#include <algorithm>
#include <vector>
#include <thread>

#include "pcreg_internal.h"
#include "pcreg_dev.cuh"
#include "pcreg_grid.cuh"
#include "pcreg_select.cuh"
#include "pcreg_math.cuh"
#include "pcreg_icp.cuh"

namespace pcreg {

struct Pose16 { double t[16]; };      // a row-major row-vector pose as a kernel argument

// One block per hypothesis.
// NT = threads per hypothesis: UPD_THREADS (the fused kernel's count, so that both sum in the same order and agree bit for
// bit) for sources the fused kernel can take, 512 for large sources (C5: 65 536 correspondences per hypothesis).
// STOP = the tolerance stop (a.stop_iter set); the STOP = 0 instantiations are the loop without it; STOP = 2 (METRIC 0 only, a.ex_state
// set as well) adds the pose extrapolation before the stop rule.
// METRIC = 1: the point-to-plane metric (a.nrm set): 29 sums, the normals gathered with the model points; 2: plane-to-plane
// (a.snx set as well): the same, and each correspondence's source normal read with the source point and rotated by the pose;
// 3 (STOP = 0 only, a.cov.cov set): the covariance pass of pcreg_icp_covariance, the final pass alone, writing a.cov instead of a pose.
template <int NT, int STOP, int METRIC>
__global__ void __launch_bounds__(NT, NT <= 256 ? 3 : 1) k_icp_update(const __grid_constant__ IcpUpdateArgs a) {
    constexpr int NS = icp_nsums<METRIC>;
    constexpr bool MNRM = METRIC != ICP_M_POINT, SNRM = METRIC == ICP_M_GICP;
    __shared__ double Ts[16];
    __shared__ double red[(NS + 1) * 32];
    __shared__ long long redll[32];
    __shared__ HistSelShared hsel;
    __shared__ unsigned long long red_u64[64];

    const int64_t h = blockIdx.x;
    const int tid = threadIdx.x;
    const int64_t ns = a.ns;
    if (STOP && a.update && a.stop_iter[h] >= 0) return;       // stopped: intermediate passes leave it alone
    if (tid < 16) Ts[tid] = a.T[h * 16 + tid];
    __syncthreads();
    const int32_t* __restrict__ idx = a.idx + h * ns;
    const double* __restrict__ d2 = a.d2 + h * ns;
    const bool reject = a.thDist2 > 0.0;

    unsigned long long vK = 0ull;
    bool all_eq = false;
    double trim_tau = INFINITY;             // KNN mode: the largest selected residual (K-th smallest distance)
    if (a.mode == PCREG_ICP_KNN) {
        unsigned long long* __restrict__ keys = a.keys + h * ns;
        long long nkept = 0;
        unsigned long long kmin = ~0ull, kmax = 0ull;
        constexpr int KU = 4;                                  // residuals / indices of a trip are loaded before any is used
        for (int64_t i0 = tid; i0 < ns; i0 += (int64_t)KU * NT) {
            double dv[KU]; int32_t jv[KU];
#pragma unroll
            for (int u = 0; u < KU; ++u) { const int64_t i = i0 + (int64_t)u * NT; const bool ok = i < ns; dv[u] = ok ? d2[i] : 0.0; jv[u] = ok ? idx[i] : -1; }
#pragma unroll
            for (int u = 0; u < KU; ++u) {
                const int64_t i = i0 + (int64_t)u * NT;
                if (i >= ns) break;
                const double d = dv[u];
                const bool keep = jv[u] >= 0 && (!reject || d < a.thDist2);
                const unsigned long long key = keep ? dbits(__dsqrt_rn(d)) : KEY_NOSEL;
                keys[i] = key;
                if (keep) { ++nkept; kmin = key < kmin ? key : kmin; kmax = key > kmax ? key : kmax; }
            }
        }
        nkept = block_sum_ll(nkept, redll);
        {   // block min / max of the kept keys
            const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long a0 = __shfl_xor_sync(0xffffffffu, kmin, o), a1 = __shfl_xor_sync(0xffffffffu, kmax, o);
                kmin = a0 < kmin ? a0 : kmin;
                kmax = a1 > kmax ? a1 : kmax;
            }
            if (lane == 0) { red_u64[warp] = kmin; red_u64[32 + warp] = kmax; }
            __syncthreads();
            kmin = ~0ull; kmax = 0ull;
            for (int w = 0; w < NT / 32; ++w) {
                kmin = red_u64[w] < kmin ? red_u64[w] : kmin;
                kmax = red_u64[32 + w] > kmax ? red_u64[32 + w] : kmax;
            }
            __syncthreads();
        }
        long long K = (long long)floor(a.k_frac * (double)nkept + 0.5);     // MATLAB round (AlignPoints_KNN.m:21)
        if (K > nkept) K = nkept;
        block_hist_select(keys, ns, K, kmin, kmax, hsel, vK, all_eq, a.tie_order);
        if (!reject && K >= 1 && K < nkept && nkept == ns) trim_tau = __longlong_as_double((long long)vK);
    }

    // ---- weights + the 17 (29) sums ----
    double s[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) s[k] = 0.0;
    long long n_used = 0;
    const double px = a.pivot[0], py = a.pivot[1], pz = a.pivot[2];
    // Branch-free body, four correspondences per trip: the index / residual / source loads and the model gathers
    // of a trip are independent, so they are all in flight together (the loop is bound by their latency).
    // A zero weight contributes exact zeros to every sum.
    auto weight_of = [&](int64_t i, int32_t j, double d) -> double {
        const bool keep = j >= 0 && (!reject || d < a.thDist2);
        double w = 0.0;
        if (a.mode == PCREG_ICP_PLAIN) {
            w = keep ? 1.0 : 0.0;
        } else if (a.mode == PCREG_ICP_KNN) {
            const unsigned long long key = a.keys[h * ns + i];
            w = (j >= 0 && key_selected(key, vK, all_eq)) ? 1.0 : 0.0;
        } else if (keep) {
            w = fmax(__dsub_rn(a.R_w, __dsqrt_rn(d)), 0.0);
        }
        if (a.w_src) w = __dmul_rn(w, a.w_src[i]);
        return w;
    };
    // The correspondence indices of a trip are loaded one trip AHEAD: the model gathers -- the only loads that depend on
    // another load -- then go out at the top of the trip together with everything else (one memory latency per trip, not two).
    constexpr int UB = 4;
    int32_t jn[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) { const int64_t i = (int64_t)tid + (int64_t)u * NT; jn[u] = i < ns ? idx[i] : -1; }
    for (int64_t i0 = tid; i0 < ns; i0 += (int64_t)UB * NT) {
        int32_t jj[UB]; double dd[UB], xs[UB], ys[UB], zs[UB], ww[UB];
        ModelPointD mm[UB], nv[MNRM ? UB : 1];
        double snx[SNRM ? UB : 1], sny[SNRM ? UB : 1], snz[SNRM ? UB : 1];
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            jj[u] = jn[u]; mm[u] = a.md[jj[u] >= 0 ? jj[u] : 0];
            if constexpr (MNRM) nv[u] = a.nrm[jj[u] >= 0 ? jj[u] : 0];
        }
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            const int64_t i = i0 + (int64_t)u * NT;
            const bool ok = i < ns;
            const int64_t ic = ok ? i : tid;                 // tid < ns is guaranteed inside the loop
            dd[u] = d2[ic];
            xs[u] = a.sx[ic]; ys[u] = a.sy[ic]; zs[u] = a.sz[ic];
            if constexpr (SNRM) { snx[u] = a.snx[ic]; sny[u] = a.sny[ic]; snz[u] = a.snz[ic]; }
            const int64_t in = i + (int64_t)UB * NT;
            jn[u] = in < ns ? idx[in] : -1;
        }
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            const int64_t i = i0 + (int64_t)u * NT;
            ww[u] = (i < ns) ? weight_of(i, jj[u], dd[u]) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < UB; ++u) {
            const double w = ww[u], d = dd[u];
            if (w > 0.0) ++n_used;
            double qx, qy, qz;
            quick_tf(Ts, xs[u], ys[u], zs[u], qx, qy, qz);
            if constexpr (SNRM) icp_accumulate_gicp(s, w, d, qx, qy, qz, mm[u], nv[u], snx[u], sny[u], snz[u], Ts, a.gicp_eps, px, py, pz);
            else if constexpr (METRIC == ICP_M_COV) icp_accumulate_cov(s, w, d, qx, qy, qz, mm[u], nv[u], px, py, pz);
            else if constexpr (MNRM) icp_accumulate_plane(s, w, d, qx, qy, qz, mm[u], nv[u], px, py, pz);
            else icp_accumulate(s, w, d, qx, qy, qz, mm[u], px, py, pz);
        }
    }
    n_used = block_sum_count<NS>(s, n_used, red);

    if (tid == 0) {
        const double sw = s[0];
        const double rmse = (sw > 0.0) ? sqrt(s[NS - 1] / sw) : nan("");
        a.rmse[h] = rmse;
        a.n_used[h] = (int32_t)n_used;
        int hist_from = a.hist_col;
        if (STOP && !a.update) {
            // final pass: a hypothesis stopped after k updates would have had its final pass at column k (converged) or k + 1
            // (frozen at pass k); every column from there holds the final rmse
            const int k = a.stop_iter[h];
            if (k >= 0) hist_from = k + a.frozen[h];
            if (a.n_iter) a.n_iter[h] = k >= 0 ? k : a.hist_col;
            if (a.converged) a.converged[h] = k >= 0 && !a.frozen[h];
            if (STOP == 2 && a.n_extrap) a.n_extrap[h] = (int32_t)a.ex_state[h * EXTRAP_STATE + 18];
        }
        if (a.rmse_hist) for (int c = hist_from; c <= a.hist_col; ++c) a.rmse_hist[h * a.hist_stride + c] = rmse;
        float moved = 0.f;
        if (METRIC != ICP_M_COV && a.update && !a.frozen[h]) {
            double Tn[16], Tc[16];
            for (int k = 0; k < 16; ++k) Tc[k] = Ts[k];
            bool ok;
            if constexpr (MNRM) ok = icp_pose_update_plane_call(s, n_used, a.pivot, Tc, Tn);
            else ok = icp_pose_update_call(s, n_used, a.pivot, a.reflection_fix != 0, Tc, Tn);
            if (!ok) {
                a.frozen[h] = 1;
                if (STOP) a.stop_iter[h] = a.hist_col;
            } else {
                // extrapolation: Tn becomes the pose actually written, so the motion bound below and the stop rule see the jump
                if constexpr (STOP == 2) icp_extrap_update(a.ex, s, a.pivot, a.ex_cen, Tc, Tn, a.hist_col + 1, a.ex_state + h * EXTRAP_STATE);
                for (int k = 0; k < 16; ++k) a.T[h * 16 + k] = Tn[k];
                if (a.delta) {
                    // upper bound of how far this update moves any source point:
                    // q' - q = (x - c)(R' - R) + [c (R' - R) + (t' - t)],  |x - c| <= r_max
                    double fro = 0.0, v[3];
                    for (int c = 0; c < 3; ++c) {
                        v[c] = Tn[12 + c] - Tc[12 + c];
                        for (int r = 0; r < 3; ++r) {
                            const double dr = Tn[r * 4 + c] - Tc[r * 4 + c];
                            fro += dr * dr;
                            v[c] += a.src_stats[r] * dr;
                        }
                    }
                    const double dl = sqrt(fro) * a.src_stats[3] + sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
                    moved = __double2float_ru(dl * (1.0 + 1e-9)) + 1e-30f;
                }
                // stopped: the pose no longer moves.  The passes up to the final one compute nothing this hypothesis uses.
                if (STOP && icp_stop_update(a.stop, Tc, Tn, a.hist_col + 1, a.stop_ring + h * (2 * ICP_STOP_WINDOW_MAX))) {
                    a.stop_iter[h] = a.hist_col + 1;
                    moved = 0.f;
                }
            }
        }
        if (a.delta) a.delta[h] = moved;
        // Lazy trimming (nn_grid.cu, k_nn_list): the NN distance is 1-Lipschitz in the query position and the next pass
        // moves no query by more than `moved`, so the K selected residuals stay <= tau + moved; a query whose residual
        // was > tau + 2 moved stays strictly outside the selected set and its search can be skipped in the next pass.
        // The same holds for a rejection threshold (residual >= sqrt(thDist2) + moved stays rejected) and for the
        // weighted mode (residual >= R_w + moved keeps weight zero).  With a rejection threshold the number of kept
        // correspondences, hence K, may change from pass to pass, so the trim bound is only used without one.
        if (a.skip_thr) {
            double thr = INFINITY;
            if (a.update && a.delta) {
                // The skipping kernel replaces the residual by  nl = sd (1 - 1e-12) - moved (1 + 1e-6)  and skips when
                // sd (1 - 1e-12) > thr: with thr = bound (1 + 1e-9) + moved (1 + 2e-6) the stored stand-in stays STRICTLY above the
                // bound it must stay above (tau + moved for the trim, sqrt(thDist2) for the rejection, R_w for the weights).
                const double mv = (double)moved * (1.0 + 2e-6);
                thr = (trim_tau + (double)moved) * (1.0 + 1e-9) + mv;
                if (reject) thr = fmin(thr, sqrt(a.thDist2) * (1.0 + 1e-9) + mv);
                if (a.mode == PCREG_ICP_WEIGHTED) thr = fmin(thr, a.R_w * (1.0 + 1e-9) + mv);
            }
            a.skip_thr[h] = thr;
        }
    }
    if constexpr (METRIC == ICP_M_COV) icp_cov_write(a.cov, s, n_used, a.pivot, h, red);
}

// centroid and radius of the source cloud (for the per-update motion bound): one block
__global__ void __launch_bounds__(1024) k_src_stats(const double* __restrict__ src, int64_t ns, double* __restrict__ stats /*[4]*/) {
    __shared__ double red[3 * 32];
    __shared__ double cen[3];
    double s[3] = {0.0, 0.0, 0.0};
    for (int64_t i = threadIdx.x; i < ns; i += blockDim.x) { s[0] += src[i]; s[1] += src[ns + i]; s[2] += src[2 * ns + i]; }
    block_sum<3>(s, red);
    if (threadIdx.x == 0) for (int k = 0; k < 3; ++k) cen[k] = s[k] / (double)ns;
    __syncthreads();
    double r2 = 0.0;
    for (int64_t i = threadIdx.x; i < ns; i += blockDim.x) {
        const double dx = src[i] - cen[0], dy = src[ns + i] - cen[1], dz = src[2 * ns + i] - cen[2];
        r2 = fmax(r2, dx * dx + dy * dy + dz * dz);
    }
    for (int o = 16; o > 0; o >>= 1) r2 = fmax(r2, __shfl_xor_sync(0xffffffffu, r2, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = r2;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, red[w]);
        stats[0] = cen[0]; stats[1] = cen[1]; stats[2] = cen[2];
        stats[3] = sqrt(m) * (1.0 + 1e-12);
    }
}

// Unweighted FP64 centroid of each window's source rows (the pose extrapolation's c), one block per window: block w sums rows
// off[w] .. off[w + 1] - 1 of src (column stride ld) in a fixed order (thread t: rows t, t + 256, ...; then block_sum's tree), so
// the result depends on the window's rows alone.
__global__ void __launch_bounds__(256) k_src_centroid(const double* __restrict__ src, int64_t ld, const int64_t* __restrict__ off,
                                                      double* __restrict__ cen /*[nwin][3]*/) {
    __shared__ double red[3 * 32];
    const int64_t r0 = off[blockIdx.x], ns = off[blockIdx.x + 1] - r0;
    double s[3] = {0.0, 0.0, 0.0};
    for (int64_t i = r0 + threadIdx.x; i < r0 + ns; i += 256) { s[0] += src[i]; s[1] += src[ld + i]; s[2] += src[2 * ld + i]; }
    block_sum<3>(s, red);
    if (threadIdx.x == 0) for (int k = 0; k < 3; ++k) cen[blockIdx.x * 3 + k] = ns > 0 ? s[k] / (double)ns : 0.0;
}

// first-index arg-min over hypotheses, NaN never wins (-1: none); one block per segment: block b takes rmse[seg[b] .. seg[b + 1] - 1]
// and writes best[b] relative to seg[b] (seg null: one segment of n).
__global__ void __launch_bounds__(1024) k_icp_argmin(const double* __restrict__ rmse, const int64_t* __restrict__ seg, int64_t n,
                                                     int64_t* __restrict__ best) {
    if (seg) { rmse += seg[blockIdx.x]; n = seg[blockIdx.x + 1] - seg[blockIdx.x]; }
    __shared__ double sv[32];
    __shared__ long long si[32];
    double bv = INFINITY;
    long long bi = -1;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const double v = rmse[i];
        if (v == v && (bi < 0 || v < bv)) { bv = v; bi = i; }     // strided scan keeps the lowest index per thread on ties
    }
    auto better = [](double v, long long i, double ov, long long oi) {
        if (oi < 0) return false;
        if (i < 0) return true;
        return ov < v || (ov == v && oi < i);
    };
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(bv, bi, ov, oi)) { bv = ov; bi = oi; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sv[warp] = bv; si[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        bv = lane < nw ? sv[lane] : INFINITY;
        bi = lane < nw ? si[lane] : -1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better(bv, bi, ov, oi)) { bv = ov; bi = oi; }
        }
        if (lane == 0) best[blockIdx.x] = bi;
    }
}

// ---- spatial sort of the source cloud (one block) ----------------------------------------------------
// Threads of a warp then work on neighbouring queries under every pose (a rigid transform keeps
// neighbours neighbours): the pyramid walks of a warp stay together and hit the same cache lines.
// Results are un-permuted at the end; the stable tie rule of the trim keeps using ORIGINAL indices.
__device__ __forceinline__ unsigned spread10(unsigned v) {
    v &= 1023u;
    v = (v | (v << 16)) & 0x030000FFu;
    v = (v | (v << 8)) & 0x0300F00Fu;
    v = (v | (v << 4)) & 0x030C30C3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
// One block per window: window b is rows off[b] .. off[b + 1] - 1 of src (column stride ld; off null: one window of ns rows).  A window
// of 64 .. 2^17 rows is sorted as the single-block sort is sized; any other gets the identity order (the single-source call does not
// launch the sort for those).  perm / inv are relative to the window's first row; keys: scratch of 2 ld entries (a window's power of
// two stays below twice its row count).
__global__ void __launch_bounds__(1024) k_src_sort(const double* __restrict__ src, const double* __restrict__ w, int64_t ld,
                                                   const int64_t* __restrict__ off, int64_t ns, unsigned long long* __restrict__ keys,
                                                   double* __restrict__ out_src, double* __restrict__ out_w, int32_t* __restrict__ perm,
                                                   int32_t* __restrict__ inv) {
    __shared__ double red[6 * 32];
    const int tid = threadIdx.x;
    if (off) {
        const int64_t r0 = off[blockIdx.x];
        ns = off[blockIdx.x + 1] - r0;
        src += r0; out_src += r0; perm += r0; inv += r0; keys += 2 * r0;
        if (w) { w += r0; out_w += r0; }
    }
    if (ns < 64 || ns > (1 << 17)) {
        for (int64_t r = tid; r < ns; r += blockDim.x) {
            perm[r] = (int32_t)r;
            inv[r] = (int32_t)r;
            out_src[r] = src[r]; out_src[ld + r] = src[ld + r]; out_src[2 * ld + r] = src[2 * ld + r];
            if (w) out_w[r] = w[r];
        }
        return;
    }
    int npow2 = 1;
    while (npow2 < ns) npow2 <<= 1;
    double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int64_t i = tid; i < ns; i += blockDim.x)
        for (int a = 0; a < 3; ++a) { const double v = src[a * ld + i]; mn[a] = fmin(mn[a], v); mx[a] = fmax(mx[a], v); }
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o > 0; o >>= 1) { mn[a] = fmin(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o)); mx[a] = fmax(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o)); }
        if ((tid & 31) == 0) { red[a * 32 + (tid >> 5)] = mn[a]; red[(3 + a) * 32 + (tid >> 5)] = mx[a]; }
    }
    __syncthreads();
    double ext = 0.0;
    for (int a = 0; a < 3; ++a) {
        double lo = INFINITY, hi = -INFINITY;
        for (int wq = 0; wq < (int)(blockDim.x >> 5); ++wq) { lo = fmin(lo, red[a * 32 + wq]); hi = fmax(hi, red[(3 + a) * 32 + wq]); }
        mn[a] = lo;
        ext = fmax(ext, hi - lo);
    }
    const double scale = ext > 0.0 ? 1023.0 / ext : 0.0;
    for (int i = tid; i < npow2; i += blockDim.x) {
        unsigned long long k = ~0ull;
        if (i < ns) {
            const unsigned cx = (unsigned)((src[i] - mn[0]) * scale), cy = (unsigned)((src[ld + i] - mn[1]) * scale),
                           cz = (unsigned)((src[2 * ld + i] - mn[2]) * scale);
            const unsigned code = spread10(cx) | (spread10(cy) << 1) | (spread10(cz) << 2);
            k = ((unsigned long long)code << 32) | (unsigned long long)(unsigned)i;
        }
        keys[i] = k;
    }
    __syncthreads();
    for (int k = 2; k <= npow2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < npow2; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const unsigned long long x = keys[i], y = keys[l];
                    const bool up = (i & k) == 0;
                    if ((x > y) == up) { keys[i] = y; keys[l] = x; }
                }
            }
            __syncthreads();
        }
    for (int64_t r = tid; r < ns; r += blockDim.x) {
        const int32_t o = (int32_t)(unsigned)(keys[r] & 0xffffffffull);
        perm[r] = o;
        inv[o] = (int32_t)r;
        out_src[r] = src[o]; out_src[ld + r] = src[ld + o]; out_src[2 * ld + r] = src[2 * ld + o];
        if (w) out_w[r] = w[o];
    }
}
// out[h][orig] = in[h][inv[orig]]
__global__ void k_unpermute_idx(const int32_t* __restrict__ in, const int32_t* __restrict__ inv, int64_t ns, int64_t nhyp,
                                int32_t* __restrict__ out) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ns * nhyp) return;
    const int64_t h = g / ns, o = g - h * ns;
    out[g] = in[h * ns + inv[o]];
}

// Source normals of the plane-to-plane metric, one thread per row: out row r (the order of the sorted source) is input row perm[r]
// (perm null: r) normalised in FP64 as pcreg_model_set_normals normalises (no contraction into FMA: the same bits as the host
// loop).  A zero or non-finite row sets *bad.  in, out: column-major, column stride ld.  Windowed calls: blockIdx.y is the window,
// rows off[y] .. off[y + 1] - 1, perm relative to the window's first row (off null: one window of ns rows).
__global__ void k_src_normals(const double* __restrict__ in, const int32_t* __restrict__ perm, int64_t ld, const int64_t* __restrict__ off,
                              int64_t ns, double* __restrict__ out, int* __restrict__ bad) {
    const int64_t r0 = off ? off[blockIdx.y] : 0;
    if (off) ns = off[blockIdx.y + 1] - r0;
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= ns) return;
    const int64_t o = r0 + (perm ? perm[r0 + r] : r);
    const double x = in[o], y = in[ld + o], z = in[2 * ld + o];
    const double n = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)));
    if (!(isfinite(n) && n > 0.0)) *bad = 1;
    out[r0 + r] = x / n; out[ld + r0 + r] = y / n; out[2 * ld + r0 + r] = z / n;
}

// MATLAB column-major 4x4 <-> internal row-major 4x4 (a transpose), batched
__global__ void k_transpose16(const double* __restrict__ in, double* __restrict__ out, int64_t n) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n * 16) return;
    const int64_t h = g >> 4;
    const int e = (int)(g & 15), r = e >> 2, c = e & 3;
    out[h * 16 + r * 4 + c] = in[h * 16 + c * 4 + r];
}

// [p 1] * T for a whole cloud (quickTF.m:5-7), T row-major in constant arguments; class of the input kept
template <typename F>
__global__ void k_quick_tf(const F* __restrict__ in, int64_t n, int64_t ld_in, F* __restrict__ out, int64_t ld_out, const __grid_constant__ Pose16 T) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double qx, qy, qz;
    quick_tf(T.t, (double)in[i], (double)in[ld_in + i], (double)in[2 * ld_in + i], qx, qy, qz);
    out[i] = (F)qx; out[ld_out + i] = (F)qy; out[2 * ld_out + i] = (F)qz;
}

void transpose16_launch(const double* d_in, double* d_out, int64_t n, cudaStream_t st) {
    k_transpose16<<<(unsigned)((n * 16 + 255) / 256), 256, 0, st>>>(d_in, d_out, n);
    PCREG_LAUNCHED();
}
template <int METRIC>
static void icp_update_launch_metric(const IcpUpdateArgs& a, int64_t nhyp, cudaStream_t st) {
    const bool stop = a.stop_iter != nullptr;
    if constexpr (METRIC == ICP_M_POINT) {
        if (a.ex_state) {
            if (a.ns > 20000) k_icp_update<512, 2, METRIC><<<(unsigned)nhyp, 512, 0, st>>>(a);
            else              k_icp_update<UPD_THREADS, 2, METRIC><<<(unsigned)nhyp, UPD_THREADS, 0, st>>>(a);
            return;
        }
    }
    if (a.ns > 20000) { if (stop) k_icp_update<512, 1, METRIC><<<(unsigned)nhyp, 512, 0, st>>>(a); else k_icp_update<512, 0, METRIC><<<(unsigned)nhyp, 512, 0, st>>>(a); }
    else if (stop)    k_icp_update<UPD_THREADS, 1, METRIC><<<(unsigned)nhyp, UPD_THREADS, 0, st>>>(a);
    else              k_icp_update<UPD_THREADS, 0, METRIC><<<(unsigned)nhyp, UPD_THREADS, 0, st>>>(a);
}
// the covariance pass has no stop and no extrapolation
template <>
void icp_update_launch_metric<ICP_M_COV>(const IcpUpdateArgs& a, int64_t nhyp, cudaStream_t st) {
    if (a.ns > 20000) k_icp_update<512, 0, ICP_M_COV><<<(unsigned)nhyp, 512, 0, st>>>(a);
    else              k_icp_update<UPD_THREADS, 0, ICP_M_COV><<<(unsigned)nhyp, UPD_THREADS, 0, st>>>(a);
}
void icp_update_launch(const IcpUpdateArgs& a, int64_t nhyp, cudaStream_t st) {
    if (a.cov.cov)  icp_update_launch_metric<ICP_M_COV>(a, nhyp, st);
    else if (a.snx) icp_update_launch_metric<ICP_M_GICP>(a, nhyp, st);
    else if (a.nrm) icp_update_launch_metric<ICP_M_PLANE>(a, nhyp, st);
    else            icp_update_launch_metric<ICP_M_POINT>(a, nhyp, st);
    PCREG_LAUNCHED();
}
void icp_argmin_launch(const double* d_rmse, int64_t nhyp, int64_t* d_best, cudaStream_t st, const int64_t* d_seg, int64_t nseg) {
    k_icp_argmin<<<(unsigned)nseg, 1024, 0, st>>>(d_rmse, d_seg, nhyp, d_best);
    PCREG_LAUNCHED();
}

// ------------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------------
struct EventPair { cudaEvent_t a, b; int kind; };
static bool debug_times() { static int v = -1; if (v < 0) { const char* e = getenv("PCREG_DEBUG_TIMES"); v = (e && e[0] == '1') ? 1 : 0; } return v == 1; }

static void icp_run(const pcreg_model* m, const double* d_src /*col-major ns x 3, ld = ns*/, int64_t ns,
                    const double* d_w, const double* d_T0_cm, int64_t nhyp, const pcreg_icp_opts& o,
                    double* d_T16_cm, double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx,
                    double* d_rmse_hist, int64_t* d_best, cudaStream_t st,
                    const pcreg_icp_stop* stop = nullptr, int32_t* d_n_iter = nullptr, int32_t* d_converged = nullptr,
                    int metric = ICP_M_POINT, const double* d_src_nrm = nullptr /*ICP_M_GICP: col-major ns x 3*/, double gicp_eps = 0.0,
                    const IcpExtrapRule* ex = nullptr /*needs stop*/, const double* d_ex_cen = nullptr /*[3]*/, int32_t* d_n_extrap = nullptr,
                    const IcpCovOut* cov = nullptr /*metric ICP_M_COV, iters 0*/) {
    PCREG_REQUIRE(m && d_src && d_T0_cm && d_T16_cm, "icp: null pointer");
    const bool plane = metric != ICP_M_POINT, gicp = metric == ICP_M_GICP;
    const ModelPointD* nrm = plane ? m->nrm.p : nullptr;
    if (plane && !nrm) throw StateError{"icp: the point-to-plane and plane-to-plane metrics need model normals (pcreg_model_set_normals / pcreg_model_compute_normals)"};
    PCREG_REQUIRE(!gicp || d_src_nrm, "icp: the plane-to-plane metric needs source normals");
    PCREG_REQUIRE(ns >= 1 && nhyp >= 1, "icp: need ns >= 1 and nhyp >= 1");
    PCREG_REQUIRE(o.iters >= 0, "icp: iters must be >= 0");
    PCREG_REQUIRE(o.mode >= PCREG_ICP_PLAIN && o.mode <= PCREG_ICP_WEIGHTED, "icp: bad mode");
    PCREG_REQUIRE(o.nn == PCREG_NN_BRUTE || o.nn == PCREG_NN_GRID, "icp: bad nn kind");
    if (o.nn == PCREG_NN_GRID) PCREG_REQUIRE(m->has_grid, "icp: grid NN requested but the model has no grid");
    Context& c = ctx();
    const bool prof = c.profiling;
    for (int i = 0; i < 32; ++i) c.profile[i] = 0.0;
    static const bool dbg_host = [] { const char* e = getenv("PCREG_DEBUG_HOST"); return e && e[0] == '1'; }();
    auto now_ms = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return 1e3 * ts.tv_sec + 1e-6 * ts.tv_nsec; };
    const double t_enter = now_ms();
    double t_alloc = 0, t_sorted = 0, t_enq = 0;

    PCREG_REQUIRE(!ex || (stop && d_ex_cen && metric == ICP_M_POINT), "icp: extrapolation needs a stop rule, the centroid and point-to-point");
    PCREG_REQUIRE((cov != nullptr) == (metric == ICP_M_COV) && (!cov || (o.iters == 0 && !stop)), "icp: the covariance pass runs alone");
    const int stop_mode = ex ? 2 : stop ? 1 : 0;
    const bool fused = icp_fused_eligible(m, ns, nhyp, o, stop_mode, metric);
    // chunk the hypotheses so that the per-correspondence scratch stays bounded
    const size_t total_b = c.total_mem;         // queried once at pcreg_init (cudaMemGetInfo costs up to tens of ms per call)
    const size_t per_hyp = (size_t)ns * (4 + 4 + 8 + (o.mode == PCREG_ICP_KNN ? 8 : 0) + (o.nn == PCREG_NN_GRID ? 8 + (m->has_vox ? 0 : 28 + 4 * 64 + 4 * 448 / 16) : 0));
    const size_t budget = std::max<size_t>((size_t)1 << 30, std::min<size_t>((size_t)24 << 30, total_b / 6));
    // Two sub-batches ("lanes") on two streams: every kernel of the loop is latency bound with a tail (a few slow
    // queries, a block per hypothesis), so the kernels of one lane fill the gaps of the other.  Profiling runs use one
    // lane so that the per-kernel event times stay meaningful.  PCREG_LANES=1 disables.
    const char* lanes_e = getenv("PCREG_LANES");                            // 1 = off, 2 = on whatever the batch size (tests)
    const int lanes_env = lanes_e ? atoi(lanes_e) : 0;
    constexpr int MAX_LANES = 4;
    const int lanes_want = lanes_env > 2 ? std::min(lanes_env, MAX_LANES) : 2;
    const int nlanes = (prof || lanes_env == 1 || nhyp < 2 || (lanes_env < 2 && (double)nhyp * (double)ns < 2.0e6)) ? 1
                       : (int)std::min<int64_t>(lanes_want, nhyp);
    int64_t hc = (int64_t)std::max<size_t>(1, budget / (per_hyp * (size_t)nlanes));
    if (const char* e = getenv("PCREG_MAX_CHUNK_HYP")) { const long v = atol(e); if (v > 0) hc = std::min<int64_t>(hc, v); }   // tests: force several chunks
    hc = std::min(hc, (nhyp + nlanes - 1) / nlanes);
    hc = std::min<int64_t>(hc, 2147483647LL / std::max<int64_t>(1, ns) );       // int32 grid.x of per-query kernels stays safe
    hc = std::max<int64_t>(hc, 1);

    DevBuf<double> Twork((size_t)nhyp * 16);
    DevBuf<int32_t> frozen((size_t)nhyp);
    DevBuf<double> rmse_tmp(d_rmse ? 0 : (size_t)nhyp);
    DevBuf<int32_t> nused_tmp(d_n_used ? 0 : (size_t)nhyp);
    DevBuf<unsigned long long> counters(16);
    IcpStopRule rule{};
    if (stop) { rule.tol_t = stop->tol_t; rule.tol_r_deg = stop->tol_r_deg; rule.window = stop->window; }
    // tolerance stop, per-pass path: per-hypothesis stop state (the fused kernel keeps it in shared memory)
    DevBuf<int32_t> stop_iter(stop && !fused ? (size_t)nhyp : 0);
    DevBuf<double> stop_ring(stop && !fused ? (size_t)nhyp * 2 * ICP_STOP_WINDOW_MAX : 0);
    DevBuf<double> ex_state(ex && !fused ? (size_t)nhyp * EXTRAP_STATE : 0);
    // profiling with the tolerance stop: the passes each hypothesis ran follow from n_iter and status
    DevBuf<int32_t> n_iter_tmp(stop && prof && !d_n_iter ? (size_t)nhyp : 0);
    if (n_iter_tmp.p) d_n_iter = n_iter_tmp.p;
    auto passes_run = [&]() -> double {       // after the stream has drained
        std::vector<int32_t> ni((size_t)nhyp), fz((size_t)nhyp);
        PCREG_CUDA(cudaMemcpy(ni.data(), d_n_iter, ni.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
        PCREG_CUDA(cudaMemcpy(fz.data(), frozen.p, fz.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
        double n = 0.0;
        for (int64_t h = 0; h < nhyp; ++h) n += (double)ni[h] + 1.0 + (double)fz[h];   // frozen at pass p: n_iter = p, p + 2 passes
        return n;
    };
    // candidate lists (grid NN, nn_grid.cu): built by the full searches once a pose has nearly stopped moving,
    // scanned instead of searching while the query stays inside its list's guarantee.  PCREG_LISTS=0 disables.
    static const bool lists_on = [] { const char* e = getenv("PCREG_LISTS"); return !(e && e[0] == '0'); }();
    static const double list_skin_cells = [] { const char* e = getenv("PCREG_LIST_SKIN"); return e ? atof(e) : 0.5; }();
    static const int list_cap = [] { const char* e = getenv("PCREG_LIST_CAP"); int v = e ? atoi(e) : 64; return std::max(4, (v + 3) & ~3); }();
    // (a model with a Voronoi voxel map answers every pass with one list scan per query: no per-query lists, nn_vox.cu)
    const bool use_lists = (o.nn == PCREG_NN_GRID) && lists_on && o.iters >= 3 && m->n <= ((int64_t)1 << 24) && !m->has_vox;
    const int ext_cap = 448;                                               // wide balls: up to list_cap + 448 candidates
    const int64_t ext_slots = use_lists ? std::max<int64_t>(1024, hc * ns / 16) : 0;
    DevBuf<float> delta(use_lists ? (size_t)nhyp : 0);
    // lazy trimming: residual above which a query of hypothesis h cannot be selected in the next pass (update kernel)
    static const bool lazy_on = [] { const char* e = getenv("PCREG_LAZY_TRIM"); return !(e && e[0] == '0'); }();
    const bool lazy_trim = use_lists && lazy_on && (o.mode == PCREG_ICP_KNN || o.mode == PCREG_ICP_WEIGHTED || o.thDist2 > 0.0);
    DevBuf<double> skip_thr(lazy_trim ? (size_t)nhyp : 0);
    struct Lane {
        cudaStream_t st = nullptr;
        DevBuf<int32_t> idxA, idxB, cl_list, cl_ext, cl_ext_list;
        DevBuf<double> d2;
        DevBuf<unsigned long long> keys;
        DevBuf<float4> cl_hdr;
        DevBuf<int2> cl_cnt;
        DevBuf<unsigned int> cl_ext_count;
        NNScratch scratch;
        GridScratch gscratch;
        CandView cl{};
        int32_t* cur = nullptr; int32_t* prev = nullptr;
        bool have_prev = false;
        int64_t h0 = 0, hn = 0;
    };
    Lane lanes[MAX_LANES];
    for (int l = 0; l < nlanes && !fused; ++l) {
        Lane& L = lanes[l];
        L.st = (nlanes == 1) ? st : lane_stream(l);
        L.idxA.alloc((size_t)hc * ns); L.idxB.alloc((size_t)hc * ns); L.d2.alloc((size_t)hc * ns);
        if (o.mode == PCREG_ICP_KNN) L.keys.alloc((size_t)hc * ns);
        if (use_lists) {
            L.cl_hdr.alloc((size_t)hc * ns); L.cl_cnt.alloc((size_t)hc * ns); L.cl_list.alloc((size_t)hc * ns * list_cap);
            L.cl_ext.alloc((size_t)hc * ns); L.cl_ext_list.alloc((size_t)ext_slots * ext_cap); L.cl_ext_count.alloc(1);
        }
    }
    GridScratch& gscratch = lanes[0].gscratch;
    t_alloc = now_ms();
    DevBuf<double> src_stats(4);
    double* rm = d_rmse ? d_rmse : rmse_tmp.p;
    int32_t* nu = d_n_used ? d_n_used : nused_tmp.p;

    PCREG_CUDA(cudaMemsetAsync(frozen.p, 0, frozen.bytes(), st));
    PCREG_CUDA(cudaMemsetAsync(counters.p, 0, counters.bytes(), st));
    if (stop_iter.p) PCREG_CUDA(cudaMemsetAsync(stop_iter.p, 0xff, stop_iter.bytes(), st));      // -1: running
    if (ex_state.p) PCREG_CUDA(cudaMemsetAsync(ex_state.p, 0, ex_state.bytes(), st));
    transpose16_launch(d_T0_cm, Twork.p, nhyp, st);

    std::vector<EventPair> evs;
    std::vector<GridScratch::Mark> marks;
    size_t ev_cursor = 0;
    if (prof) { gscratch.timing = &marks; gscratch.ev_cursor = &ev_cursor; }
    auto ev_begin = [&](int kind) {
        if (!prof) return;
        EventPair e; e.kind = kind;
        e.a = pooled_event(ev_cursor++); e.b = pooled_event(ev_cursor++);
        PCREG_CUDA(cudaEventRecord(e.a, st));
        evs.push_back(e);
    };
    auto ev_end = [&]() { if (prof) PCREG_CUDA(cudaEventRecord(evs.back().b, st)); };

    // spatial sort of the source (skipped for very large clouds: the single-block sort is sized for <= 2^17)
    const bool sorted = ns >= 64 && ns <= (1 << 17);
    DevBuf<double> src_sorted(sorted ? (size_t)ns * 3 : 0), w_sorted(sorted && d_w ? (size_t)ns : 0);
    DevBuf<int32_t> sperm(sorted ? (size_t)ns : 0), sinv(sorted ? (size_t)ns : 0);
    if (sorted) {
        int npow2 = 1;
        while (npow2 < ns) npow2 <<= 1;
        DevBuf<unsigned long long> skeys((size_t)npow2);
        k_src_sort<<<1, 1024, 0, st>>>(d_src, d_w, ns, nullptr, ns, skeys.p, src_sorted.p, d_w ? w_sorted.p : nullptr, sperm.p, sinv.p);
        PCREG_LAUNCHED();
        PCREG_CUDA(cudaStreamSynchronize(st));      // skeys is released here
        d_src = src_sorted.p;
        if (d_w) d_w = w_sorted.p;
    }
    // plane-to-plane: the source normals normalised and checked on the device, in the order of the source arrays.  The flag is read
    // before any ICP kernel runs, so a bad normal never reaches them.
    DevBuf<double> snrm(gicp ? (size_t)ns * 3 : 0);
    if (gicp) {
        DevBuf<int> bad(1);
        int h_bad = 0;
        PCREG_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), st));
        k_src_normals<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(d_src_nrm, sorted ? sperm.p : nullptr, ns, nullptr, ns, snrm.p, bad.p);
        PCREG_LAUNCHED();
        PCREG_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        PCREG_CUDA(cudaStreamSynchronize(st));
        PCREG_REQUIRE(!h_bad, "icp: zero or non-finite source normal");
    }
    const double* snx = gicp ? snrm.p : nullptr;
    const double* sny = gicp ? snrm.p + ns : nullptr;
    const double* snz = gicp ? snrm.p + 2 * ns : nullptr;
    t_sorted = now_ms();
    const double* sx = d_src; const double* sy = d_src + ns; const double* sz = d_src + 2 * ns;
    if (fused) {
        // One launch for the whole batch: each block runs every pass of one hypothesis (icp_fused.cu).
        FusedArgs fa{};
        fa.g.g = m->grid; fa.g.md = m->md.p; fa.g.vox = m->vox;
        fa.sx = sx; fa.sy = sy; fa.sz = sz; fa.w_src = d_w; fa.ns = (int32_t)ns;
        for (int k = 0; k < 3; ++k) fa.pivot[k] = m->pivot[k];
        fa.T = Twork.p; fa.frozen = frozen.p; fa.rmse = rm; fa.n_used = nu;
        fa.rmse_hist = d_rmse_hist; fa.hist_stride = o.iters + 1;
        fa.idx_out = d_idx; fa.perm = sorted ? sperm.p : nullptr; fa.tie_order = sorted ? sinv.p : nullptr;
        fa.mode = o.mode; fa.k_frac = o.k_frac; fa.R_w = o.R_w; fa.thDist2 = o.thDist2; fa.reflection_fix = o.reflection_fix; fa.iters = o.iters;
        fa.counters = (prof && c.profiling_counters) ? counters.p : nullptr;
        fa.stop = rule; fa.n_iter = d_n_iter; fa.converged = d_converged; fa.nrm = nrm;
        fa.snx = snx; fa.sny = sny; fa.snz = snz; fa.gicp_eps = gicp_eps;
        if (ex) { fa.ex = *ex; fa.ex_cen = d_ex_cen; fa.n_extrap = d_n_extrap; }
        if (cov) fa.cov = *cov;
        ev_begin(0);
        icp_fused_launch(fa, nhyp, stop_mode, st);
        ev_end();
        transpose16_launch(Twork.p, d_T16_cm, nhyp, st);
        if (d_status) PCREG_CUDA(cudaMemcpyAsync(d_status, frozen.p, (size_t)nhyp * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        if (d_best) icp_argmin_launch(rm, nhyp, d_best, st);
        PCREG_CUDA(cudaStreamSynchronize(st));
        if (prof) {
            float ms = 0.f;
            PCREG_CUDA(cudaEventElapsedTime(&ms, evs[0].a, evs[0].b));
            unsigned long long hcnt[16] = {0};
            PCREG_CUDA(cudaMemcpy(hcnt, counters.p, sizeof hcnt, cudaMemcpyDeviceToHost));
            // with the tolerance stop a block runs as many passes as its hypothesis needs
            const double nq = (double)ns * (stop ? passes_run() : (double)nhyp * (double)(o.iters + 1));
            c.profile[0] = 1; c.profile[1] = ms; c.profile[2] = nq; c.profile[6] = nq;
            c.profile[11] = (double)hcnt[4]; c.profile[10] = nq - (double)hcnt[4];
            c.profile[13] = (double)hcnt[6]; c.profile[14] = (double)hcnt[7];
            c.profile[17] = ms; c.profile[20] = 1;
            c.profile[26] = 1.0; c.profile[27] = 1.0;
            // share of a block's cycles spent in each phase (clock64 of thread 0, summed over the blocks)
            const double tot = (double)hcnt[11] + (double)hcnt[12] + (double)hcnt[13] + (double)hcnt[14];
            for (int k = 0; k < 4; ++k) c.profile[28 + k] = tot > 0.0 ? (double)hcnt[11 + k] / tot : 0.0;
        }
        return;
    }
    k_src_stats<<<1, 1024, 0, st>>>(d_src, ns, src_stats.p);
    PCREG_LAUNCHED();
    if (use_lists) {
        static const double build_frac = [] { const char* e = getenv("PCREG_LIST_BUILD"); return e ? atof(e) : 1.5; }();
        for (int l = 0; l < nlanes; ++l) {
            Lane& L = lanes[l];
            CandView& cl = L.cl;
            cl.hdr = L.cl_hdr.p; cl.cnt = L.cl_cnt.p; cl.list = L.cl_list.p; cl.cap = list_cap;
            cl.ext = L.cl_ext.p; cl.ext_list = L.cl_ext_list.p; cl.ext_count = L.cl_ext_count.p; cl.ext_cap = ext_cap; cl.ext_slots = (int32_t)ext_slots;
            cl.gap_cells = (float)list_skin_cells;
            cl.skin = (double)cl.gap_cells * m->grid.cell * (1.0 - 1e-6);
            cl.build_max_delta = (float)(build_frac * cl.skin);
            cl.inv_level = (float)(255.0 / (2.0 * cl.skin));
        }
        PCREG_CUDA(cudaMemsetAsync(delta.p, 0x7f, delta.bytes(), st));      // "large" until the first update writes it
        if (lazy_trim) PCREG_CUDA(cudaMemsetAsync(skip_thr.p, 0x7f, skip_thr.bytes(), st));
    }
    if (nlanes > 1) {                                                       // fork: the lanes start after everything queued on st
        cudaEvent_t fork = pooled_event(ev_cursor++);
        PCREG_CUDA(cudaEventRecord(fork, st));
        for (int l = 0; l < nlanes; ++l) PCREG_CUDA(cudaStreamWaitEvent(lanes[l].st, fork, 0));
    }
    double nn_launches = 0, upd_launches = 0;
    for (int64_t base = 0; base < nhyp; base += hc * nlanes) {
        for (int l = 0; l < nlanes; ++l) {
            Lane& L = lanes[l];
            L.h0 = std::min(nhyp, base + l * hc);
            L.hn = std::min(hc, nhyp - L.h0);
            L.cur = L.idxA.p; L.prev = L.idxB.p; L.have_prev = false;
            if (use_lists && L.hn > 0) {
                PCREG_CUDA(cudaMemsetAsync(L.cl_cnt.p, 0xff, (size_t)L.hn * ns * sizeof(int2), L.st));        // -1: no list yet
                PCREG_CUDA(cudaMemsetAsync(L.cl_ext.p, 0xff, (size_t)L.hn * ns * sizeof(int32_t), L.st));     // -1: no extension slot
                PCREG_CUDA(cudaMemsetAsync(L.cl_ext_count.p, 0, sizeof(unsigned int), L.st));
                L.cl.delta = delta.p + L.h0;
            }
        }
        for (int it = 0; it <= o.iters; ++it) {
            const bool last = (it == o.iters);
            for (int l = 0; l < nlanes; ++l) {
                Lane& L = lanes[l];
                if (L.hn <= 0) continue;
                cudaStream_t ls = L.st;
                const int64_t h0 = L.h0, hn = L.hn;
                int32_t* out_idx = (last && d_idx && !sorted) ? d_idx + h0 * ns : L.cur;
                ev_begin(0);
                if (o.nn == PCREG_NN_BRUTE)
                    nn_brute_launch(m, sx, sy, sz, ns, Twork.p + h0 * 16, hn, L.have_prev ? L.prev : nullptr, out_idx, L.d2.p, L.scratch, ls);
                else
                    nn_grid_launch(m, sx, sy, sz, ns, Twork.p + h0 * 16, hn, L.have_prev ? L.prev : nullptr, out_idx, L.d2.p,
                                   (prof && c.profiling_counters) ? counters.p : nullptr, L.gscratch, use_lists ? &L.cl : nullptr, it >= 2,
                                   (lazy_trim && it >= 2 && !last) ? skip_thr.p + h0 : nullptr, ls,
                                   (stop && !last) ? stop_iter.p + h0 : nullptr);
                ev_end();
                nn_launches += 1;
                IcpUpdateArgs ua{};
                ua.md = m->md.p; ua.nrm = nrm;
                ua.snx = snx; ua.sny = sny; ua.snz = snz; ua.gicp_eps = gicp_eps;
                for (int k = 0; k < 3; ++k) ua.pivot[k] = m->pivot[k];
                ua.sx = sx; ua.sy = sy; ua.sz = sz; ua.w_src = d_w; ua.ns = ns;
                ua.T = Twork.p + h0 * 16; ua.idx = out_idx; ua.d2 = L.d2.p; ua.keys = L.keys.p;
                ua.tie_order = sorted ? sinv.p : nullptr;
                ua.delta = use_lists ? delta.p + h0 : nullptr;
                ua.skip_thr = lazy_trim ? skip_thr.p + h0 : nullptr;
                ua.src_stats = src_stats.p;
                ua.mode = o.mode; ua.k_frac = o.k_frac; ua.R_w = o.R_w; ua.thDist2 = o.thDist2; ua.reflection_fix = o.reflection_fix;
                ua.update = last ? 0 : 1;
                ua.frozen = frozen.p + h0; ua.rmse = rm + h0; ua.n_used = nu + h0;
                ua.rmse_hist = d_rmse_hist ? d_rmse_hist + h0 * (o.iters + 1) : nullptr;
                ua.hist_stride = o.iters + 1; ua.hist_col = it;
                if (stop) {
                    ua.stop_iter = stop_iter.p + h0; ua.stop_ring = stop_ring.p + h0 * 2 * ICP_STOP_WINDOW_MAX; ua.stop = rule;
                    ua.n_iter = d_n_iter ? d_n_iter + h0 : nullptr; ua.converged = d_converged ? d_converged + h0 : nullptr;
                }
                if (ex) {
                    ua.ex = *ex; ua.ex_state = ex_state.p + h0 * EXTRAP_STATE; ua.ex_cen = d_ex_cen;
                    ua.n_extrap = d_n_extrap ? d_n_extrap + h0 : nullptr;
                }
                if (cov) ua.cov = cov_out_at(*cov, h0);
                ev_begin(1);
                icp_update_launch(ua, hn, ls);
                ev_end();
                upd_launches += 1;
                if (last && d_idx && sorted) {
                    k_unpermute_idx<<<(unsigned)((hn * ns + 255) / 256), 256, 0, ls>>>(out_idx, sinv.p, ns, hn, d_idx + h0 * ns);
                    PCREG_LAUNCHED();
                }
                std::swap(L.cur, L.prev);       // what was just written becomes the warm start
                L.have_prev = true;
            }
        }
    }
    if (nlanes > 1) {                                                       // join
        for (int l = 0; l < nlanes; ++l) {
            cudaEvent_t done = pooled_event(ev_cursor++);
            PCREG_CUDA(cudaEventRecord(done, lanes[l].st));
            PCREG_CUDA(cudaStreamWaitEvent(st, done, 0));
        }
    }
    transpose16_launch(Twork.p, d_T16_cm, nhyp, st);
    if (d_status) PCREG_CUDA(cudaMemcpyAsync(d_status, frozen.p, (size_t)nhyp * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    if (d_best) icp_argmin_launch(rm, nhyp, d_best, st);

    // scratch is freed when this function returns: the stream must have drained
    t_enq = now_ms();
    PCREG_CUDA(cudaStreamSynchronize(st));
    if (dbg_host) fprintf(stderr, "[pcreg host] alloc %.2f  sort+sync %.2f  enqueue %.2f  drain %.2f ms\n", t_alloc - t_enter, t_sorted - t_alloc,
                          t_enq - t_sorted, now_ms() - t_enq);
    if (prof) {
        double nn_ms = 0, upd_ms = 0;
        for (auto& e : evs) {
            float ms = 0.f;
            PCREG_CUDA(cudaEventElapsedTime(&ms, e.a, e.b));
            (e.kind == 0 ? nn_ms : upd_ms) += ms;
            if (debug_times()) fprintf(stderr, "[pcreg] %s %.3f ms\n", e.kind == 0 ? "nn" : "update", ms);
        }
        unsigned long long hcnt[16] = {0};
        PCREG_CUDA(cudaMemcpy(hcnt, counters.p, sizeof hcnt, cudaMemcpyDeviceToHost));
        for (int k = 3; k < 10; ++k) c.profile[7 + k] = (double)hcnt[k];       // out[10..16]
        c.profile[23] = (double)hcnt[10];                                       // queries skipped by lazy trimming
        // per-kernel time of the grid path: the span from each mark to the next one of the same pass
        for (size_t k = 0; k + 1 < marks.size(); ++k) {
            if (marks[k].kind == 3) continue;
            float ms = 0.f;
            PCREG_CUDA(cudaEventElapsedTime(&ms, marks[k].ev, marks[k + 1].ev));
            c.profile[17 + marks[k].kind] += ms;
            c.profile[20 + marks[k].kind] += 1.0;
        }
        const double nq = (double)nhyp * (double)ns * (double)(o.iters + 1);
        // with the tolerance stop, the update kernel and the voxel-map NN kernel skip a stopped hypothesis until the final
        // pass; the brute-force and map-less grid NN kernels still search for it
        const double nq_run = stop ? (double)ns * passes_run() : nq;
        const bool vox_nn = o.nn == PCREG_NN_GRID && m->has_vox;
        c.profile[0] = nn_launches; c.profile[1] = nn_ms; c.profile[2] = vox_nn ? nq_run : nq;
        c.profile[3] = (o.nn == PCREG_NN_BRUTE) ? nq * (double)m->n : 0.0;
        c.profile[4] = upd_launches; c.profile[5] = upd_ms; c.profile[6] = nq_run;
        c.profile[7] = (double)hcnt[0]; c.profile[8] = (double)hcnt[1]; c.profile[9] = (double)hcnt[2];
        c.profile[26] = (o.nn == PCREG_NN_GRID && m->has_vox) ? 1.0 : 0.0;
    }
}

// ---- windowed calls (pcreg_icp_batch_windows{,_dev}) ----------------------------------------------------------------------
// Host-side layout of a windowed call: window w owns source rows src_off[w] .. src_off[w + 1] - 1 and hypotheses hyp_off[w] ..
// hyp_off[w + 1] - 1; its [H_w][ns_w] block of idx starts at idx_off[w].
struct WindowLayout {
    int64_t nwin = 0, nrows = 0, nhyp = 0, ns_max = 0;
    std::vector<int64_t> src_off, hyp_off, idx_off;
    WindowLayout(const int64_t* so, const int64_t* ho, int64_t nw) : nwin(nw), src_off(so, so + nw + 1), hyp_off(ho, ho + nw + 1), idx_off((size_t)nw + 1, 0) {
        for (int64_t w = 0; w < nw; ++w) {
            const int64_t ns = src_off[w + 1] - src_off[w];
            ns_max = std::max(ns_max, ns);
            idx_off[w + 1] = idx_off[w] + (hyp_off[w + 1] - hyp_off[w]) * ns;
        }
        nrows = src_off[nw]; nhyp = hyp_off[nw];
    }
    int64_t ns(int64_t w) const { return src_off[w + 1] - src_off[w]; }
    int64_t nh(int64_t w) const { return hyp_off[w + 1] - hyp_off[w]; }
    int64_t window_of(int64_t h) const {       // the window that holds hypothesis h
        return (int64_t)(std::upper_bound(hyp_off.begin(), hyp_off.end(), h) - hyp_off.begin()) - 1;
    }
    int64_t idx_at(int64_t h) const { const int64_t w = window_of(h); return idx_off[w] + (h - hyp_off[w]) * ns(w); }
};

// When a windowed call runs as one launch of the fused kernel.  The alternative is a loop over the windows through icp_run, each
// window at least an NN and an update launch per pass plus host synchronisations (DESIGN.md section 3.3 has the measurements).
static bool windows_use_fused(const pcreg_model* m, const WindowLayout& L, const pcreg_icp_opts& o, int stop, int metric) {
    if (!icp_fused_windows_fit(m, L.ns_max, o, stop, metric)) return false;
    if (const char* e = getenv("PCREG_FUSED")) { if (e[0] == '0') return false; if (e[0] == '1') return true; }
    int64_t busy = 0;                          // windows with hypotheses
    for (int64_t w = 0; w < L.nwin; ++w) busy += L.nh(w) > 0;
    return busy >= 2 || L.nhyp >= ctx().sm_count;
}

// One device: d_src column-major with column stride L.nrows (the windows' rows one after the other), d_w / d_src_nrm at the same
// rows, d_T0_cm / outputs indexed by hypothesis as in icp_run, d_idx in the ragged window-major layout, d_best [nwin] (relative).
static void icp_windows_run(const pcreg_model* m, const WindowLayout& L, const double* d_src, const double* d_w, const double* d_src_nrm,
                            const double* d_T0_cm, const pcreg_icp_opts& o, const pcreg_icp_stop* stop, int metric, double gicp_eps,
                            double* d_T16_cm, double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx, double* d_rmse_hist,
                            int64_t* d_best, int32_t* d_n_iter, int32_t* d_converged, cudaStream_t st,
                            const IcpExtrapRule* ex = nullptr, int32_t* d_n_extrap = nullptr, const IcpCovOut* cov = nullptr) {
    PCREG_REQUIRE(m && d_T16_cm && (L.nrows == 0 || d_src) && (L.nhyp == 0 || d_T0_cm), "icp windows: null pointer");
    const bool gicp = metric == ICP_M_GICP;
    const ModelPointD* nrm = metric != ICP_M_POINT ? m->nrm.p : nullptr;
    if (metric != ICP_M_POINT && !nrm) throw StateError{"icp: the point-to-plane and plane-to-plane metrics need model normals (pcreg_model_set_normals / pcreg_model_compute_normals)"};
    PCREG_REQUIRE(!gicp || d_src_nrm, "icp: the plane-to-plane metric needs source normals");
    PCREG_REQUIRE(o.iters >= 0, "icp: iters must be >= 0");
    PCREG_REQUIRE(o.mode >= PCREG_ICP_PLAIN && o.mode <= PCREG_ICP_WEIGHTED, "icp: bad mode");
    PCREG_REQUIRE(o.nn == PCREG_NN_BRUTE || o.nn == PCREG_NN_GRID, "icp: bad nn kind");
    if (o.nn == PCREG_NN_GRID) PCREG_REQUIRE(m->has_grid, "icp: grid NN requested but the model has no grid");
    Context& c = ctx();
    const bool prof = c.profiling;
    const int64_t nrows = L.nrows, nhyp = L.nhyp;
    DevBuf<int64_t> offs((size_t)(3 * L.nwin + 2));            // src_off [nwin + 1], hyp_off [nwin + 1], idx_off [nwin]
    int64_t* d_soff = offs.p; int64_t* d_hoff = offs.p + L.nwin + 1; int64_t* d_ioff = offs.p + 2 * (L.nwin + 1);
    PCREG_CUDA(cudaMemcpyAsync(d_soff, L.src_off.data(), (size_t)(L.nwin + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    PCREG_CUDA(cudaMemcpyAsync(d_hoff, L.hyp_off.data(), (size_t)(L.nwin + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    PCREG_CUDA(cudaMemcpyAsync(d_ioff, L.idx_off.data(), (size_t)L.nwin * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    // pose extrapolation: it runs with the caller's stop rule, or with one that never stops (a tolerance of 0 changes no bit)
    const pcreg_icp_stop never{0.0, 0.0, 1};
    if (ex && !stop) { stop = &never; d_n_iter = nullptr; d_converged = nullptr; }
    const int stop_mode = ex ? 2 : stop ? 1 : 0;
    // the source centroid of every window, from the caller's rows in their order (both paths read it)
    DevBuf<double> cen(ex ? (size_t)L.nwin * 3 : 0);
    if (ex) {
        k_src_centroid<<<(unsigned)L.nwin, 256, 0, st>>>(d_src, nrows, d_soff, cen.p);
        PCREG_LAUNCHED();
    }
    const bool fused = nhyp > 0 && windows_use_fused(m, L, o, stop_mode, metric);
    // plane-to-plane: every window's source normals normalised and checked before any ICP kernel runs (in the windows' sorted order
    // on the fused path; the loop normalises each window again inside icp_run, from the caller's rows)
    DevBuf<int32_t> sperm(fused ? (size_t)nrows : 0), sinv(fused ? (size_t)nrows : 0);
    DevBuf<double> src_sorted(fused ? (size_t)nrows * 3 : 0), w_sorted(fused && d_w ? (size_t)nrows : 0);
    if (fused && nrows > 0) {
        DevBuf<unsigned long long> skeys((size_t)nrows * 2);
        k_src_sort<<<(unsigned)L.nwin, 1024, 0, st>>>(d_src, d_w, nrows, d_soff, 0, skeys.p, src_sorted.p, d_w ? w_sorted.p : nullptr, sperm.p, sinv.p);
        PCREG_LAUNCHED();
        PCREG_CUDA(cudaStreamSynchronize(st));      // skeys is released here
    }
    DevBuf<double> snrm(gicp ? (size_t)nrows * 3 : 0);
    if (gicp && nrows > 0) {
        DevBuf<int> bad(1);
        int h_bad = 0;
        PCREG_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), st));
        for (int64_t w0 = 0; w0 < L.nwin; w0 += 65535) {         // grid.y: at most 65 535 windows per launch
            const dim3 grid((unsigned)((L.ns_max + 255) / 256), (unsigned)std::min<int64_t>(65535, L.nwin - w0));
            k_src_normals<<<grid, 256, 0, st>>>(d_src_nrm, fused ? sperm.p : nullptr, nrows, d_soff + w0, 0, snrm.p, bad.p);
            PCREG_LAUNCHED();
        }
        PCREG_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        PCREG_CUDA(cudaStreamSynchronize(st));
        PCREG_REQUIRE(!h_bad, "icp: zero or non-finite source normal");
    }
    if (d_best) PCREG_CUDA(cudaMemsetAsync(d_best, 0xff, (size_t)L.nwin * sizeof(int64_t), st));     // -1: no hypothesis
    if (!fused) {
        // one icp_run per window with hypotheses, on its rows copied out of the concatenation and its slices of every output
        double prof_sum[32] = {0};
        const size_t hs = (size_t)o.iters + 1;
        for (int64_t w = 0; w < L.nwin; ++w) {
            const int64_t ns = L.ns(w), nh = L.nh(w), r0 = L.src_off[w], h0 = L.hyp_off[w];
            if (nh == 0) continue;
            DevBuf<double> src_w((size_t)ns * 3), nrm_w(gicp ? (size_t)ns * 3 : 0);
            for (int a = 0; a < 3; ++a) {
                PCREG_CUDA(cudaMemcpyAsync(src_w.p + a * ns, d_src + a * nrows + r0, (size_t)ns * sizeof(double), cudaMemcpyDeviceToDevice, st));
                if (gicp) PCREG_CUDA(cudaMemcpyAsync(nrm_w.p + a * ns, d_src_nrm + a * nrows + r0, (size_t)ns * sizeof(double), cudaMemcpyDeviceToDevice, st));
            }
            const IcpCovOut cw = cov ? cov_out_at(*cov, h0) : IcpCovOut{};
            icp_run(m, src_w.p, ns, d_w ? d_w + r0 : nullptr, d_T0_cm + h0 * 16, nh, o, d_T16_cm + h0 * 16, d_rmse ? d_rmse + h0 : nullptr,
                    d_n_used ? d_n_used + h0 : nullptr, d_status ? d_status + h0 : nullptr, d_idx ? d_idx + L.idx_off[w] : nullptr,
                    d_rmse_hist ? d_rmse_hist + h0 * hs : nullptr, d_best ? d_best + w : nullptr, st, stop,
                    d_n_iter ? d_n_iter + h0 : nullptr, d_converged ? d_converged + h0 : nullptr, metric, gicp ? nrm_w.p : nullptr, gicp_eps,
                    ex, ex ? cen.p + 3 * w : nullptr, d_n_extrap ? d_n_extrap + h0 : nullptr, cov ? &cw : nullptr);
            if (prof) {
                for (int k = 0; k < 26; ++k) prof_sum[k] += c.profile[k];
                prof_sum[26] = std::max(prof_sum[26], c.profile[26]);
            }
        }
        PCREG_CUDA(cudaStreamSynchronize(st));
        for (int k = 0; k < 32; ++k) c.profile[k] = prof_sum[k];       // out[27] = 0: the loop ran
        return;
    }
    for (int i = 0; i < 32; ++i) c.profile[i] = 0.0;
    // one launch of the fused kernel for every hypothesis of every window (k_icp_fused<*, *, *, true>)
    DevBuf<double> Twork((size_t)nhyp * 16);
    DevBuf<int32_t> frozen((size_t)nhyp);
    DevBuf<double> rmse_tmp(d_rmse ? 0 : (size_t)nhyp);
    DevBuf<int32_t> nused_tmp(d_n_used ? 0 : (size_t)nhyp);
    DevBuf<unsigned long long> counters(16);
    DevBuf<int32_t> n_iter_tmp(stop && prof && !d_n_iter ? (size_t)nhyp : 0);
    if (n_iter_tmp.p) d_n_iter = n_iter_tmp.p;
    double* rm = d_rmse ? d_rmse : rmse_tmp.p;
    PCREG_CUDA(cudaMemsetAsync(frozen.p, 0, frozen.bytes(), st));
    PCREG_CUDA(cudaMemsetAsync(counters.p, 0, counters.bytes(), st));
    transpose16_launch(d_T0_cm, Twork.p, nhyp, st);
    FusedWinArgs fa{};
    fa.g.g = m->grid; fa.g.md = m->md.p; fa.g.vox = m->vox;
    fa.sx = src_sorted.p; fa.sy = src_sorted.p + nrows; fa.sz = src_sorted.p + 2 * nrows; fa.w_src = d_w ? w_sorted.p : nullptr;
    fa.ns = (int32_t)L.ns_max;
    for (int k = 0; k < 3; ++k) fa.pivot[k] = m->pivot[k];
    fa.T = Twork.p; fa.frozen = frozen.p; fa.rmse = rm; fa.n_used = d_n_used ? d_n_used : nused_tmp.p;
    fa.rmse_hist = d_rmse_hist; fa.hist_stride = o.iters + 1;
    fa.idx_out = d_idx; fa.perm = sperm.p; fa.tie_order = sinv.p;
    fa.mode = o.mode; fa.k_frac = o.k_frac; fa.R_w = o.R_w; fa.thDist2 = o.thDist2; fa.reflection_fix = o.reflection_fix; fa.iters = o.iters;
    fa.counters = (prof && c.profiling_counters) ? counters.p : nullptr;
    if (stop) { fa.stop.tol_t = stop->tol_t; fa.stop.tol_r_deg = stop->tol_r_deg; fa.stop.window = stop->window; }
    fa.n_iter = d_n_iter; fa.converged = d_converged; fa.nrm = nrm;
    fa.snx = gicp ? snrm.p : nullptr; fa.sny = gicp ? snrm.p + nrows : nullptr; fa.snz = gicp ? snrm.p + 2 * nrows : nullptr; fa.gicp_eps = gicp_eps;
    fa.win_src = d_soff; fa.win_hyp = d_hoff; fa.win_idx = d_ioff; fa.nwin = (int32_t)L.nwin;
    if (ex) { fa.ex = *ex; fa.ex_cen = cen.p; fa.n_extrap = d_n_extrap; }
    if (cov) fa.cov = *cov;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (prof) { e0 = pooled_event(0); e1 = pooled_event(1); PCREG_CUDA(cudaEventRecord(e0, st)); }
    icp_fused_windows_launch(fa, nhyp, stop_mode, st);
    if (prof) PCREG_CUDA(cudaEventRecord(e1, st));
    transpose16_launch(Twork.p, d_T16_cm, nhyp, st);
    if (d_status) PCREG_CUDA(cudaMemcpyAsync(d_status, frozen.p, (size_t)nhyp * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    if (d_best) icp_argmin_launch(rm, nhyp, d_best, st, d_hoff, L.nwin);
    PCREG_CUDA(cudaStreamSynchronize(st));
    if (prof) {
        float ms = 0.f;
        PCREG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        unsigned long long hcnt[16] = {0};
        PCREG_CUDA(cudaMemcpy(hcnt, counters.p, sizeof hcnt, cudaMemcpyDeviceToHost));
        // queries of the passes each hypothesis ran (with the tolerance stop: n_iter + 1, one more after a freeze)
        double nq = 0.0;
        if (stop) {
            std::vector<int32_t> ni((size_t)nhyp), fz((size_t)nhyp);
            PCREG_CUDA(cudaMemcpy(ni.data(), d_n_iter, ni.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
            PCREG_CUDA(cudaMemcpy(fz.data(), frozen.p, fz.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
            for (int64_t h = 0; h < nhyp; ++h) nq += (double)L.ns(L.window_of(h)) * ((double)ni[h] + 1.0 + (double)fz[h]);
        } else {
            for (int64_t w = 0; w < L.nwin; ++w) nq += (double)L.nh(w) * (double)L.ns(w) * (double)(o.iters + 1);
        }
        c.profile[0] = 1; c.profile[1] = ms; c.profile[2] = nq; c.profile[6] = nq;
        c.profile[11] = (double)hcnt[4]; c.profile[10] = nq - (double)hcnt[4];
        c.profile[13] = (double)hcnt[6]; c.profile[14] = (double)hcnt[7];
        c.profile[17] = ms; c.profile[20] = 1;
        c.profile[26] = 1.0; c.profile[27] = 1.0;
        const double tot = (double)hcnt[11] + (double)hcnt[12] + (double)hcnt[13] + (double)hcnt[14];
        for (int k = 0; k < 4; ++k) c.profile[28 + k] = tot > 0.0 ? (double)hcnt[11 + k] / tot : 0.0;
    }
}

// host column-major (float or double, ld) -> contiguous double column-major ns x 3
static std::vector<double> to_double_cm(const void* p, int is_double, int64_t n, int64_t ld) {
    std::vector<double> out((size_t)n * 3);
    for (int a = 0; a < 3; ++a)
        for (int64_t i = 0; i < n; ++i)
            out[(size_t)a * n + i] = is_double ? ((const double*)p)[a * ld + i] : (double)((const float*)p)[a * ld + i];
    return out;
}

}  // namespace pcreg

using namespace pcreg;

extern "C" {

void pcreg_icp_opts_default(pcreg_icp_opts* o) {
    if (!o) return;
    o->mode = PCREG_ICP_PLAIN; o->iters = 50; o->k_frac = 0.85; o->R_w = 3.5; o->thDist2 = 0.0;
    o->nn = PCREG_NN_BRUTE; o->reflection_fix = 0;
}

void pcreg_icp_stop_default(pcreg_icp_stop* s) {
    if (!s) return;
    s->tol_t = 0.01; s->tol_r_deg = 0.5; s->window = 3;
}

static void check_stop(const pcreg_icp_stop* s) {
    PCREG_REQUIRE(s, "icp stop: null pointer");
    PCREG_REQUIRE(s->tol_t >= 0.0 && s->tol_r_deg >= 0.0, "icp stop: tolerances must be >= 0 (NaN is rejected; +inf disables one)");
    PCREG_REQUIRE(s->window >= 1 && s->window <= ICP_STOP_WINDOW_MAX, "icp stop: window must be in [1, 16]");
}

int pcreg_icp_batch_dev(const pcreg_model* m, const double* d_src, int64_t ns, const double* d_w_src,
                        const double* d_T0_16, int64_t nhyp, const pcreg_icp_opts* opts, double* d_T16,
                        double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx, double* d_rmse_hist,
                        int64_t* d_best, void* stream) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(opts, "pcreg_icp_batch_dev: opts is null");
    PCREG_CUDA(cudaSetDevice(ctx().device));
    icp_run(m, d_src, ns, d_w_src, d_T0_16, nhyp, *opts, d_T16, d_rmse, d_n_used, d_status, d_idx, d_rmse_hist,
            d_best, (cudaStream_t)stream);
    return PCREG_OK;
    PCREG_API_END
}

int pcreg_icp_batch_stop_dev(const pcreg_model* m, const double* d_src, int64_t ns, const double* d_w_src,
                             const double* d_T0_16, int64_t nhyp, const pcreg_icp_opts* opts, const pcreg_icp_stop* stop,
                             double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx,
                             double* d_rmse_hist, int64_t* d_best, int32_t* d_n_iter, int32_t* d_converged, void* stream) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(opts, "pcreg_icp_batch_stop_dev: opts is null");
    check_stop(stop);
    PCREG_CUDA(cudaSetDevice(ctx().device));
    icp_run(m, d_src, ns, d_w_src, d_T0_16, nhyp, *opts, d_T16, d_rmse, d_n_used, d_status, d_idx, d_rmse_hist,
            d_best, (cudaStream_t)stream, stop, d_n_iter, d_converged);
    return PCREG_OK;
    PCREG_API_END
}

// One device's share [h0, h0 + hn) of a host-buffer batch, on the calling thread's slot.  Output pointers are the caller's
// arrays (whole batch); every copy lands in its own contiguous slice, which is the "all-gather" of SURVEY.md section 8e.
static void icp_batch_host_slice(const pcreg_model* m, const std::vector<double>& hs, int64_t ns, const double* w_src,
                                 const double* T0_16, int64_t h0, int64_t hn, const pcreg_icp_opts& o, double* T16, double* rmse,
                                 int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                                 const pcreg_icp_stop* stop, int32_t* n_iter, int32_t* converged, int metric,
                                 const std::vector<double>& hnrm, double gicp_eps) {
    PCREG_CUDA(cudaSetDevice(ctx().device));
    cudaStream_t st = 0;
    DevBuf<double> d_src((size_t)ns * 3), d_w(w_src ? (size_t)ns : 0), d_T0((size_t)hn * 16), d_T((size_t)hn * 16);
    DevBuf<double> d_nrm(hnrm.size());                  // plane-to-plane: the source normals, copied to every device as the source is
    DevBuf<double> d_rmse((size_t)hn), d_hist(rmse_hist ? (size_t)hn * (o.iters + 1) : 0);
    DevBuf<int32_t> d_nu((size_t)hn), d_st((size_t)hn), d_idx(idx ? (size_t)hn * ns : 0);
    DevBuf<int32_t> d_nit(n_iter ? (size_t)hn : 0), d_conv(converged ? (size_t)hn : 0);
    PCREG_CUDA(cudaMemcpyAsync(d_src.p, hs.data(), d_src.bytes(), cudaMemcpyHostToDevice, st));
    if (w_src) PCREG_CUDA(cudaMemcpyAsync(d_w.p, w_src, d_w.bytes(), cudaMemcpyHostToDevice, st));
    if (d_nrm.p) PCREG_CUDA(cudaMemcpyAsync(d_nrm.p, hnrm.data(), d_nrm.bytes(), cudaMemcpyHostToDevice, st));
    PCREG_CUDA(cudaMemcpyAsync(d_T0.p, T0_16 + h0 * 16, d_T0.bytes(), cudaMemcpyHostToDevice, st));
    icp_run(m, d_src.p, ns, w_src ? d_w.p : nullptr, d_T0.p, hn, o, d_T.p, d_rmse.p, d_nu.p, d_st.p,
            idx ? d_idx.p : nullptr, rmse_hist ? d_hist.p : nullptr, nullptr, st, stop, d_nit.p, d_conv.p, metric, d_nrm.p, gicp_eps);
    PCREG_CUDA(cudaMemcpyAsync(T16 + h0 * 16, d_T.p, d_T.bytes(), cudaMemcpyDeviceToHost, st));
    PCREG_CUDA(cudaMemcpyAsync(rmse + h0, d_rmse.p, d_rmse.bytes(), cudaMemcpyDeviceToHost, st));
    if (n_used) PCREG_CUDA(cudaMemcpyAsync(n_used + h0, d_nu.p, d_nu.bytes(), cudaMemcpyDeviceToHost, st));
    if (status) PCREG_CUDA(cudaMemcpyAsync(status + h0, d_st.p, d_st.bytes(), cudaMemcpyDeviceToHost, st));
    if (idx) PCREG_CUDA(cudaMemcpyAsync(idx + h0 * ns, d_idx.p, d_idx.bytes(), cudaMemcpyDeviceToHost, st));
    if (rmse_hist) PCREG_CUDA(cudaMemcpyAsync(rmse_hist + h0 * (o.iters + 1), d_hist.p, d_hist.bytes(), cudaMemcpyDeviceToHost, st));
    if (n_iter) PCREG_CUDA(cudaMemcpyAsync(n_iter + h0, d_nit.p, d_nit.bytes(), cudaMemcpyDeviceToHost, st));
    if (converged) PCREG_CUDA(cudaMemcpyAsync(converged + h0, d_conv.p, d_conv.bytes(), cudaMemcpyDeviceToHost, st));
    PCREG_CUDA(cudaStreamSynchronize(st));
}

// pcreg_icp_batch, pcreg_icp_batch_stop (stop != nullptr), pcreg_icp_batch_metric and pcreg_icp_batch_gicp (src_nrm: the source
// normals, same type and ld as src)
static int icp_batch_host(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld, const double* w_src,
                          const double* T0_16, int64_t nhyp, const pcreg_icp_opts* opts, double* T16, double* rmse,
                          int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist, int64_t* best,
                          const pcreg_icp_stop* stop, int32_t* n_iter, int32_t* converged, int metric = ICP_M_POINT,
                          const void* src_nrm = nullptr, double gicp_eps = 0.0) {
    require_init();
    PCREG_REQUIRE(m && src && T0_16 && T16 && opts, "pcreg_icp_batch: null pointer");
    PCREG_REQUIRE(ns >= 1 && ld >= ns && nhyp >= 1, "pcreg_icp_batch: bad sizes");
    const std::vector<double> hs = to_double_cm(src, is_double, ns, ld);
    const std::vector<double> hnrm = src_nrm ? to_double_cm(src_nrm, is_double, ns, ld) : std::vector<double>();
    std::vector<double> rmse_tmp(rmse ? 0 : (size_t)nhyp);
    double* rm = rmse ? rmse : rmse_tmp.data();
    // Hypotheses are independent (the reference runs them under parfor: slideMatchingWindow_v2.m:178, completeExperiment.m:265):
    // contiguous shares, one host thread + stream per selected device, the model replicated by pcreg_model_create; no
    // communication until the result records land in the caller's arrays.
    const int nd = (int)std::min<int64_t>(num_slots(), std::min<int64_t>(nhyp, (int64_t)m->replicas.size() + 1));
    const int64_t per = (nhyp + nd - 1) / nd;
    std::vector<int> rc((size_t)nd, PCREG_OK);
    std::vector<std::thread> workers;
    for (int k = 1; k < nd; ++k) {
        const int64_t h0 = k * per, hn = std::min(per, nhyp - h0);
        if (hn <= 0) continue;
        workers.emplace_back([&, k, h0, hn]() {
            rc[k] = guarded([&]() { use_slot(k); icp_batch_host_slice(m->on_slot(k), hs, ns, w_src, T0_16, h0, hn, *opts, T16, rm, n_used, status, idx, rmse_hist,
                                                                 stop, n_iter, converged, metric, hnrm, gicp_eps); });
        });
    }
    rc[0] = guarded([&]() { use_slot(0); icp_batch_host_slice(m, hs, ns, w_src, T0_16, 0, std::min(per, nhyp), *opts, T16, rm, n_used, status, idx, rmse_hist,
                                                         stop, n_iter, converged, metric, hnrm, gicp_eps); });
    for (auto& w : workers) w.join();
    use_slot(0);
    for (int k = 0; k < nd; ++k) if (rc[k] != PCREG_OK) return rc[k];
    if (best) {                                           // first-index arg-min, NaN never wins (ransac.m:69-73 tie rule mirrored)
        int64_t bi = -1;
        for (int64_t h = 0; h < nhyp; ++h) if (rm[h] == rm[h] && (bi < 0 || rm[h] < rm[bi])) bi = h;
        *best = bi;
    }
    return PCREG_OK;
}

int pcreg_icp_batch(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld, const double* w_src,
                    const double* T0_16, int64_t nhyp, const pcreg_icp_opts* opts, double* T16, double* rmse,
                    int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist, int64_t* best) {
    PCREG_API_BEGIN
    return icp_batch_host(m, src, is_double, ns, ld, w_src, T0_16, nhyp, opts, T16, rmse, n_used, status, idx, rmse_hist, best,
                          nullptr, nullptr, nullptr);
    PCREG_API_END
}

int pcreg_icp_batch_stop(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld, const double* w_src,
                         const double* T0_16, int64_t nhyp, const pcreg_icp_opts* opts, const pcreg_icp_stop* stop,
                         double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                         int64_t* best, int32_t* n_iter, int32_t* converged) {
    PCREG_API_BEGIN
    check_stop(stop);
    return icp_batch_host(m, src, is_double, ns, ld, w_src, T0_16, nhyp, opts, T16, rmse, n_used, status, idx, rmse_hist, best,
                          stop, n_iter, converged);
    PCREG_API_END
}

static void check_metric(int metric, const pcreg_icp_stop* stop) {
    PCREG_REQUIRE(metric == PCREG_ICP_POINT_TO_POINT || metric == PCREG_ICP_POINT_TO_PLANE, "icp: unknown metric");
    if (stop) check_stop(stop);
}

int pcreg_icp_batch_metric(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld, const double* w_src,
                           const double* T0_16, int64_t nhyp, const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                           double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                           int64_t* best, int32_t* n_iter, int32_t* converged) {
    PCREG_API_BEGIN
    check_metric(metric, stop);
    return icp_batch_host(m, src, is_double, ns, ld, w_src, T0_16, nhyp, opts, T16, rmse, n_used, status, idx, rmse_hist, best,
                          stop, stop ? n_iter : nullptr, stop ? converged : nullptr, metric);
    PCREG_API_END
}

int pcreg_icp_batch_metric_dev(const pcreg_model* m, const double* d_src, int64_t ns, const double* d_w_src,
                               const double* d_T0_16, int64_t nhyp, const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                               double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx,
                               double* d_rmse_hist, int64_t* d_best, int32_t* d_n_iter, int32_t* d_converged, void* stream) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(opts, "pcreg_icp_batch_metric_dev: opts is null");
    check_metric(metric, stop);
    PCREG_CUDA(cudaSetDevice(ctx().device));
    icp_run(m, d_src, ns, d_w_src, d_T0_16, nhyp, *opts, d_T16, d_rmse, d_n_used, d_status, d_idx, d_rmse_hist,
            d_best, (cudaStream_t)stream, stop, stop ? d_n_iter : nullptr, stop ? d_converged : nullptr, metric);
    return PCREG_OK;
    PCREG_API_END
}

static void check_gicp(const void* src_nrm, double eps, const pcreg_icp_stop* stop) {
    PCREG_REQUIRE(src_nrm, "pcreg_icp_batch_gicp: the source normals are null");
    PCREG_REQUIRE(std::isfinite(eps) && eps > 0.0 && eps <= 1.0, "pcreg_icp_batch_gicp: eps must be finite and in (0, 1]");
    if (stop) check_stop(stop);
}

int pcreg_icp_batch_gicp(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld, const double* w_src,
                         const void* src_nrm, double eps, const double* T0_16, int64_t nhyp, const pcreg_icp_opts* opts,
                         const pcreg_icp_stop* stop, double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx,
                         double* rmse_hist, int64_t* best, int32_t* n_iter, int32_t* converged) {
    PCREG_API_BEGIN
    check_gicp(src_nrm, eps, stop);
    return icp_batch_host(m, src, is_double, ns, ld, w_src, T0_16, nhyp, opts, T16, rmse, n_used, status, idx, rmse_hist, best,
                          stop, stop ? n_iter : nullptr, stop ? converged : nullptr, ICP_M_GICP, src_nrm, eps);
    PCREG_API_END
}

int pcreg_icp_batch_gicp_dev(const pcreg_model* m, const double* d_src, int64_t ns, const double* d_w_src, const double* d_src_nrm,
                             double eps, const double* d_T0_16, int64_t nhyp, const pcreg_icp_opts* opts, const pcreg_icp_stop* stop,
                             double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx,
                             double* d_rmse_hist, int64_t* d_best, int32_t* d_n_iter, int32_t* d_converged, void* stream) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(opts, "pcreg_icp_batch_gicp_dev: opts is null");
    check_gicp(d_src_nrm, eps, stop);
    PCREG_CUDA(cudaSetDevice(ctx().device));
    icp_run(m, d_src, ns, d_w_src, d_T0_16, nhyp, *opts, d_T16, d_rmse, d_n_used, d_status, d_idx, d_rmse_hist,
            d_best, (cudaStream_t)stream, stop, stop ? d_n_iter : nullptr, stop ? d_converged : nullptr, ICP_M_GICP, d_src_nrm, eps);
    return PCREG_OK;
    PCREG_API_END
}

static void check_windows(const pcreg_model* m, const int64_t* src_off, const int64_t* hyp_off, int64_t nwin, const pcreg_icp_opts* opts,
                               int metric, const void* src_nrm, double eps, const pcreg_icp_stop* stop) {
    PCREG_REQUIRE(m && opts, "pcreg_icp_batch_windows: null pointer");
    PCREG_REQUIRE(nwin >= 1, "icp windows: need nwin >= 1");
    PCREG_REQUIRE(src_off && hyp_off, "icp windows: null offsets");
    PCREG_REQUIRE(src_off[0] == 0 && hyp_off[0] == 0, "icp windows: offsets must start at 0");
    for (int64_t w = 0; w < nwin; ++w) {
        PCREG_REQUIRE(src_off[w + 1] >= src_off[w] && hyp_off[w + 1] >= hyp_off[w], "icp windows: decreasing offsets");
        PCREG_REQUIRE(hyp_off[w + 1] == hyp_off[w] || src_off[w + 1] > src_off[w], "icp windows: a window with hypotheses has no source rows");
        PCREG_REQUIRE(src_off[w + 1] - src_off[w] < ((int64_t)1 << 31), "icp windows: a window holds at most 2^31 - 1 source rows");
    }
    PCREG_REQUIRE(metric >= PCREG_ICP_POINT_TO_POINT && metric <= PCREG_ICP_PLANE_TO_PLANE, "icp: unknown metric");
    if (metric == PCREG_ICP_PLANE_TO_PLANE) check_gicp(src_nrm, eps, nullptr);
    if (stop) check_stop(stop);
    if (metric != PCREG_ICP_POINT_TO_POINT && !m->nrm.p)
        throw StateError{"icp: the point-to-plane and plane-to-plane metrics need model normals (pcreg_model_set_normals / pcreg_model_compute_normals)"};
}

// Host outputs and inputs of pcreg_icp_covariance (the covariance pass; its status goes to the call's status array)
struct CovHost {
    double ref[3];
    const double* targets; int64_t ntarget;     // [3][ntarget] column-major or null
    double* cov; double* info; double* sigma2; double* tre;
};

// One device's share [h0, h1) of a windowed host call: the windows it touches (a share may start or end inside a window), their rows
// and rebased offsets; every output lands in its own slice of the caller's arrays.
static void icp_windows_host_slice(const pcreg_model* m, const WindowLayout& L, const std::vector<double>& hs, const double* w_src,
                                   const std::vector<double>& hnrm, const double* T0_16, int64_t h0, int64_t h1, const pcreg_icp_opts& o,
                                   const pcreg_icp_stop* stop, int metric, double eps, double* T16, double* rmse, int32_t* n_used,
                                   int32_t* status, int32_t* idx, double* rmse_hist, int32_t* n_iter, int32_t* converged,
                                   const IcpExtrapRule* ex, int32_t* n_extrap, const CovHost* cv) {
    PCREG_CUDA(cudaSetDevice(ctx().device));
    cudaStream_t st = 0;
    const int64_t wa = L.window_of(h0), wb = L.window_of(h1 - 1), nw = wb - wa + 1;
    const int64_t ra = L.src_off[wa], nr = L.src_off[wb + 1] - ra, hn = h1 - h0;
    std::vector<int64_t> so((size_t)nw + 1), ho((size_t)nw + 1);
    for (int64_t k = 0; k <= nw; ++k) {
        so[k] = L.src_off[wa + k] - ra;
        ho[k] = std::min(std::max(L.hyp_off[wa + k], h0), h1) - h0;
    }
    const WindowLayout S(so.data(), ho.data(), nw);
    const int64_t i0 = L.idx_at(h0), ni = S.idx_off[nw];
    DevBuf<double> d_src((size_t)nr * 3), d_w(w_src ? (size_t)nr : 0), d_nrm(hnrm.empty() ? 0 : (size_t)nr * 3);
    DevBuf<double> d_T0((size_t)hn * 16), d_T((size_t)hn * 16), d_rmse((size_t)hn), d_hist(rmse_hist ? (size_t)hn * (o.iters + 1) : 0);
    DevBuf<int32_t> d_nu((size_t)hn), d_st((size_t)hn), d_idx(idx ? (size_t)ni : 0);
    DevBuf<int32_t> d_nit(n_iter ? (size_t)hn : 0), d_conv(converged ? (size_t)hn : 0), d_nex(n_extrap ? (size_t)hn : 0);
    for (int a = 0; a < 3; ++a) {
        PCREG_CUDA(cudaMemcpyAsync(d_src.p + a * nr, hs.data() + a * L.nrows + ra, (size_t)nr * sizeof(double), cudaMemcpyHostToDevice, st));
        if (d_nrm.p) PCREG_CUDA(cudaMemcpyAsync(d_nrm.p + a * nr, hnrm.data() + a * L.nrows + ra, (size_t)nr * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    if (w_src) PCREG_CUDA(cudaMemcpyAsync(d_w.p, w_src + ra, d_w.bytes(), cudaMemcpyHostToDevice, st));
    PCREG_CUDA(cudaMemcpyAsync(d_T0.p, T0_16 + h0 * 16, d_T0.bytes(), cudaMemcpyHostToDevice, st));
    const int64_t nt = cv ? cv->ntarget : 0;
    DevBuf<double> c_cov(cv ? (size_t)hn * 36 : 0), c_info(cv && cv->info ? (size_t)hn * 36 : 0), c_sig(cv ? (size_t)hn : 0);
    DevBuf<double> c_tre(cv && cv->tre ? (size_t)(hn * nt) : 0), c_tg((size_t)nt * 3);
    IcpCovOut co{};
    if (cv) {
        co.cov = c_cov.p; co.info = c_info.p; co.sigma2 = c_sig.p; co.status = d_st.p; co.tre = c_tre.p;
        co.targets = c_tg.p; co.ntarget = (int32_t)nt;
        for (int k = 0; k < 3; ++k) co.ref[k] = cv->ref[k];
        if (nt) PCREG_CUDA(cudaMemcpyAsync(c_tg.p, cv->targets, c_tg.bytes(), cudaMemcpyHostToDevice, st));
    }
    icp_windows_run(m, S, d_src.p, d_w.p, d_nrm.p, d_T0.p, o, stop, metric, eps, d_T.p, d_rmse.p, d_nu.p, cv ? nullptr : d_st.p, d_idx.p,
                    d_hist.p, nullptr, d_nit.p, d_conv.p, st, ex, d_nex.p, cv ? &co : nullptr);
    if (cv) {
        PCREG_CUDA(cudaMemcpyAsync(cv->cov + h0 * 36, c_cov.p, c_cov.bytes(), cudaMemcpyDeviceToHost, st));
        if (cv->info) PCREG_CUDA(cudaMemcpyAsync(cv->info + h0 * 36, c_info.p, c_info.bytes(), cudaMemcpyDeviceToHost, st));
        PCREG_CUDA(cudaMemcpyAsync(cv->sigma2 + h0, c_sig.p, c_sig.bytes(), cudaMemcpyDeviceToHost, st));
        if (c_tre.p) PCREG_CUDA(cudaMemcpyAsync(cv->tre + h0 * nt, c_tre.p, c_tre.bytes(), cudaMemcpyDeviceToHost, st));
    }
    PCREG_CUDA(cudaMemcpyAsync(T16 + h0 * 16, d_T.p, d_T.bytes(), cudaMemcpyDeviceToHost, st));
    PCREG_CUDA(cudaMemcpyAsync(rmse + h0, d_rmse.p, d_rmse.bytes(), cudaMemcpyDeviceToHost, st));
    if (n_used) PCREG_CUDA(cudaMemcpyAsync(n_used + h0, d_nu.p, d_nu.bytes(), cudaMemcpyDeviceToHost, st));
    if (status) PCREG_CUDA(cudaMemcpyAsync(status + h0, d_st.p, d_st.bytes(), cudaMemcpyDeviceToHost, st));
    if (idx) PCREG_CUDA(cudaMemcpyAsync(idx + i0, d_idx.p, d_idx.bytes(), cudaMemcpyDeviceToHost, st));
    if (rmse_hist) PCREG_CUDA(cudaMemcpyAsync(rmse_hist + h0 * (o.iters + 1), d_hist.p, d_hist.bytes(), cudaMemcpyDeviceToHost, st));
    if (n_iter) PCREG_CUDA(cudaMemcpyAsync(n_iter + h0, d_nit.p, d_nit.bytes(), cudaMemcpyDeviceToHost, st));
    if (converged) PCREG_CUDA(cudaMemcpyAsync(converged + h0, d_conv.p, d_conv.bytes(), cudaMemcpyDeviceToHost, st));
    if (n_extrap) PCREG_CUDA(cudaMemcpyAsync(n_extrap + h0, d_nex.p, d_nex.bytes(), cudaMemcpyDeviceToHost, st));
    PCREG_CUDA(cudaStreamSynchronize(st));
}

// pcreg_icp_batch_windows and pcreg_icp_batch_extrap (ex != nullptr) after the argument checks
static int icp_windows_host(const pcreg_model* m, const void* src, int is_double, int64_t ld, const int64_t* src_offsets,
                            const double* w_src, const void* src_nrm, double gicp_eps, const int64_t* hyp_offsets, int64_t nwin,
                            const double* T0_16, const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                            double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                            int64_t* best, int32_t* n_iter, int32_t* converged, const IcpExtrapRule* ex, int32_t* n_extrap,
                            const CovHost* cv = nullptr) {
    const WindowLayout L(src_offsets, hyp_offsets, nwin);
    PCREG_REQUIRE((L.nrows == 0 || src) && (L.nhyp == 0 || (T0_16 && T16)) && ld >= L.nrows, "pcreg_icp_batch_windows: null pointer or bad ld");
    const bool gicp = metric == PCREG_ICP_PLANE_TO_PLANE;
    const std::vector<double> hs = to_double_cm(src, is_double, L.nrows, ld);
    const std::vector<double> hnrm = gicp ? to_double_cm(src_nrm, is_double, L.nrows, ld) : std::vector<double>();
    for (size_t i = 0; i < (size_t)L.nrows && gicp; ++i) {    // every window's normals, also those of windows no device runs
        const double x = hnrm[i], y = hnrm[L.nrows + i], z = hnrm[2 * L.nrows + i];
        const double n = std::sqrt((x * x + y * y) + z * z);
        PCREG_REQUIRE(std::isfinite(n) && n > 0.0, "icp: zero or non-finite source normal");
    }
    if (!stop) { n_iter = nullptr; converged = nullptr; }
    std::vector<double> rmse_tmp(rmse ? 0 : (size_t)L.nhyp);
    double* rm = rmse ? rmse : rmse_tmp.data();
    // contiguous shares of the hypotheses, one host thread + stream per selected device, as icp_batch_host
    const int nd = (int)std::min<int64_t>(num_slots(), std::min<int64_t>(L.nhyp, (int64_t)m->replicas.size() + 1));
    if (nd >= 1) {
        const int64_t per = (L.nhyp + nd - 1) / nd;
        std::vector<int> rc((size_t)nd, PCREG_OK);
        std::vector<std::thread> workers;
        auto run = [&](int k) {
            const int64_t h0 = k * per, h1 = std::min(L.nhyp, h0 + per);
            if (h1 <= h0) return;
            rc[k] = guarded([&]() { use_slot(k); icp_windows_host_slice(m->on_slot(k), L, hs, w_src, hnrm, T0_16, h0, h1, *opts, stop, metric, gicp_eps,
                                                                      T16, rm, n_used, status, idx, rmse_hist, n_iter, converged, ex, n_extrap,
                                                                      cv); });
        };
        for (int k = 1; k < nd; ++k) workers.emplace_back(run, k);
        run(0);
        for (auto& w : workers) w.join();
        use_slot(0);
        for (int k = 0; k < nd; ++k) if (rc[k] != PCREG_OK) return rc[k];
    }
    if (best) {                                           // per window: first-index arg-min, NaN never wins, relative to the window
        for (int64_t w = 0; w < nwin; ++w) {
            int64_t bi = -1;
            for (int64_t h = L.hyp_off[w]; h < L.hyp_off[w + 1]; ++h)
                if (rm[h] == rm[h] && (bi < 0 || rm[h] < rm[L.hyp_off[w] + bi])) bi = h - L.hyp_off[w];
            best[w] = bi;
        }
    }
    return PCREG_OK;
}

int pcreg_icp_batch_windows(const pcreg_model* m, const void* src, int is_double, int64_t ld, const int64_t* src_offsets,
                            const double* w_src, const void* src_nrm, double gicp_eps, const int64_t* hyp_offsets, int64_t nwin,
                            const double* T0_16, const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                            double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                            int64_t* best, int32_t* n_iter, int32_t* converged) {
    PCREG_API_BEGIN
    require_init();
    check_windows(m, src_offsets, hyp_offsets, nwin, opts, metric, src_nrm, gicp_eps, stop);
    return icp_windows_host(m, src, is_double, ld, src_offsets, w_src, src_nrm, gicp_eps, hyp_offsets, nwin, T0_16, opts, metric, stop, T16,
                            rmse, n_used, status, idx, rmse_hist, best, n_iter, converged, nullptr, nullptr);
    PCREG_API_END
}

int pcreg_icp_batch_windows_dev(const pcreg_model* m, const double* d_src, const int64_t* src_offsets, const double* d_w_src,
                                const double* d_src_nrm, double gicp_eps, const int64_t* hyp_offsets, int64_t nwin, const double* d_T0_16,
                                const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop, double* d_T16, double* d_rmse,
                                int32_t* d_n_used, int32_t* d_status, int32_t* d_idx, double* d_rmse_hist, int64_t* d_best,
                                int32_t* d_n_iter, int32_t* d_converged, void* stream) {
    PCREG_API_BEGIN
    require_init();
    check_windows(m, src_offsets, hyp_offsets, nwin, opts, metric, d_src_nrm, gicp_eps, stop);
    PCREG_CUDA(cudaSetDevice(ctx().device));
    const WindowLayout L(src_offsets, hyp_offsets, nwin);
    icp_windows_run(m, L, d_src, d_w_src, d_src_nrm, d_T0_16, *opts, stop, metric, gicp_eps, d_T16, d_rmse, d_n_used, d_status, d_idx,
                    d_rmse_hist, d_best, stop ? d_n_iter : nullptr, stop ? d_converged : nullptr, (cudaStream_t)stream);
    return PCREG_OK;
    PCREG_API_END
}

void pcreg_icp_extrap_default(pcreg_icp_extrap* e) {
    if (!e) return;
    e->angle_deg = 10.0; e->vmax_scale = 25.0;
}

static void check_extrap(const pcreg_icp_extrap* e) {
    if (!e) return;
    PCREG_REQUIRE(e->angle_deg > 0.0 && e->angle_deg <= 180.0, "icp extrap: angle_deg must be in (0, 180]");
    PCREG_REQUIRE(std::isfinite(e->vmax_scale) && e->vmax_scale > 0.0, "icp extrap: vmax_scale must be finite and > 0");
}

int pcreg_icp_batch_extrap(const pcreg_model* m, const void* src, int is_double, int64_t ld, const int64_t* src_offsets,
                           const double* w_src, const int64_t* hyp_offsets, int64_t nwin, const double* T0_16,
                           const pcreg_icp_opts* opts, const pcreg_icp_stop* stop, const pcreg_icp_extrap* ex,
                           double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                           int64_t* best, int32_t* n_iter, int32_t* converged, int32_t* n_extrap) {
    PCREG_API_BEGIN
    require_init();
    check_windows(m, src_offsets, hyp_offsets, nwin, opts, PCREG_ICP_POINT_TO_POINT, nullptr, 0.0, stop);
    check_extrap(ex);
    const IcpExtrapRule rule = ex ? IcpExtrapRule{ex->angle_deg, ex->vmax_scale} : IcpExtrapRule{};
    return icp_windows_host(m, src, is_double, ld, src_offsets, w_src, nullptr, 0.0, hyp_offsets, nwin, T0_16, opts, PCREG_ICP_POINT_TO_POINT,
                            stop, T16, rmse, n_used, status, idx, rmse_hist, best, n_iter, converged, ex ? &rule : nullptr,
                            ex ? n_extrap : nullptr);
    PCREG_API_END
}

int pcreg_icp_batch_extrap_dev(const pcreg_model* m, const double* d_src, const int64_t* src_offsets, const double* d_w_src,
                               const int64_t* hyp_offsets, int64_t nwin, const double* d_T0_16, const pcreg_icp_opts* opts,
                               const pcreg_icp_stop* stop, const pcreg_icp_extrap* ex, double* d_T16, double* d_rmse,
                               int32_t* d_n_used, int32_t* d_status, int32_t* d_idx, double* d_rmse_hist, int64_t* d_best,
                               int32_t* d_n_iter, int32_t* d_converged, int32_t* d_n_extrap, void* stream) {
    PCREG_API_BEGIN
    require_init();
    check_windows(m, src_offsets, hyp_offsets, nwin, opts, PCREG_ICP_POINT_TO_POINT, nullptr, 0.0, stop);
    check_extrap(ex);
    PCREG_CUDA(cudaSetDevice(ctx().device));
    const WindowLayout L(src_offsets, hyp_offsets, nwin);
    const IcpExtrapRule rule = ex ? IcpExtrapRule{ex->angle_deg, ex->vmax_scale} : IcpExtrapRule{};
    icp_windows_run(m, L, d_src, d_w_src, nullptr, d_T0_16, *opts, stop, PCREG_ICP_POINT_TO_POINT, 0.0, d_T16, d_rmse, d_n_used, d_status,
                    d_idx, d_rmse_hist, d_best, stop ? d_n_iter : nullptr, stop ? d_converged : nullptr, (cudaStream_t)stream,
                    ex ? &rule : nullptr, ex ? d_n_extrap : nullptr);
    return PCREG_OK;
    PCREG_API_END
}

// pcreg_icp_covariance{,_dev}: the checks of the windows entry (metric 1: model normals needed), then the pass's own
static pcreg_icp_opts check_cov(const pcreg_model* m, const int64_t* src_off, const int64_t* hyp_off, int64_t nwin, const pcreg_icp_opts* opts,
                                const double* ref, const double* targets, int64_t ntarget, const void* cov36, const void* sigma2,
                                const void* status, CovHost& cv) {
    check_windows(m, src_off, hyp_off, nwin, opts, PCREG_ICP_POINT_TO_PLANE, nullptr, 0.0, nullptr);
    PCREG_REQUIRE(cov36 && sigma2 && status, "pcreg_icp_covariance: cov36, sigma2 and status are required");
    PCREG_REQUIRE(ntarget >= 0 && ntarget < ((int64_t)1 << 31) && (ntarget == 0 || targets), "pcreg_icp_covariance: bad targets");
    for (int k = 0; k < 3; ++k) {
        cv.ref[k] = ref ? ref[k] : 0.0;
        PCREG_REQUIRE(std::isfinite(cv.ref[k]), "pcreg_icp_covariance: ref must be finite");
    }
    for (int64_t i = 0; i < 3 * ntarget; ++i) PCREG_REQUIRE(std::isfinite(targets[i]), "pcreg_icp_covariance: targets must be finite");
    cv.targets = ntarget ? targets : nullptr; cv.ntarget = ntarget;
    pcreg_icp_opts o = *opts;
    o.iters = 0;
    o.reflection_fix = 0;
    return o;
}

int pcreg_icp_covariance(const pcreg_model* m, const void* src, int is_double, int64_t ld, const int64_t* src_offsets,
                         const double* w_src, const int64_t* hyp_offsets, int64_t nwin, const double* T16, const pcreg_icp_opts* opts,
                         const double* ref, const double* targets, int64_t ntarget, double* cov36, double* info36, double* sigma2,
                         double* rmse, int32_t* n_used, int32_t* status, double* tre) {
    PCREG_API_BEGIN
    require_init();
    CovHost cv{};
    const pcreg_icp_opts o = check_cov(m, src_offsets, hyp_offsets, nwin, opts, ref, targets, ntarget, cov36, sigma2, status, cv);
    cv.cov = cov36; cv.info = info36; cv.sigma2 = sigma2; cv.tre = ntarget ? tre : nullptr;
    std::vector<double> T_out((size_t)std::max<int64_t>(1, hyp_offsets[nwin]) * 16);      // the pass leaves the poses alone
    return icp_windows_host(m, src, is_double, ld, src_offsets, w_src, nullptr, 0.0, hyp_offsets, nwin, T16, &o, ICP_M_COV, nullptr,
                            T_out.data(), rmse, n_used, status, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, &cv);
    PCREG_API_END
}

int pcreg_icp_covariance_dev(const pcreg_model* m, const double* d_src, const int64_t* src_offsets, const double* d_w_src,
                             const int64_t* hyp_offsets, int64_t nwin, const double* d_T16, const pcreg_icp_opts* opts, const double* ref,
                             const double* targets, int64_t ntarget, double* d_cov36, double* d_info36, double* d_sigma2, double* d_rmse,
                             int32_t* d_n_used, int32_t* d_status, double* d_tre, void* stream) {
    PCREG_API_BEGIN
    require_init();
    CovHost cv{};
    const pcreg_icp_opts o = check_cov(m, src_offsets, hyp_offsets, nwin, opts, ref, targets, ntarget, d_cov36, d_sigma2, d_status, cv);
    PCREG_CUDA(cudaSetDevice(ctx().device));
    cudaStream_t st = (cudaStream_t)stream;
    const WindowLayout L(src_offsets, hyp_offsets, nwin);
    DevBuf<double> T_out((size_t)std::max<int64_t>(1, L.nhyp) * 16), d_tg((size_t)ntarget * 3);
    if (ntarget) PCREG_CUDA(cudaMemcpyAsync(d_tg.p, targets, d_tg.bytes(), cudaMemcpyHostToDevice, st));
    IcpCovOut co{};
    co.cov = d_cov36; co.info = d_info36; co.sigma2 = d_sigma2; co.status = d_status; co.tre = ntarget ? d_tre : nullptr;
    co.targets = d_tg.p; co.ntarget = (int32_t)ntarget;
    for (int k = 0; k < 3; ++k) co.ref[k] = cv.ref[k];
    icp_windows_run(m, L, d_src, d_w_src, nullptr, d_T16, o, nullptr, ICP_M_COV, 0.0, T_out.p, d_rmse, d_n_used, nullptr, nullptr, nullptr,
                    nullptr, nullptr, nullptr, st, nullptr, nullptr, &co);
    return PCREG_OK;
    PCREG_API_END
}

int pcreg_quick_tf(const void* pts, int is_double, int64_t n, int64_t ld, const double* T16, int mode, void* out, int64_t ld_out) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(pts && T16 && out, "pcreg_quick_tf: null pointer");
    PCREG_REQUIRE(n >= 1 && ld >= n && ld_out >= n, "pcreg_quick_tf: bad sizes");
    PCREG_REQUIRE(mode >= PCREG_TF_FORWARD && mode <= PCREG_TF_MRDIVIDE, "pcreg_quick_tf: bad mode");
    // math layout M[r][c] from the column-major record
    double M[4][4];
    for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) M[r][c] = T16[c * 4 + r];
    Pose16 P{};
    if (mode == PCREG_TF_FORWARD) {
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) P.t[r * 4 + c] = M[r][c];
    } else if (mode == PCREG_TF_INVERT) {               // invertTF.m:5-7: [R' 0; -t R' 1]
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) P.t[r * 4 + c] = M[c][r];
        for (int c = 0; c < 3; ++c) P.t[12 + c] = -(M[3][0] * M[c][0] + M[3][1] * M[c][1] + M[3][2] * M[c][2]);
        P.t[3] = P.t[7] = P.t[11] = 0.0; P.t[15] = 1.0;
    } else {                                            // [p 1] / T: the general inverse (AutoAlignPointclouds.m:8), Gauss-Jordan with pivoting
        double A[4][8];
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) { A[r][c] = M[r][c]; A[r][4 + c] = r == c ? 1.0 : 0.0; }
        for (int k = 0; k < 4; ++k) {
            int piv = k;
            for (int r = k + 1; r < 4; ++r) if (fabs(A[r][k]) > fabs(A[piv][k])) piv = r;
            PCREG_REQUIRE(A[piv][k] != 0.0, "pcreg_quick_tf: singular transform");
            if (piv != k) for (int c = 0; c < 8; ++c) std::swap(A[k][c], A[piv][c]);
            const double d = A[k][k];
            for (int c = 0; c < 8; ++c) A[k][c] /= d;
            for (int r = 0; r < 4; ++r) if (r != k) { const double f = A[r][k]; for (int c = 0; c < 8; ++c) A[r][c] -= f * A[k][c]; }
        }
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) P.t[r * 4 + c] = A[r][4 + c];
    }
    PCREG_CUDA(cudaSetDevice(ctx().device));
    cudaStream_t st = 0;
    const size_t el = is_double ? 8 : 4;
    DevBuf<unsigned char> d_in((size_t)n * 3 * el), d_out((size_t)n * 3 * el);
    for (int a = 0; a < 3; ++a)
        PCREG_CUDA(cudaMemcpyAsync(d_in.p + (size_t)a * n * el, (const unsigned char*)pts + (size_t)a * ld * el, (size_t)n * el, cudaMemcpyHostToDevice, st));
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (is_double) k_quick_tf<double><<<blocks, 256, 0, st>>>((const double*)d_in.p, n, n, (double*)d_out.p, n, P);
    else           k_quick_tf<float><<<blocks, 256, 0, st>>>((const float*)d_in.p, n, n, (float*)d_out.p, n, P);
    PCREG_LAUNCHED();
    for (int a = 0; a < 3; ++a)
        PCREG_CUDA(cudaMemcpyAsync((unsigned char*)out + (size_t)a * ld_out * el, d_out.p + (size_t)a * n * el, (size_t)n * el, cudaMemcpyDeviceToHost, st));
    PCREG_CUDA(cudaStreamSynchronize(st));
    return PCREG_OK;
    PCREG_API_END
}

int pcreg_nn_search(const pcreg_model* m, const void* q, int is_double, int64_t nq, int64_t ld, int nn_kind,
                    int32_t* idx, double* d2) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(m && q && idx, "pcreg_nn_search: null pointer");
    PCREG_REQUIRE(nq >= 1 && ld >= nq, "pcreg_nn_search: bad sizes");
    PCREG_REQUIRE(nn_kind == PCREG_NN_BRUTE || nn_kind == PCREG_NN_GRID, "pcreg_nn_search: bad nn kind");
    PCREG_CUDA(cudaSetDevice(ctx().device));
    cudaStream_t st = 0;
    Context& c = ctx();
    for (int i = 0; i < 32; ++i) c.profile[i] = 0.0;
    std::vector<double> hq = to_double_cm(q, is_double, nq, ld);
    const double I16[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    DevBuf<double> d_q((size_t)nq * 3), d_T(16), d_d2((size_t)nq);
    DevBuf<int32_t> d_idx((size_t)nq);
    DevBuf<unsigned long long> counters(16);
    NNScratch scratch;
    GridScratch gscratch;
    PCREG_CUDA(cudaMemcpyAsync(d_q.p, hq.data(), d_q.bytes(), cudaMemcpyHostToDevice, st));
    PCREG_CUDA(cudaMemcpyAsync(d_T.p, I16, sizeof I16, cudaMemcpyHostToDevice, st));
    PCREG_CUDA(cudaMemsetAsync(counters.p, 0, counters.bytes(), st));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (c.profiling) { PCREG_CUDA(cudaEventCreate(&e0)); PCREG_CUDA(cudaEventCreate(&e1)); PCREG_CUDA(cudaEventRecord(e0, st)); }
    if (nn_kind == PCREG_NN_BRUTE)
        nn_brute_launch(m, d_q.p, d_q.p + nq, d_q.p + 2 * nq, nq, d_T.p, 1, nullptr, d_idx.p, d_d2.p, scratch, st);
    else
        nn_grid_launch(m, d_q.p, d_q.p + nq, d_q.p + 2 * nq, nq, d_T.p, 1, nullptr, d_idx.p, d_d2.p,
                       (c.profiling && c.profiling_counters) ? counters.p : nullptr, gscratch, nullptr, false, nullptr, st);
    if (c.profiling) PCREG_CUDA(cudaEventRecord(e1, st));
    PCREG_CUDA(cudaMemcpyAsync(idx, d_idx.p, d_idx.bytes(), cudaMemcpyDeviceToHost, st));
    if (d2) PCREG_CUDA(cudaMemcpyAsync(d2, d_d2.p, d_d2.bytes(), cudaMemcpyDeviceToHost, st));
    PCREG_CUDA(cudaStreamSynchronize(st));
    if (c.profiling) {
        float ms = 0.f;
        PCREG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        unsigned long long hcnt[16] = {0};
        PCREG_CUDA(cudaMemcpy(hcnt, counters.p, sizeof hcnt, cudaMemcpyDeviceToHost));
        for (int k = 3; k < 10; ++k) c.profile[7 + k] = (double)hcnt[k];
        c.profile[0] = 1; c.profile[1] = ms; c.profile[2] = (double)nq;
        c.profile[3] = nn_kind == PCREG_NN_BRUTE ? (double)nq * (double)m->n : 0.0;
        c.profile[7] = (double)hcnt[0]; c.profile[8] = (double)hcnt[1]; c.profile[9] = (double)hcnt[2];
        c.profile[26] = (nn_kind == PCREG_NN_GRID && m->has_vox) ? 1.0 : 0.0;
    }
    return PCREG_OK;
    PCREG_API_END
}

}  // extern "C"
