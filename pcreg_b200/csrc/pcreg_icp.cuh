// pcreg_icp.cuh -- the per-correspondence arithmetic of one ICP pass, shared by k_icp_update (icp.cu, one launch per pass)
// and the fused per-hypothesis kernel (icp_fused.cu) so that both produce the same bits:
//   rejection   squared-distance compare (ransac.m:49: dist < thDist keeps)
//   weights     w = max(R_w - r, 0) (AlignPoints_weighted.m:16-18), times the caller's w_src
//   17 sums     estimateTransform.m:41-58 as one pass (sum w, sum w q, sum w m, sum w q m', sum w d^2), relative to a pivot
//   pose update estimateTransform.m:60-71 (kabsch_from_sums) and T <- T * dT
#pragma once
#include "pcreg_internal.h"
#include "pcreg_dev.cuh"
#include "pcreg_math.cuh"

namespace pcreg {

// ICP passes sum over the correspondences of one hypothesis with this many threads (thread t takes i = t, t + N, ...);
// both kernels use the same count so that their fixed-tree reductions agree bit for bit
#ifdef UPD_THREADS_OVERRIDE
constexpr int UPD_THREADS = UPD_THREADS_OVERRIDE;
#else
constexpr int UPD_THREADS = 256;       // fused kernel, C3 step, same-session A/B (threads x blocks per SM, registers): 256 x 2 (128) 38.9 ms;
#endif                                 // 224 x 2: 40.0; 320 x 2 (96): 40.4; 192 x 2 (168): 42.0; 384 x 2 (80, spills): 44.4; 512 x 1 (128): 45.0;
                                       // 160 x 2: 47.7; 512 x 2 (64): 48-53; 256 x 3 (80): 51.5; 128 x 2 (212, no spills): 53.7
#ifndef FUSED_MIN_BLOCKS
#define FUSED_MIN_BLOCKS 2
#endif

__device__ __forceinline__ void icp_accumulate(double (&s)[KABSCH_NSUMS], double w, double d, double qx, double qy, double qz,
                                               const ModelPointD& m, double px, double py, double pz) {
    const double q0 = qx - px, q1 = qy - py, q2 = qz - pz;
    const double m0 = m.x - px, m1 = m.y - py, m2 = m.z - pz;
    const double wq0 = w * q0, wq1 = w * q1, wq2 = w * q2;
    s[0] += w;
    s[1] += wq0; s[2] += wq1; s[3] += wq2;
    s[4] += w * m0; s[5] += w * m1; s[6] += w * m2;
    s[7] += wq0 * m0; s[8] += wq0 * m1; s[9] += wq0 * m2;
    s[10] += wq1 * m0; s[11] += wq1 * m1; s[12] += wq1 * m2;
    s[13] += wq2 * m0; s[14] += wq2 * m1; s[15] += wq2 * m2;
    s[16] += w * d;
}

// Thread 0 of a hypothesis after the block reduction: rigid fit from the sums (with the ICP rank rule of kabsch_from_sums) and
// T <- T * dT.  Returns false (pose left
// alone, hypothesis to be frozen) with fewer than 3 usable correspondences.  Tc: current pose (row-major), Tn: new pose.
__device__ __forceinline__ bool icp_pose_update(const double (&s)[KABSCH_NSUMS], long long n_used, const double* pivot, bool reflection_fix,
                                                const double* Tc, double* Tn) {
    const double sw = s[0];
    if (n_used < 3 || !(sw > 0.0)) return false;
    KabschSums ks;
    ks.sw = sw;
    for (int k = 0; k < 3; ++k) { ks.sq[k] = s[1 + k]; ks.sm[k] = s[4 + k]; }
    for (int k = 0; k < 9; ++k) ks.sqm[k] = s[7 + k];
    ks.swd2 = s[16];
    double dT[16];
    kabsch_from_sums(ks, pivot, pivot, reflection_fix, dT, true);      // rank <= 2: the proper solution (ICP_RANK2_TAU)
    mul4(Tc, dT, Tn);
    return true;
}

// out-of-line copy for the kernels' hot loops' sake: one thread per hypothesis runs it, its SVD must not claim their registers
__device__ __noinline__ static bool icp_pose_update_call(const double (&s)[KABSCH_NSUMS], long long n_used, const double* pivot,
                                                         bool reflection_fix, const double* Tc, double* Tn) {
    return icp_pose_update(s, n_used, pivot, reflection_fix, Tc, Tn);
}

// Point-to-plane metric (PCREG_ICP_POINT_TO_PLANE): with q~ = q - p, m~ = m - p and the model normal n of the correspondence,
// a = (q~ x n, n), b = (m~ - q~) . n; the 29 sums (pcreg_math.cuh: PLANE_NSUMS) are sw, A = sum w a a' (upper triangle),
// g = sum w a b and sum w d^2.  The rmse stays Euclidean: s[PLANE_NSUMS - 1] is sum w d^2 as s[16] of the 17 sums.
__device__ __forceinline__ void icp_accumulate_plane(double (&s)[PLANE_NSUMS], double w, double d, double qx, double qy, double qz,
                                                     const ModelPointD& m, const ModelPointD& n, double px, double py, double pz) {
    const double q0 = qx - px, q1 = qy - py, q2 = qz - pz;
    const double b = ((m.x - px) - q0) * n.x + ((m.y - py) - q1) * n.y + ((m.z - pz) - q2) * n.z;
    const double a[6] = {q1 * n.z - q2 * n.y, q2 * n.x - q0 * n.z, q0 * n.y - q1 * n.x, n.x, n.y, n.z};
    s[0] += w;
    int k = 1;
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        const double wa = w * a[r];
#pragma unroll
        for (int c = r; c < 6; ++c) s[k++] += wa * a[c];
        s[22 + r] += wa * b;
    }
    s[28] += w * d;
}

// Thread 0 after the block reduction: x = (omega, tau) from A x = g, dR = Rodrigues(omega)', dT = [dR 0; p - p dR + tau, 1] and
// T <- T * dT.  Returns false (pose left alone, hypothesis to be frozen) with fewer than 6 usable correspondences, no weight
// or a pivot of the LDL' factorisation at or below 1e-12 max A_kk.
__device__ __forceinline__ bool icp_pose_update_plane(const double (&s)[PLANE_NSUMS], long long n_used, const double* pivot,
                                                      const double* Tc, double* Tn) {
    if (n_used < 6 || !(s[0] > 0.0)) return false;
    double x[6];
    if (!ldlt6_solve(s + 1, s + 22, x)) return false;
    double R[9];
    rodrigues(x, R);
    double dT[16];
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) dT[r * 4 + c] = R[c * 3 + r];
        dT[r * 4 + 3] = 0.0;
    }
    for (int c = 0; c < 3; ++c)
        dT[12 + c] = (pivot[c] - (pivot[0] * dT[0 * 4 + c] + pivot[1] * dT[1 * 4 + c] + pivot[2] * dT[2 * 4 + c])) + x[3 + c];
    dT[15] = 1.0;
    mul4(Tc, dT, Tn);
    return true;
}

// out of line for the same reason as icp_pose_update_call
__device__ __noinline__ static bool icp_pose_update_plane_call(const double (&s)[PLANE_NSUMS], long long n_used, const double* pivot,
                                                               const double* Tc, double* Tn) {
    return icp_pose_update_plane(s, n_used, pivot, Tc, Tn);
}

// Plane-to-plane metric (pcreg_icp_batch_gicp): sn = the source normal of the correspondence's source point, carried by the
// current pose Ts (row-major, row-vector: n_q = n_s R); the arithmetic is gicp_accumulate (pcreg_math.cuh), which both kernels call
// in the same thread order.
__device__ __forceinline__ void icp_accumulate_gicp(double (&s)[PLANE_NSUMS], double w, double d, double qx, double qy, double qz,
                                                    const ModelPointD& m, const ModelPointD& n, double snx, double sny, double snz,
                                                    const double* Ts, double eps, double px, double py, double pz) {
    const double qt[3] = {qx - px, qy - py, qz - pz}, mt[3] = {m.x - px, m.y - py, m.z - pz};
    const double nm[3] = {n.x, n.y, n.z};
    double nq[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) nq[c] = snx * Ts[0 * 4 + c] + sny * Ts[1 * 4 + c] + snz * Ts[2 * 4 + c];
    gicp_accumulate(s, w, d, qt, mt, nq, nm, eps);
}

// Covariance pass (pcreg_icp_covariance): the point-to-plane accumulation of A in the same order, with sum w b^2 in the first slot
// of g (s[COV_SUM_B2]) instead of g; s[23..27] stay zero.
__device__ __forceinline__ void icp_accumulate_cov(double (&s)[PLANE_NSUMS], double w, double d, double qx, double qy, double qz,
                                                   const ModelPointD& m, const ModelPointD& n, double px, double py, double pz) {
    const double q0 = qx - px, q1 = qy - py, q2 = qz - pz;
    const double b = ((m.x - px) - q0) * n.x + ((m.y - py) - q1) * n.y + ((m.z - pz) - q2) * n.z;
    const double a[6] = {q1 * n.z - q2 * n.y, q2 * n.x - q0 * n.z, q0 * n.y - q1 * n.x, n.x, n.y, n.z};
    s[0] += w;
    int k = 1;
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        const double wa = w * a[r];
#pragma unroll
        for (int c = r; c < 6; ++c) s[k++] += wa * a[c];
    }
    s[COV_SUM_B2] += (w * b) * b;
    s[28] += w * d;
}

// Thread 0's part of the covariance outputs of hypothesis h; cov goes to sh[0..35] as well.  Out of line: one thread runs it.
__device__ __noinline__ static void icp_cov_thread0(const IcpCovOut& o, const double* s, long long n_used, const double* pivot, int64_t h,
                                                    double* sh) {
    double cov[36];
    const int st = pose_cov_from_sums(s, n_used, pivot, o.ref, cov, o.info ? o.info + h * 36 : nullptr, o.sigma2 + h);
    o.status[h] = st;
    for (int k = 0; k < 36; ++k) { o.cov[h * 36 + k] = cov[k]; sh[k] = cov[k]; }
}

// Every thread of the block, after the block reduction (s: the reduced sums, valid in every thread; sh: >= 36 doubles of free shared
// memory): the covariance outputs of hypothesis h, then tre over the targets (thread t: targets t, t + blockDim.x, ...).
__device__ __forceinline__ void icp_cov_write(const IcpCovOut& o, const double (&s)[PLANE_NSUMS], long long n_used, const double* pivot,
                                              int64_t h, double* sh) {
    if (threadIdx.x == 0) icp_cov_thread0(o, s, n_used, pivot, h, sh);
    __syncthreads();
    if (o.tre) {
        for (int k = threadIdx.x; k < o.ntarget; k += blockDim.x) {
            const double x[3] = {o.targets[k], o.targets[o.ntarget + k], o.targets[2 * (int64_t)o.ntarget + k]};
            o.tre[h * o.ntarget + k] = pose_cov_tre(sh, o.ref, x);
        }
    }
    __syncthreads();
}

// ICP metrics of the kernels' METRIC template parameter: 0 point-to-point (17 sums, Kabsch), 1 point-to-plane and 2 plane-to-plane
// (29 sums, the LDL' step), 3 the covariance pass (29 sums, no update: pcreg_icp_covariance); the last sum is sum w d^2 in all of them
constexpr int ICP_M_POINT = 0, ICP_M_PLANE = 1, ICP_M_GICP = 2, ICP_M_COV = 3;
template <int METRIC> constexpr int icp_nsums = METRIC != ICP_M_POINT ? PLANE_NSUMS : KABSCH_NSUMS;
template <int METRIC>
__device__ __forceinline__ bool icp_pose_update_m(const double (&s)[icp_nsums<METRIC>], long long n_used, const double* pivot,
                                                  bool reflection_fix, const double* Tc, double* Tn) {
    if constexpr (METRIC != ICP_M_POINT) return icp_pose_update_plane(s, n_used, pivot, Tc, Tn);
    else return icp_pose_update(s, n_used, pivot, reflection_fix, Tc, Tn);
}

// Tolerance stop (pcreg_icp_stop, include/pcreg.h).  Update u (1-based) took Tc = T_{u-1} to Tn = T_u = T_{u-1} dT.  Its motion
//   dt_u = |t_u - t_{u-1}|                                   (translation rows)
//   dr_u = atan2(|v|, (trace dR - 1) / 2) in degrees,  dR = R_{u-1}' R_u,  v = (dR32 - dR23, dR13 - dR31, dR21 - dR12) / 2
// goes to slot (u-1) % window of the ring (dt in ring[0..15], dr in ring[16..31]).  Once u >= window, returns true when the
// means of the last `window` updates (left-to-right FP64 sums over u-window+1 .. u, divided by window) are both strictly below
// their tolerances.  Both ICP paths call this one function, so the fused and the per-pass kernels stop at the same update.
__device__ __noinline__ static bool icp_stop_update(const IcpStopRule& r, const double* Tc, const double* Tn, int u, double* ring) {
    double dR[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            dR[i * 3 + j] = Tc[0 * 4 + i] * Tn[0 * 4 + j] + Tc[1 * 4 + i] * Tn[1 * 4 + j] + Tc[2 * 4 + i] * Tn[2 * 4 + j];
    const double v0 = 0.5 * (dR[7] - dR[5]), v1 = 0.5 * (dR[2] - dR[6]), v2 = 0.5 * (dR[3] - dR[1]);
    const double c = 0.5 * (dR[0] + dR[4] + dR[8] - 1.0);
    const double dr = atan2(sqrt(v0 * v0 + v1 * v1 + v2 * v2), c) * (180.0 / 3.14159265358979323846);
    const double x = Tn[12] - Tc[12], y = Tn[13] - Tc[13], z = Tn[14] - Tc[14];
    const double dt = sqrt(x * x + y * y + z * z);
    const int w = r.window;
    ring[(u - 1) % w] = dt;
    ring[ICP_STOP_WINDOW_MAX + (u - 1) % w] = dr;
    if (u < w) return false;
    double st = 0.0, sr = 0.0;
    for (int k = u - w; k < u; ++k) { st += ring[k % w]; sr += ring[ICP_STOP_WINDOW_MAX + k % w]; }
    return st / (double)w < r.tol_t && sr / (double)w < r.tol_r_deg;
}

// Pose extrapolation (pcreg_icp_extrap, include/pcreg.h; the rule is extrap_step in pcreg_math.cuh).  Update u took Tc = T_{u-1} to
// Tn = K_u; on return Tn is the pose to write, T_u.  Both ICP paths call this one function, so their poses agree bit for bit.
__device__ __noinline__ static void icp_extrap_update(const IcpExtrapRule& r, const double* s, const double* pivot, const double* cen,
                                                      const double* Tc, double* Tn, int u, double* state) {
    extrap_step(r.angle_deg, r.vmax_scale, s, pivot, cen, Tc, Tn, u, state, nullptr);
}

}  // namespace pcreg
