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

// Thread 0 of a hypothesis after the block reduction: rigid fit from the sums and T <- T * dT.  Returns false (pose left
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
    kabsch_from_sums(ks, pivot, pivot, reflection_fix, dT);
    mul4(Tc, dT, Tn);
    return true;
}

// out-of-line copy for the kernels' hot loops' sake: one thread per hypothesis runs it, its SVD must not claim their registers
__device__ __noinline__ static bool icp_pose_update_call(const double (&s)[KABSCH_NSUMS], long long n_used, const double* pivot,
                                                         bool reflection_fix, const double* Tc, double* Tn) {
    return icp_pose_update(s, n_used, pivot, reflection_fix, Tc, Tn);
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

}  // namespace pcreg
