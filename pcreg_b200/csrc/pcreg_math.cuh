// pcreg_math.cuh -- small FP64 linear algebra shared by every kernel (host + device).
//
// 3x3 one-sided Jacobi SVD, symmetric 3x3 Jacobi eigen-solver, Kabsch pose from the 16 weighted
// sums, row-vector 4x4 composition, the 6x6 LDL' solve and the Rodrigues rotation of the point-to-plane step.  Matrices are ROW-MAJOR double[9] / double[16] in here
// (element (r,c) at [r*3+c] / [r*4+c]); the C ABI converts to MATLAB column-major at the edge.
//
// Reference arithmetic restated (not copied): estimateTransform.m:41-71 (centroids, H = m_c*d_c',
// svd, R = V*U', t = cd - R*cm, T = [R t;0 1]'), MATLAB pca/eig documentation for the eigen part.
#pragma once
#include <math.h>
#include <float.h>

#if defined(__CUDACC__)
#define PCREG_HD __host__ __device__ __forceinline__
#else
#define PCREG_HD inline
#endif

namespace pcreg {

PCREG_HD double det3(const double* A) {
    return A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) +
           A[2] * (A[3] * A[7] - A[4] * A[6]);
}

// C = A * B (3x3 row-major)
PCREG_HD void mul3(const double* A, const double* B, double* C) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c)
            C[r * 3 + c] = A[r * 3 + 0] * B[0 * 3 + c] + A[r * 3 + 1] * B[1 * 3 + c] + A[r * 3 + 2] * B[2 * 3 + c];
}

// C = A * B (4x4 row-major)
PCREG_HD void mul4(const double* A, const double* B, double* C) {
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) {
            double s = 0.0;
            for (int k = 0; k < 4; ++k) s += A[r * 4 + k] * B[k * 4 + c];
            C[r * 4 + c] = s;
        }
}

// One-sided (Hestenes) Jacobi SVD of a 3x3:  A = U * diag(S) * V^T, S descending, V a proper or
// improper orthogonal matrix built from plane rotations (+ the descending sort permutation).
// Accurate to a few ulp of the largest singular value for EVERY singular value (no A^T A squaring).
// Columns of U belonging to singular values below `tiny` are completed by cross products.
PCREG_HD void svd3(const double* A, double* U, double* S, double* V) {
    double G[9];
    for (int i = 0; i < 9; ++i) { G[i] = A[i]; V[i] = 0.0; }
    V[0] = V[4] = V[8] = 1.0;
    for (int sweep = 0; sweep < 40; ++sweep) {
        bool rotated = false;
        for (int pq = 0; pq < 3; ++pq) {
            const int p = (pq == 2) ? 1 : 0;
            const int q = (pq == 0) ? 1 : 2;
            double alpha = 0.0, beta = 0.0, gamma = 0.0;
            for (int i = 0; i < 3; ++i) {
                alpha += G[i * 3 + p] * G[i * 3 + p];
                beta  += G[i * 3 + q] * G[i * 3 + q];
                gamma += G[i * 3 + p] * G[i * 3 + q];
            }
            if (gamma == 0.0 || fabs(gamma) <= 1.1e-16 * sqrt(alpha * beta)) continue;
            rotated = true;
            const double zeta = (beta - alpha) / (2.0 * gamma);
            const double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
            const double c = 1.0 / sqrt(1.0 + t * t);
            const double s = c * t;
            for (int i = 0; i < 3; ++i) {
                const double gp = G[i * 3 + p], gq = G[i * 3 + q];
                G[i * 3 + p] = c * gp - s * gq;
                G[i * 3 + q] = s * gp + c * gq;
                const double vp = V[i * 3 + p], vq = V[i * 3 + q];
                V[i * 3 + p] = c * vp - s * vq;
                V[i * 3 + q] = s * vp + c * vq;
            }
        }
        if (!rotated) break;
    }
    double s[3];
    for (int k = 0; k < 3; ++k)
        s[k] = sqrt(G[0 * 3 + k] * G[0 * 3 + k] + G[1 * 3 + k] * G[1 * 3 + k] + G[2 * 3 + k] * G[2 * 3 + k]);
    // descending sort (3 elements), permuting columns of G and V
    for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2 - a; ++b)
            if (s[b] < s[b + 1]) {
                double tmp = s[b]; s[b] = s[b + 1]; s[b + 1] = tmp;
                for (int i = 0; i < 3; ++i) {
                    tmp = G[i * 3 + b]; G[i * 3 + b] = G[i * 3 + b + 1]; G[i * 3 + b + 1] = tmp;
                    tmp = V[i * 3 + b]; V[i * 3 + b] = V[i * 3 + b + 1]; V[i * 3 + b + 1] = tmp;
                }
            }
    const double tiny = s[0] * 1e-300 + DBL_MIN;
    const double rel  = s[0] * 4.0 * DBL_EPSILON;      // below this a direction is numerically null
    int nvalid = 0;
    for (int k = 0; k < 3; ++k) {
        S[k] = s[k];
        if (s[k] > rel && s[k] > tiny) {
            for (int i = 0; i < 3; ++i) U[i * 3 + k] = G[i * 3 + k] / s[k];
            nvalid = k + 1;
        }
    }
    if (nvalid == 3) return;
    if (nvalid == 2) {           // u2 = u0 x u1
        U[0 * 3 + 2] = U[1 * 3 + 0] * U[2 * 3 + 1] - U[2 * 3 + 0] * U[1 * 3 + 1];
        U[1 * 3 + 2] = U[2 * 3 + 0] * U[0 * 3 + 1] - U[0 * 3 + 0] * U[2 * 3 + 1];
        U[2 * 3 + 2] = U[0 * 3 + 0] * U[1 * 3 + 1] - U[1 * 3 + 0] * U[0 * 3 + 1];
        return;
    }
    if (nvalid == 0) {           // zero matrix: U = I
        for (int i = 0; i < 9; ++i) U[i] = 0.0;
        U[0] = U[4] = U[8] = 1.0;
        return;
    }
    // nvalid == 1: complete u0 to an orthonormal basis
    {
        const double ux = U[0], uy = U[3], uz = U[6];
        int m = 0;                                  // axis least aligned with u0
        if (fabs(uy) < fabs(ux)) m = 1;
        if (fabs(uz) < fabs(m == 0 ? ux : uy)) m = 2;
        double e[3] = {0.0, 0.0, 0.0};
        e[m] = 1.0;
        double bx = uy * e[2] - uz * e[1], by = uz * e[0] - ux * e[2], bz = ux * e[1] - uy * e[0];
        const double bn = sqrt(bx * bx + by * by + bz * bz);
        bx /= bn; by /= bn; bz /= bn;
        U[1] = bx; U[4] = by; U[7] = bz;
        U[2] = uy * bz - uz * by; U[5] = uz * bx - ux * bz; U[8] = ux * by - uy * bx;
    }
}

// Cyclic Jacobi eigen-decomposition of a symmetric 3x3 (only the upper triangle of A is trusted,
// the matrix is symmetrised first).  Returns eigenvalues w (unsorted) and eigenvectors as the
// COLUMNS of V (row-major storage).
PCREG_HD void eigsym3(const double* Ain, double* w, double* V) {
    double A[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) A[r * 3 + c] = 0.5 * (Ain[r * 3 + c] + Ain[c * 3 + r]);
    for (int i = 0; i < 9; ++i) V[i] = 0.0;
    V[0] = V[4] = V[8] = 1.0;
    for (int sweep = 0; sweep < 50; ++sweep) {
        const double off = fabs(A[1]) + fabs(A[2]) + fabs(A[5]);
        const double dia = fabs(A[0]) + fabs(A[4]) + fabs(A[8]);
        if (off == 0.0 || off <= 1e-18 * dia) break;
        for (int pq = 0; pq < 3; ++pq) {
            const int p = (pq == 2) ? 1 : 0;
            const int q = (pq == 0) ? 1 : 2;
            const double apq = A[p * 3 + q];
            if (apq == 0.0) continue;
            const double app = A[p * 3 + p], aqq = A[q * 3 + q];
            const double theta = (aqq - app) / (2.0 * apq);
            const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(1.0 + theta * theta));
            const double c = 1.0 / sqrt(1.0 + t * t);
            const double s = t * c;
            // A <- J^T A J with J = rotation in the (p,q) plane
            for (int k = 0; k < 3; ++k) {               // columns p,q
                const double akp = A[k * 3 + p], akq = A[k * 3 + q];
                A[k * 3 + p] = c * akp - s * akq;
                A[k * 3 + q] = s * akp + c * akq;
            }
            for (int k = 0; k < 3; ++k) {               // rows p,q
                const double apk = A[p * 3 + k], aqk = A[q * 3 + k];
                A[p * 3 + k] = c * apk - s * aqk;
                A[q * 3 + k] = s * apk + c * aqk;
            }
            A[p * 3 + q] = 0.0; A[q * 3 + p] = 0.0;
            for (int k = 0; k < 3; ++k) {
                const double vkp = V[k * 3 + p], vkq = V[k * 3 + q];
                V[k * 3 + p] = c * vkp - s * vkq;
                V[k * 3 + q] = s * vkp + c * vkq;
            }
        }
    }
    w[0] = A[0]; w[1] = A[4]; w[2] = A[8];
}

// Sort eigenpairs (columns of V) ascending (dir = +1) or descending (dir = -1), stable.
PCREG_HD void eigsort3(double* w, double* V, int dir) {
    for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2 - a; ++b) {
            const bool sw = (dir > 0) ? (w[b] > w[b + 1]) : (w[b] < w[b + 1]);
            if (sw) {
                double tmp = w[b]; w[b] = w[b + 1]; w[b + 1] = tmp;
                for (int i = 0; i < 3; ++i) {
                    tmp = V[i * 3 + b]; V[i * 3 + b] = V[i * 3 + b + 1]; V[i * 3 + b + 1] = tmp;
                }
            }
        }
}

// The 17 running sums of one weighted correspondence set.  "q" is the moving (query / pts2 / "m" of
// estimateTransform.m:42) side, "m" the fixed (model / pts1 / "d" of :41) side, both taken
// RELATIVE TO A PIVOT to keep the one-pass cross-covariance well conditioned.
struct KabschSums {
    double sw;        // sum w
    double sq[3];     // sum w * q
    double sm[3];     // sum w * m
    double sqm[9];    // sum w * q_a * m_b   (row a, col b)
    double swd2;      // sum w * d^2  (for rmse)
};
constexpr int KABSCH_NSUMS = 17;

// ICP updates (include/pcreg.h: pcreg_icp_opts.reflection_fix): the cross-covariance H is taken as of numerical rank <= 2 when
// S[2] <= ICP_RANK2_TAU * S[0], or when it is rounding noise (S[0] <= ICP_RANK2_TAU * |sum w q~ m~'|_F, the uncentred sum it was
// cancelled from: coincident correspondences); the update is then the proper solution whatever reflection_fix says.  There the
// rotation and the reflection fit the correspondences equally well and the sign of det(V U') is set by how svd3 completes the null
// direction, not by the data.  The bound: the one-pass pivot-relative sums leave S[2] / S[0] of an exactly planar set at up to
// about 4e-15 (D / L)^2 (200 correspondences on a patch of size L at distance D >= L from the pivot; 4e-11 at D = 100 L,
// tests/test_icp_degenerate_cpu.py), so tau keeps a factor 8 of margin up to D = 500 L, while a curved patch has
// S[2] / S[0] ~ (sag / L)^2, 1e-8 only at a relative sag of 1e-4.
constexpr double ICP_RANK2_TAU = 1e-8;

// dT (row-major, row-vector convention) with [q,1]*dT ~ [m,1]  (estimateTransform(pts1 = m, pts2 = q)).
// pivot_q / pivot_m: what was subtracted from the q side / the m side before summing.  icp_rule: the ICP update's rank rule
// (ICP_RANK2_TAU); estimateTransform / RANSAC pass false and keep R = V*U' (with reflection_fix alone deciding the flip).
PCREG_HD void kabsch_from_sums(const KabschSums& s, const double* pivot_q, const double* pivot_m, bool reflection_fix, double* dT,
                               bool icp_rule = false) {
    const double inv = 1.0 / s.sw;
    double cq[3], cm[3], H[9];
    for (int a = 0; a < 3; ++a) { cq[a] = s.sq[a] * inv; cm[a] = s.sm[a] * inv; }
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) H[a * 3 + b] = s.sqm[a * 3 + b] - s.sq[a] * cm[b];   // estimateTransform.m:58
    double f2 = 0.0;                                                                       // |sum w q~ m~'|_F^2 (ICP rank rule)
    if (icp_rule)
        for (int k = 0; k < 9; ++k) f2 += s.sqm[k] * s.sqm[k];
    double U[9], S[3], V[9];
    svd3(H, U, S, V);                                                                      // :60
    const bool fix = reflection_fix || (icp_rule && (S[2] <= ICP_RANK2_TAU * S[0] || S[0] <= ICP_RANK2_TAU * sqrt(f2)));
    double R[9];
    for (int pass = 0; pass < 2; ++pass) {
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c)                                                   // R = V * U'  (:62)
                R[r * 3 + c] = V[r * 3 + 0] * U[c * 3 + 0] + V[r * 3 + 1] * U[c * 3 + 1] + V[r * 3 + 2] * U[c * 3 + 2];
        if (pass == 1 || !fix || det3(R) >= 0.0) break;
        for (int i = 0; i < 3; ++i) V[i * 3 + 2] = -V[i * 3 + 2];                        // flip the weakest direction
    }
    // t = cd - R*cm (:63) with cd = model centroid, cm = query centroid, pivot restored
    double t[3];
    for (int r = 0; r < 3; ++r) {
        const double Rcq = R[r * 3 + 0] * (cq[0] + pivot_q[0]) + R[r * 3 + 1] * (cq[1] + pivot_q[1]) + R[r * 3 + 2] * (cq[2] + pivot_q[2]);
        t[r] = (cm[r] + pivot_m[r]) - Rcq;
    }
    // T = [R t; 0 1]'  (:66-71)
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) dT[r * 4 + c] = R[c * 3 + r];
    dT[0 * 4 + 3] = 0.0; dT[1 * 4 + 3] = 0.0; dT[2 * 4 + 3] = 0.0;
    dT[3 * 4 + 0] = t[0]; dT[3 * 4 + 1] = t[1]; dT[3 * 4 + 2] = t[2]; dT[3 * 4 + 3] = 1.0;
}

// ---- point-to-plane ICP step (include/pcreg.h: PCREG_ICP_POINT_TO_PLANE) ----
// 29 running sums: sw, the 21 upper-triangle entries of A = sum w a a' (row-major: (0,0), (0,1), .. (0,5), (1,1), ..), the 6 of
// g = sum w a b, sum w d^2
constexpr int PLANE_NSUMS = 29;

// A x = g for a symmetric 6x6 A given by its upper triangle (row-major, 21 entries): A = L D L' without pivoting, unknowns in
// their natural order.  Returns false (x untouched) when some pivot D_k is not above 1e-12 * max_k A_kk (a flat patch leaves a
// direction of the pose unconstrained).
PCREG_HD bool ldlt6_solve(const double* Au, const double* g, double* x) {
    double A[36];
    for (int r = 0, k = 0; r < 6; ++r)
        for (int c = r; c < 6; ++c, ++k) { A[r * 6 + c] = Au[k]; A[c * 6 + r] = Au[k]; }
    double amax = 0.0;
    for (int k = 0; k < 6; ++k) amax = fmax(amax, A[k * 7]);
    const double tiny = 1e-12 * amax;
    double L[36], D[6];
    for (int j = 0; j < 6; ++j) {
        double d = A[j * 7];
        for (int k = 0; k < j; ++k) d -= L[j * 6 + k] * L[j * 6 + k] * D[k];
        if (!(d > tiny)) return false;
        D[j] = d;
        for (int i = j + 1; i < 6; ++i) {
            double v = A[i * 6 + j];
            for (int k = 0; k < j; ++k) v -= L[i * 6 + k] * L[j * 6 + k] * D[k];
            L[i * 6 + j] = v / d;
        }
    }
    double y[6];
    for (int i = 0; i < 6; ++i) {
        double v = g[i];
        for (int k = 0; k < i; ++k) v -= L[i * 6 + k] * y[k];
        y[i] = v;
    }
    for (int i = 5; i >= 0; --i) {
        double v = y[i] / D[i];
        for (int k = i + 1; k < 6; ++k) v -= L[k * 6 + i] * x[k];
        x[i] = v;
    }
    return true;
}

// Rodrigues: R = I + (sin t / t) [w]x + ((1 - cos t) / t^2) [w]x^2, t = |w|; R = I at t = 0.  Column-vector convention (R v =
// v + w x v + ...), row-major storage.
PCREG_HD void rodrigues(const double* w, double* R) {
    const double t2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    const double t = sqrt(t2);
    for (int i = 0; i < 9; ++i) R[i] = 0.0;
    R[0] = R[4] = R[8] = 1.0;
    if (!(t > 0.0)) return;
    const double a = sin(t) / t, b = (1.0 - cos(t)) / t2;
    const double K[9] = {0.0, -w[2], w[1], w[2], 0.0, -w[0], -w[1], w[0], 0.0};
    double K2[9];
    mul3(K, K, K2);
    for (int i = 0; i < 9; ++i) R[i] += a * K[i] + b * K2[i];
}

// ---- plane-to-plane (generalized ICP) step (include/pcreg.h: pcreg_icp_batch_gicp) ----
// One correspondence of weight w into the 29 sums of the point-to-plane layout.  qt = q - p, mt = m - p (p the pivot), nq the
// source normal carried by the pose, nm the model normal, eps in (0, 1]:
//   C = 2I - (1 - eps)(nm nm' + nq nq'),  M = C^-1 = adj(C) / det(C),  e = mt - qt,  J' = [[qt]x; I]  (6 x 3),
//   A += w J' M J = w [[qt]x M [qt]x', [qt]x M; M [qt]x', M]  (upper triangle, row-major),  g += w J' M e = w (qt x Me, Me).
// With M = n n' this is the point-to-plane accumulation: J' n = (qt x n, n) is its a and n' e its b.  C enters only through the
// products n_i n_j, so the sign of either normal changes no bit.  s[0] += w and s[28] += w d as in the other metrics.
PCREG_HD void gicp_accumulate(double* s, double w, double d, const double* qt, const double* mt, const double* nq, const double* nm,
                              double eps) {
    const double a = 1.0 - eps;
    const double c00 = 2.0 - a * (nm[0] * nm[0] + nq[0] * nq[0]), c11 = 2.0 - a * (nm[1] * nm[1] + nq[1] * nq[1]);
    const double c22 = 2.0 - a * (nm[2] * nm[2] + nq[2] * nq[2]);
    const double c01 = -a * (nm[0] * nm[1] + nq[0] * nq[1]), c02 = -a * (nm[0] * nm[2] + nq[0] * nq[2]);
    const double c12 = -a * (nm[1] * nm[2] + nq[1] * nq[2]);
    const double a00 = c11 * c22 - c12 * c12, a01 = c02 * c12 - c01 * c22, a02 = c01 * c12 - c02 * c11;
    const double a11 = c00 * c22 - c02 * c02, a12 = c01 * c02 - c00 * c12, a22 = c00 * c11 - c01 * c01;
    const double f = w / (c00 * a00 + c01 * a01 + c02 * a02);              // w / det(C): w M = f adj(C)
    const double M[9] = {f * a00, f * a01, f * a02, f * a01, f * a11, f * a12, f * a02, f * a12, f * a22};
    const double e[3] = {mt[0] - qt[0], mt[1] - qt[1], mt[2] - qt[2]};
    double Me[3], P[9];                                                    // w M e and P = [qt]x w M (row-major)
    for (int r = 0; r < 3; ++r) Me[r] = M[r * 3 + 0] * e[0] + M[r * 3 + 1] * e[1] + M[r * 3 + 2] * e[2];
    for (int c = 0; c < 3; ++c) {
        P[0 * 3 + c] = qt[1] * M[2 * 3 + c] - qt[2] * M[1 * 3 + c];
        P[1 * 3 + c] = qt[2] * M[0 * 3 + c] - qt[0] * M[2 * 3 + c];
        P[2 * 3 + c] = qt[0] * M[1 * 3 + c] - qt[1] * M[0 * 3 + c];
    }
    // [qt]x w M [qt]x' = P [qt]x': entry (r, c) is (qt x row r of P)_c
    const double T00 = qt[1] * P[2] - qt[2] * P[1], T01 = qt[2] * P[0] - qt[0] * P[2], T02 = qt[0] * P[1] - qt[1] * P[0];
    const double T11 = qt[2] * P[3] - qt[0] * P[5], T12 = qt[0] * P[4] - qt[1] * P[3];
    const double T22 = qt[0] * P[7] - qt[1] * P[6];
    s[0] += w;
    s[1] += T00; s[2] += T01; s[3] += T02; s[4] += P[0]; s[5] += P[1]; s[6] += P[2];
    s[7] += T11; s[8] += T12; s[9] += P[3]; s[10] += P[4]; s[11] += P[5];
    s[12] += T22; s[13] += P[6]; s[14] += P[7]; s[15] += P[8];
    s[16] += M[0]; s[17] += M[1]; s[18] += M[2];
    s[19] += M[4]; s[20] += M[5];
    s[21] += M[8];
    s[22] += qt[1] * Me[2] - qt[2] * Me[1]; s[23] += qt[2] * Me[0] - qt[0] * Me[2]; s[24] += qt[0] * Me[1] - qt[1] * Me[0];
    s[25] += Me[0]; s[26] += Me[1]; s[27] += Me[2];
    s[28] += w * d;
}

// ---- pose extrapolation of the point-to-point ICP (include/pcreg.h: pcreg_icp_extrap; Besl & McKay 1992, section IV) ----
// Poses are row-vector 4x4 (rotation block R(r, c) = T[r * 4 + c], translation row T[12..14]).  A pose's state is
// x(T) = (qR, qT) in R^7: qR = (w, x, y, z) the unit quaternion of R, qT = c R + t the image of the source centroid c.

// Shepperd's conversion: the largest of (trace, R00, R11, R22) picks the component computed from a square root.
PCREG_HD void rot_to_quat(const double* T, double* q) {
    const double r00 = T[0], r01 = T[1], r02 = T[2], r10 = T[4], r11 = T[5], r12 = T[6], r20 = T[8], r21 = T[9], r22 = T[10];
    const double tr = r00 + r11 + r22;
    if (tr >= r00 && tr >= r11 && tr >= r22) {
        const double w = 0.5 * sqrt(1.0 + tr), f = 0.25 / w;
        q[0] = w; q[1] = (r21 - r12) * f; q[2] = (r02 - r20) * f; q[3] = (r10 - r01) * f;
    } else if (r00 >= r11 && r00 >= r22) {
        const double x = 0.5 * sqrt(1.0 + r00 - r11 - r22), f = 0.25 / x;
        q[0] = (r21 - r12) * f; q[1] = x; q[2] = (r01 + r10) * f; q[3] = (r02 + r20) * f;
    } else if (r11 >= r22) {
        const double y = 0.5 * sqrt(1.0 - r00 + r11 - r22), f = 0.25 / y;
        q[0] = (r02 - r20) * f; q[1] = (r01 + r10) * f; q[2] = y; q[3] = (r12 + r21) * f;
    } else {
        const double z = 0.5 * sqrt(1.0 - r00 - r11 + r22), f = 0.25 / z;
        q[0] = (r10 - r01) * f; q[1] = (r02 + r20) * f; q[2] = (r12 + r21) * f; q[3] = z;
    }
}

// The rotation block of T from a unit quaternion (the inverse of rot_to_quat); the other entries of T are left alone.
PCREG_HD void quat_to_rot(const double* q, double* T) {
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    T[0] = 1.0 - 2.0 * (y * y + z * z); T[1] = 2.0 * (x * y - z * w);       T[2] = 2.0 * (x * z + y * w);
    T[4] = 2.0 * (x * y + z * w);       T[5] = 1.0 - 2.0 * (x * x + z * z); T[6] = 2.0 * (y * z - x * w);
    T[8] = 2.0 * (x * z - y * w);       T[9] = 2.0 * (y * z + x * w);       T[10] = 1.0 - 2.0 * (x * x + y * y);
}

// x(T) for source centroid c.  Sign of qR: with qprev (a previous state's quaternion) the one with qR . qprev >= 0; without, w >= 0
// and, at w = 0, the first nonzero component positive.
PCREG_HD void pose_state(const double* T, const double* c, const double* qprev, double* x) {
    rot_to_quat(T, x);
    bool flip;
    if (qprev) {
        flip = x[0] * qprev[0] + x[1] * qprev[1] + x[2] * qprev[2] + x[3] * qprev[3] < 0.0;
    } else {
        int k = 0;
        while (k < 3 && x[k] == 0.0) ++k;
        flip = x[k] < 0.0;
    }
    if (flip) for (int k = 0; k < 4; ++k) x[k] = -x[k];
    for (int b = 0; b < 3; ++b) x[4 + b] = c[0] * T[0 * 4 + b] + c[1] * T[1 * 4 + b] + c[2] * T[2 * 4 + b] + T[12 + b];
}

// Weighted mean-square error sum w |m - quickTF(s, T)|^2 / sum w of the correspondences behind the 17 sums s (taken at pose Tc,
// relative to pivot p) at another pose T.  With E = Tc^-1 T = [RE 0; tE 1] a source point moves from q to q RE + tE; with centred
// q^ = q - p - cq, m^ = m - p - cm (cq, cm the weighted centroids relative to p) and H = sum w q^ m^' the centred cross-covariance:
//   sum w |e|^2 = (s16 - sw |cm - cq|^2) + 2 sum_ab (I - RE)_ab H_ab + sw |cm - cq RE - tau|^2,  tau = (tE + p RE) - p
//               = (t - p) - (tc - p) RE.
// Every term is small where the result is small, so a cloud far from the pivot loses no accuracy to cancellation.
PCREG_HD double sums_mse_at(const double* s, const double* p, const double* Tc, const double* T) {
    const double sw = s[0], inv = 1.0 / sw;
    double cq[3], cm[3], RE[9];
    for (int a = 0; a < 3; ++a) { cq[a] = s[1 + a] * inv; cm[a] = s[4 + a] * inv; }
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) RE[a * 3 + b] = Tc[0 * 4 + a] * T[0 * 4 + b] + Tc[1 * 4 + a] * T[1 * 4 + b] + Tc[2 * 4 + a] * T[2 * 4 + b];
    double e0 = 0.0, rot = 0.0, dl = 0.0;
    for (int a = 0; a < 3; ++a) e0 += (cm[a] - cq[a]) * (cm[a] - cq[a]);
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) {
            const double H = s[7 + a * 3 + b] - s[1 + a] * cm[b];
            rot += ((a == b ? 1.0 : 0.0) - RE[a * 3 + b]) * H;
        }
    for (int b = 0; b < 3; ++b) {
        double tau = T[12 + b] - p[b], cqR = 0.0;
        for (int a = 0; a < 3; ++a) { tau -= (Tc[12 + a] - p[a]) * RE[a * 3 + b]; cqR += cq[a] * RE[a * 3 + b]; }
        const double r = cm[b] - cqR - tau;
        dl += r * r;
    }
    return ((s[16] - sw * e0) + 2.0 * rot + sw * dl) * inv;
}

// Zero of the least-squares line through (v_i, D_i), i = 0..2 (NaN or infinite when the line is flat).
PCREG_HD double extrap_line_zero(const double* v, const double* D) {
    const double vm = (v[0] + v[1] + v[2]) / 3.0, Dm = (D[0] + D[1] + D[2]) / 3.0;
    double sxy = 0.0, sxx = 0.0;
    for (int i = 0; i < 3; ++i) { sxy += (v[i] - vm) * (D[i] - Dm); sxx += (v[i] - vm) * (v[i] - vm); }
    return vm - Dm / (sxy / sxx);
}

// Vertex -b / (2a) of the parabola a v^2 + b v + c through the three points (Newton's divided differences).
PCREG_HD double extrap_parabola_vertex(const double* v, const double* D) {
    const double f01 = (D[1] - D[0]) / (v[1] - v[0]), f12 = (D[2] - D[1]) / (v[2] - v[1]);
    const double a = (f12 - f01) / (v[2] - v[0]);
    const double b = f01 - a * (v[0] + v[1]);
    return -b / (2.0 * a);
}

// The step along the update direction (Besl & McKay's choice between the line zero v1, the parabola vertex v2 and the cap vmax).
// Strict compares; NaN fails each.  Returns the branch: 1 = v2, 2 = v1, 3 = vmax, 0 = no step (*dv = 0).
PCREG_HD int extrap_branch(double v1, double v2, double vmax, double* dv) {
    if ((0.0 < v2 && v2 < v1 && v1 < vmax) || (0.0 < v2 && v2 < vmax && vmax < v1)) { *dv = v2; return 1; }
    if ((0.0 < v1 && v1 < v2 && v2 < vmax) || (0.0 < v1 && v1 < vmax && vmax < v2) || (v2 < 0.0 && 0.0 < v1 && v1 < vmax)) { *dv = v1; return 2; }
    if (v1 > vmax && v2 > vmax) { *dv = vmax; return 3; }
    *dv = 0.0;
    return 0;
}

// Per-hypothesis state of the extrapolation: x_{u-1} [0..6], Delta_{u-1} [7..13], n_{u-1} [14], theta_{u-1} [15] (NaN: undefined),
// d_{u-1} [16], d_{u-2} [17], updates extrapolated so far [18], 1 when the history restarts at the next update [19].  All zero
// before the first update.
constexpr int EXTRAP_STATE = 20;
constexpr int EXTRAP_NTRACE = 5;       // theta_u, v1, v2, dv, branch of one update (host tests)

// det of the rotation block of a row-major 4x4 pose
PCREG_HD double det_rot4(const double* T) {
    return T[0] * (T[5] * T[10] - T[6] * T[9]) - T[1] * (T[4] * T[10] - T[6] * T[8]) + T[2] * (T[4] * T[9] - T[5] * T[8]);
}

// Update u >= 1 (not degenerate) of one hypothesis: Tc = T_{u-1}, Tn = K_u = T_{u-1} dT on entry, T_u on return; s = the update's
// 17 sums (relative to pivot p), c = the source centroid.  Returns the branch (0: T_u = K_u).
// An improper K_u or T_{u-1} (reflection_fix = 0 reproducing R = V*U') has no quaternion state: that update is not extrapolated
// (T_u = K_u) and the history restarts at the next update, which takes its T_{u-1} as update 1 takes T_0.  So every returned pose
// has the handedness of its Kabsch pose.
PCREG_HD int extrap_step(double angle_deg, double vmax_scale, const double* s, const double* p, const double* c, const double* Tc,
                         double* Tn, int u, double* st, double* trace) {
    const double nan_v = NAN;
    if (!(det_rot4(Tc) > 0.0 && det_rot4(Tn) > 0.0)) {
        st[19] = 1.0;
        if (trace) { trace[0] = nan_v; trace[1] = nan_v; trace[2] = nan_v; trace[3] = 0.0; trace[4] = 0.0; }
        return 0;
    }
    if (u == 1 || st[19] != 0.0) {
        pose_state(Tc, c, nullptr, st);
        for (int k = 7; k < 18; ++k) st[k] = nan_v;
        st[19] = 0.0;
    }
    double xk[7], dl[7], n2 = 0.0;
    pose_state(Tn, c, st, xk);
    for (int k = 0; k < 7; ++k) { dl[k] = xk[k] - st[k]; n2 += dl[k] * dl[k]; }
    const double n = sqrt(n2), np = st[14];
    double th = nan_v;
    if (u >= 2 && n > 0.0 && np > 0.0) {
        double dot = 0.0;
        for (int k = 0; k < 7; ++k) dot += dl[k] * st[7 + k];
        const double cs = fmin(fmax(dot / (n * np), -1.0), 1.0);
        th = acos(cs) * (180.0 / 3.14159265358979323846);
    }
    const double dK = sums_mse_at(s, p, Tc, Tn);
    double v1 = nan_v, v2 = nan_v, dv = 0.0;
    int br = 0;
    if (u >= 3 && th < angle_deg && st[15] < angle_deg) {
        const double v[3] = {0.0, -n, -n - np}, D[3] = {dK, st[16], st[17]};
        v1 = extrap_line_zero(v, D);
        v2 = extrap_parabola_vertex(v, D);
        br = extrap_branch(v1, v2, vmax_scale * n, &dv);
    }
    double dU = dK;
    if (dv > 0.0) {
        const double f = dv / n;
        for (int k = 0; k < 7; ++k) xk[k] += f * dl[k];
        const double qn = sqrt(xk[0] * xk[0] + xk[1] * xk[1] + xk[2] * xk[2] + xk[3] * xk[3]);
        for (int k = 0; k < 4; ++k) xk[k] /= qn;
        quat_to_rot(xk, Tn);
        for (int b = 0; b < 3; ++b) Tn[12 + b] = xk[4 + b] - (c[0] * Tn[0 * 4 + b] + c[1] * Tn[1 * 4 + b] + c[2] * Tn[2 * 4 + b]);
        dU = sums_mse_at(s, p, Tc, Tn);
        st[18] += 1.0;
    }
    for (int k = 0; k < 7; ++k) { st[k] = xk[k]; st[7 + k] = dl[k]; }
    st[14] = n; st[15] = th; st[17] = st[16]; st[16] = dU;
    if (trace) { trace[0] = th; trace[1] = v1; trace[2] = v2; trace[3] = dv; trace[4] = (double)br; }
    return br;
}

// MATLAB eps(x) for x >= 0: spacing of doubles at x.
PCREG_HD double spacing(double x) {
    if (!(x > 0.0)) return 4.9406564584124654e-324;
    int e;
    frexp(x, &e);                       // x = f * 2^e, f in [0.5, 1)
    const double sp = ldexp(1.0, e - 53);
    return sp > 0.0 ? sp : 4.9406564584124654e-324;
}

// MATLAB rank() of an n x 3 matrix given its singular values: count(s > max(n,3) * eps(max s)).
PCREG_HD int rank_from_sv(const double* s, long long n) {
    double smax = s[0];
    if (s[1] > smax) smax = s[1];
    if (s[2] > smax) smax = s[2];
    const double tol = (double)(n > 3 ? n : 3) * spacing(smax);
    return (s[0] > tol) + (s[1] > tol) + (s[2] > tol);
}

}  // namespace pcreg
