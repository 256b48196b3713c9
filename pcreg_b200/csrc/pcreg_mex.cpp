// pcreg_mex.cpp -- MEX gateway: MATLAB <-> the C ABI of include/pcreg.h.  Pure marshaling.
//
//   out = pcreg_mex('command', args...)
//
// Build (on a host with MATLAB):  mex -R2018a pcreg_mex.cpp -I../../include -L.. -lpcreg_b200
// Conventions: inputs are borrowed read-only (mxGetData, never written); outputs are allocated with
// mxCreate* (MATLAB owns them); "the reference returns []" -> a 0x0 double; CUDA / argument errors ->
// mexErrMsgIdAndTxt (which long-jumps: it is only called after every C++ object of the frame is gone,
// via the fail() pattern below).  The model handle travels as a uint64 scalar.  Indices are converted
// to MATLAB's 1-based convention here.
//
// Commands (the matlab/*.m shims call these with the reference's own signatures):
//   'init'[, devices]                                  -> []      (scalar or vector of CUDA ordinals)
//   'model_create', pts(Nx3 single|double)[, grid]     -> handle (uint64)
//   'model_destroy', handle
//   'nn_search', handle, q(Nx3)[, 'grid']              -> idx (Nx1 double, 1-based), d2 (Nx1)
//   'align', kind, pts(Nx3)[, C1, C2 | K]              -> pts_aligned, coeff_unambig, c      (AlignPoints*.m)
//   'estimate_transform', pts1, pts2                   -> T (4x4) or []                      (estimateTransform.m)
//   'ransac', pts1, pts2, coef(struct), triplets(Hx3, 1-based)
//                                                      -> T, inlierIdx, numSuccess, maxInliers, pct  (ransac.m)
//   'ransac_seeded', pts1, pts2, coef(struct incl. iterNum), seed
//                                                      -> same five outputs, samples drawn on the device (pcreg_ransac_run)
//   'ransac_batch', pts1(Nx3), pts2(Nx3), offsets((W+1)x1, 0-based row offsets of the windows), coef(struct incl. iterNum), seeds(Wx1)
//                                                      -> T (16xW, NaN where ransac.m returns []), inlierMask (Nx1), numSuccess (Wx1),
//                                                         maxInliers (Wx1), pct (Wx1)   (one ransac.m call per window, pcreg_ransac_batch)
//   'local_points', handle, c(Kx3 double), R, min_points, max_points
//                                                      -> pts_sphere (concatenated, relative to their centre), dists,
//                                                         counts (Kx1; 0 where the reference returns [])   (getLocalPoints.m)
//   'spatial_histogram', handle, sample_pts(Kx3 double), options(struct), r_bins, theta_bins, phi_bins
//                                                      -> feat (Vx3), desc (Vx(nr*nt*np))     (getSpacialHistogramDescriptors.m)
//   'get_matches', descSurface(N1xD double), descModel(N2xD double), par(struct)
//                                                      -> matches (Px2 uint32, 1-based), matchMetric (Px1)   (getMatches.m)
//   'icp', handle, src(Nx3), T0(4x4xH), opts(struct)[, w_src]
//                                                      -> T(4x4xH), rmse(Hx1), n_used, status, best(1-based), idx(NxH)
// The ICP of many matching windows in one call has a gateway of its own (pcreg_mex_windows.cpp).
#include <string.h>
#include <string>
#include <vector>

#include "mex.h"
#include "../../include/pcreg.h"
#include "pcreg_mex_util.h"

namespace {

bool g_init = false;
std::string g_fail;                // set instead of throwing; reported after the frame unwinds

void at_exit() { pcreg_shutdown(); g_init = false; }

// devices: a MATLAB scalar or vector of CUDA ordinals (pcreg_mex('init', 0:7) drives eight GPUs from this one process)
bool ensure_init(const mxArray* devices) {
    if (g_init) return true;
    int dev[16] = {0};
    int nd = 1;
    if (devices && !mxIsEmpty(devices)) {
        nd = (int)mxGetNumberOfElements(devices);
        if (nd > 16 || !mxIsDouble(devices)) { g_fail = "init: devices must be a double vector of at most 16 ordinals"; return false; }
        for (int k = 0; k < nd; ++k) dev[k] = (int)mxGetPr(devices)[k];
    }
    if (pcreg_init(dev, nd) != PCREG_OK) { g_fail = pcreg_last_error(); return false; }
    mexLock();
    mexAtExit(at_exit);
    g_init = true;
    return true;
}

mxArray* empty() { return mxCreateDoubleMatrix(0, 0, mxREAL); }

// ---- commands: each returns false with g_fail set on error ----
bool cmd_model_create(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 2 || !is_pts(prhs[1])) { g_fail = "model_create: pts must be N x 3 single or double"; return false; }
    pcreg_model_opts o;
    memset(&o, 0, sizeof o);
    o.build_grid = (nrhs > 2) ? (mxGetScalar(prhs[2]) != 0) : 1;
    pcreg_model* m = nullptr;
    const int64_t n = (int64_t)mxGetM(prhs[1]);
    if (pcreg_model_create(mxGetData(prhs[1]), mxIsDouble(prhs[1]), n, n, &o, &m) != PCREG_OK) { g_fail = pcreg_last_error(); return false; }
    plhs[0] = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
    *(uint64_t*)mxGetData(plhs[0]) = (uint64_t)(uintptr_t)m;
    return true;
}

bool cmd_nn_search(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    pcreg_model* m = nrhs > 1 ? handle_of(prhs[1]) : nullptr;
    if (!m || nrhs < 3 || !is_pts(prhs[2])) { g_fail = "nn_search: need (handle, q Nx3)"; return false; }
    const int64_t nq = (int64_t)mxGetM(prhs[2]);
    std::vector<int32_t> idx((size_t)nq);
    plhs[0] = mxCreateDoubleMatrix((mwSize)nq, 1, mxREAL);
    mxArray* d2 = mxCreateDoubleMatrix((mwSize)nq, 1, mxREAL);
    const int kind = (nrhs > 3) ? PCREG_NN_GRID : PCREG_NN_BRUTE;
    const int rc = pcreg_nn_search(m, mxGetData(prhs[2]), mxIsDouble(prhs[2]), nq, nq, kind, idx.data(), mxGetPr(d2));
    if (rc != PCREG_OK) { g_fail = pcreg_last_error(); mxDestroyArray(d2); mxDestroyArray(plhs[0]); plhs[0] = nullptr; return false; }
    double* o = mxGetPr(plhs[0]);
    for (int64_t i = 0; i < nq; ++i) o[i] = (double)idx[(size_t)i] + 1.0;
    if (nlhs > 1) plhs[1] = d2; else mxDestroyArray(d2);
    return true;
}

// pts_tf = pcreg_mex('quick_tf', pts, TF[, mode])   mode 0: [pts 1]*TF (quickTF.m), 1: [pts 1]*invertTF(TF), 2: [pts 1]/TF
bool cmd_quick_tf(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 3 || !is_pts(prhs[1]) || !mxIsDouble(prhs[2]) || mxGetM(prhs[2]) != 4 || mxGetN(prhs[2]) != 4) {
        g_fail = "quick_tf: need (pts Nx3 single or double, TF 4x4 double[, mode])"; return false;
    }
    const int64_t n = (int64_t)mxGetM(prhs[1]);
    const int mode = nrhs > 3 ? (int)mxGetScalar(prhs[3]) : PCREG_TF_FORWARD;
    if (n == 0) { plhs[0] = mxCreateNumericMatrix(0, 3, mxIsDouble(prhs[1]) ? mxDOUBLE_CLASS : mxSINGLE_CLASS, mxREAL); return true; }
    plhs[0] = mxCreateNumericMatrix((mwSize)n, 3, mxIsDouble(prhs[1]) ? mxDOUBLE_CLASS : mxSINGLE_CLASS, mxREAL);
    const int rc = pcreg_quick_tf(mxGetData(prhs[1]), mxIsDouble(prhs[1]), n, n, mxGetPr(prhs[2]), mode, mxGetData(plhs[0]), n);
    if (rc != PCREG_OK) { g_fail = pcreg_last_error(); mxDestroyArray(plhs[0]); plhs[0] = nullptr; return false; }
    return true;
}

bool cmd_local_points(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    pcreg_model* m = nrhs > 1 ? handle_of(prhs[1]) : nullptr;
    if (!m || nrhs < 6 || !is_pts(prhs[2]) || !mxIsDouble(prhs[2])) { g_fail = "local_points: need (handle, c Kx3 double, R, min_points, max_points)"; return false; }
    const int64_t nc = (int64_t)mxGetM(prhs[2]);
    const double R = mxGetScalar(prhs[3]), mx = mxGetScalar(prhs[5]);
    const int64_t min_points = (int64_t)mxGetScalar(prhs[4]);
    const int64_t max_points = (mx > 9.0e18) ? -1 : (int64_t)mx;                 // inf (AlignPoints_c.m:14)
    std::vector<int64_t> counts((size_t)nc), offsets((size_t)nc + 1, 0);
    std::vector<int32_t> status((size_t)nc);
    if (pcreg_local_points_count(m, mxGetPr(prhs[2]), nc, nc, R, min_points, max_points, counts.data(), status.data()) != PCREG_OK) {
        g_fail = pcreg_last_error();
        return false;
    }
    for (int64_t k = 0; k < nc; ++k) offsets[(size_t)k + 1] = offsets[(size_t)k] + (status[(size_t)k] ? 0 : counts[(size_t)k]);
    const int64_t nt = offsets[(size_t)nc];
    if (nt == 0) {                                                              // getLocalPoints.m:17-19,31-34: [] , []
        plhs[0] = empty();
        if (nlhs > 1) plhs[1] = empty();
    } else {
        mxArray* pts = mxCreateDoubleMatrix((mwSize)nt, 3, mxREAL);
        mxArray* dists = mxCreateDoubleMatrix((mwSize)nt, 1, mxREAL);
        if (pcreg_local_points_fill(m, mxGetPr(prhs[2]), nc, nc, R, offsets.data(), status.data(), mxGetPr(pts), nt, mxGetPr(dists), nullptr) != PCREG_OK) {
            g_fail = pcreg_last_error();
            mxDestroyArray(pts); mxDestroyArray(dists);
            return false;
        }
        plhs[0] = pts;
        if (nlhs > 1) plhs[1] = dists; else mxDestroyArray(dists);
    }
    if (nlhs > 2) {
        plhs[2] = mxCreateDoubleMatrix((mwSize)nc, 1, mxREAL);
        for (int64_t k = 0; k < nc; ++k) mxGetPr(plhs[2])[k] = status[(size_t)k] ? 0.0 : (double)counts[(size_t)k];
    }
    return true;
}

bool cmd_spatial_histogram(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    pcreg_model* m = nrhs > 1 ? handle_of(prhs[1]) : nullptr;
    if (!m || nrhs < 7 || !is_pts(prhs[2]) || !mxIsDouble(prhs[2]) || !mxIsStruct(prhs[3]) || !mxIsDouble(prhs[4]) ||
        !mxIsDouble(prhs[5]) || !mxIsDouble(prhs[6])) {
        g_fail = "spatial_histogram: need (handle, sample_pts Kx3 double, options struct, r_bins, theta_bins, phi_bins)";
        return false;
    }
    const mxArray* opt = prhs[3];
    pcreg_desc_opts o;
    pcreg_desc_opts_default(&o);
    o.min_pts = (int64_t)field_or(opt, "min_pts", (double)o.min_pts);
    const double mx = field_or(opt, "max_pts", (double)o.max_pts);
    o.max_pts = (mx > 9.0e18) ? -1 : (int64_t)mx;
    o.R = field_or(opt, "R", o.R);
    const mxArray* th = mxGetField(opt, 0, "thVar");
    if (th && mxIsDouble(th) && mxGetNumberOfElements(th) >= 2) { o.thVar[0] = mxGetPr(th)[0]; o.thVar[1] = mxGetPr(th)[1]; }
    const mxArray* kf = mxGetField(opt, 0, "k");                                // 'all' or a fraction (getSpacialHistogramDescriptors.m:74)
    o.k_frac = (kf && !mxIsChar(kf) && !mxIsEmpty(kf)) ? mxGetScalar(kf) : 0.0;
    o.align_points = field_or(opt, "ALIGN_POINTS", 1.0) != 0.0;
    const int nr = (int)mxGetNumberOfElements(prhs[4]) - 1, nt = (int)mxGetNumberOfElements(prhs[5]) - 1, np = (int)mxGetNumberOfElements(prhs[6]) - 1;
    const int64_t nk = (int64_t)mxGetM(prhs[2]);
    if (nr < 1 || nt < 1 || np < 1) { g_fail = "spatial_histogram: every edge vector needs at least two values"; return false; }
    const int64_t nb = (int64_t)nr * nt * np;
    std::vector<double> desc((size_t)nk * (size_t)nb);
    std::vector<int32_t> status((size_t)nk);
    if (pcreg_spatial_histogram(m, mxGetPr(prhs[2]), nk, nk, &o, mxGetPr(prhs[4]), nr, mxGetPr(prhs[5]), nt, mxGetPr(prhs[6]), np,
                                desc.data(), status.data(), nullptr) != PCREG_OK) {
        g_fail = pcreg_last_error();
        return false;
    }
    int64_t nv = 0;
    for (int64_t k = 0; k < nk; ++k) nv += status[(size_t)k] == 0;
    // only the surviving keypoints, in keypoint order (getSpacialHistogramDescriptors.m:176-179)
    plhs[0] = mxCreateDoubleMatrix((mwSize)nv, 3, mxREAL);
    mxArray* D = mxCreateDoubleMatrix((mwSize)nv, (mwSize)nb, mxREAL);
    const double* kp = mxGetPr(prhs[2]);
    int64_t v = 0;
    for (int64_t k = 0; k < nk; ++k) {
        if (status[(size_t)k] != 0) continue;
        for (int a = 0; a < 3; ++a) mxGetPr(plhs[0])[a * nv + v] = kp[a * nk + k];
        for (int64_t j = 0; j < nb; ++j) mxGetPr(D)[j * nv + v] = desc[(size_t)k * (size_t)nb + (size_t)j];
        ++v;
    }
    if (nlhs > 1) plhs[1] = D; else mxDestroyArray(D);
    return true;
}

bool cmd_align(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 3 || !is_pts(prhs[2])) { g_fail = "align: need (kind, pts Nx3)"; return false; }
    const int kind = (int)mxGetScalar(prhs[1]);
    pcreg_align_opts o;
    pcreg_align_opts_default(&o);
    if (kind == PCREG_ALIGN_KNN_FRAC && nrhs >= 5) { o.C1 = mxGetScalar(prhs[3]) != 0; o.C2 = mxGetScalar(prhs[4]) != 0; }
    if (kind == PCREG_ALIGN_KNN_ABS && nrhs >= 4) o.k_abs = (int64_t)mxGetScalar(prhs[3]);
    const int64_t n = (int64_t)mxGetM(prhs[2]);
    const int is_double = mxIsDouble(prhs[2]);
    const int64_t offsets[2] = {0, n};
    mxArray* out = mxCreateNumericMatrix((mwSize)n, 3, is_double ? mxDOUBLE_CLASS : mxSINGLE_CLASS, mxREAL);
    mxArray* coeff = mxCreateDoubleMatrix(3, 3, mxREAL);
    mxArray* c = mxCreateDoubleMatrix(1, 3, mxREAL);
    int32_t status = 0;
    const int rc = pcreg_align_points(kind, mxGetData(prhs[2]), is_double, n, offsets, 1, &o, mxGetData(out), mxGetPr(coeff), mxGetPr(c), &status);
    if (rc != PCREG_OK) { g_fail = pcreg_last_error(); mxDestroyArray(out); mxDestroyArray(coeff); mxDestroyArray(c); return false; }
    if (status != 0) {                      // AlignPoints_c.m:16-18 / AlignPoints_KNN_c.m:53-56: [] , []
        mxDestroyArray(out); mxDestroyArray(coeff);
        out = empty(); coeff = empty();
    }
    plhs[0] = out;
    if (nlhs > 1) plhs[1] = coeff; else mxDestroyArray(coeff);
    if (nlhs > 2) plhs[2] = c; else mxDestroyArray(c);
    return true;
}

bool cmd_estimate_transform(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 3 || !mxIsDouble(prhs[1]) || !mxIsDouble(prhs[2]) || mxGetN(prhs[1]) != 3 || mxGetN(prhs[2]) != 3 ||
        mxGetM(prhs[1]) != mxGetM(prhs[2])) { g_fail = "estimate_transform: need two N x 3 double arrays"; return false; }
    const int64_t n = (int64_t)mxGetM(prhs[1]);
    const int64_t offsets[2] = {0, n};
    mxArray* T = mxCreateDoubleMatrix(4, 4, mxREAL);
    int32_t status = 0;
    const int rc = pcreg_kabsch_batch(mxGetPr(prhs[1]), mxGetPr(prhs[2]), nullptr, n, offsets, 1, 0, mxGetPr(T), &status);
    if (rc != PCREG_OK) { g_fail = pcreg_last_error(); mxDestroyArray(T); return false; }
    if (status != 0) { mxDestroyArray(T); T = empty(); }              // estimateTransform.m:11-14
    plhs[0] = T;
    return true;
}

bool cmd_ransac(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[], bool seeded) {
    if (nrhs < 5 || !mxIsDouble(prhs[1]) || !mxIsDouble(prhs[2]) || !mxIsStruct(prhs[3]) || !mxIsDouble(prhs[4]) ||
        mxGetN(prhs[1]) != 3 || mxGetN(prhs[2]) != 3 || (!seeded && mxGetN(prhs[4]) != 3)) {
        g_fail = "ransac: need (pts1, pts2, coef, triplets Hx3 | seed)";
        return false;
    }
    const int64_t P = (int64_t)mxGetM(prhs[1]);
    const int64_t H = seeded ? (int64_t)field_or(prhs[3], "iterNum", 1000.0) : (int64_t)mxGetM(prhs[4]);
    pcreg_ransac_opts o;
    o.thDist = field_or(prhs[3], "thDist", 0.5);
    o.thInlrRatio = field_or(prhs[3], "thInlrRatio", 0.1);
    o.refine = field_or(prhs[3], "REFINE", 1.0) != 0;
    o.reflection_fix = 0;
    std::vector<int32_t> tri(seeded ? 0 : (size_t)H * 3), inl((size_t)P);
    double T16[16];
    int64_t n_inl = 0, n_succ = 0, max_inl = 0, best = -1;
    int rc;
    if (seeded) {
        rc = pcreg_ransac_run(mxGetPr(prhs[1]), mxGetPr(prhs[2]), P, P, H, (uint64_t)mxGetScalar(prhs[4]), &o, T16, inl.data(), &n_inl,
                              &n_succ, &max_inl, &best, nullptr);
    } else {
        const double* t = mxGetPr(prhs[4]);
        for (int64_t h = 0; h < H; ++h)
            for (int k = 0; k < 3; ++k) tri[(size_t)h * 3 + k] = (int32_t)t[k * H + h] - 1;
        rc = pcreg_ransac_score(mxGetPr(prhs[1]), mxGetPr(prhs[2]), P, P, tri.data(), H, &o, T16, inl.data(), &n_inl, &n_succ,
                                &max_inl, &best, nullptr, nullptr, nullptr);
    }
    if (rc < 0) { g_fail = pcreg_last_error(); return false; }
    if (rc == PCREG_DEGENERATE) {                                       // ransac.m:75-89
        plhs[0] = empty();
        if (nlhs > 1) plhs[1] = empty();
        for (int k = 2; k < nlhs && k < 5; ++k) plhs[k] = mxCreateDoubleScalar(0.0);
        return true;
    }
    plhs[0] = mxCreateDoubleMatrix(4, 4, mxREAL);
    memcpy(mxGetPr(plhs[0]), T16, sizeof T16);
    if (nlhs > 1) {
        plhs[1] = mxCreateDoubleMatrix((mwSize)n_inl, 1, mxREAL);
        for (int64_t i = 0; i < n_inl; ++i) mxGetPr(plhs[1])[i] = (double)inl[(size_t)i] + 1.0;
    }
    if (nlhs > 2) plhs[2] = mxCreateDoubleScalar((double)n_succ);
    if (nlhs > 3) plhs[3] = mxCreateDoubleScalar((double)max_inl);
    if (nlhs > 4) plhs[4] = mxCreateDoubleScalar(100.0 * (double)max_inl / (double)P);
    return true;
}

bool cmd_ransac_batch(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 6 || !mxIsDouble(prhs[1]) || !mxIsDouble(prhs[2]) || !mxIsDouble(prhs[3]) || !mxIsStruct(prhs[4]) || !mxIsDouble(prhs[5]) ||
        mxGetN(prhs[1]) != 3 || mxGetN(prhs[2]) != 3 || mxGetM(prhs[1]) != mxGetM(prhs[2]) || mxGetNumberOfElements(prhs[3]) < 2 ||
        mxGetNumberOfElements(prhs[5]) + 1 != mxGetNumberOfElements(prhs[3])) {
        g_fail = "ransac_batch: need (pts1 Nx3, pts2 Nx3, offsets (W+1), coef, seeds W)";
        return false;
    }
    const int64_t N = (int64_t)mxGetM(prhs[1]);
    const int64_t W = (int64_t)mxGetNumberOfElements(prhs[5]);
    const int64_t H = (int64_t)field_or(prhs[4], "iterNum", 1000.0);
    pcreg_ransac_opts o;
    o.thDist = field_or(prhs[4], "thDist", 0.5);
    o.thInlrRatio = field_or(prhs[4], "thInlrRatio", 0.1);
    o.refine = field_or(prhs[4], "REFINE", 1.0) != 0;
    o.reflection_fix = 0;
    std::vector<int64_t> off((size_t)W + 1), n_inl((size_t)W), n_succ((size_t)W), max_inl((size_t)W), best((size_t)W);
    std::vector<uint64_t> seeds((size_t)W);
    std::vector<int32_t> inl((size_t)(N > 0 ? N : 1)), status((size_t)W);
    for (int64_t w = 0; w <= W; ++w) off[(size_t)w] = (int64_t)mxGetPr(prhs[3])[w];
    for (int64_t w = 0; w < W; ++w) seeds[(size_t)w] = (uint64_t)mxGetPr(prhs[5])[w];
    if (off[0] != 0 || off[(size_t)W] != N) { g_fail = "ransac_batch: offsets must run from 0 to size(pts1,1)"; return false; }
    mxArray* T = mxCreateDoubleMatrix(16, (mwSize)W, mxREAL);
    const int rc = pcreg_ransac_batch(mxGetPr(prhs[1]), mxGetPr(prhs[2]), N > 0 ? N : 1, off.data(), W, H, nullptr, seeds.data(), &o,
                                      mxGetPr(T), inl.data(), n_inl.data(), n_succ.data(), max_inl.data(), best.data(), status.data());
    if (rc != PCREG_OK) { g_fail = pcreg_last_error(); mxDestroyArray(T); return false; }
    plhs[0] = T;
    if (nlhs > 1) {
        plhs[1] = mxCreateDoubleMatrix((mwSize)N, 1, mxREAL);                  // zero-filled
        for (int64_t w = 0; w < W; ++w)
            for (int64_t k = 0; k < n_inl[(size_t)w]; ++k) mxGetPr(plhs[1])[off[(size_t)w] + inl[(size_t)(off[(size_t)w] + k)]] = 1.0;
    }
    for (int k = 2; k < nlhs && k < 5; ++k) {
        plhs[k] = mxCreateDoubleMatrix((mwSize)W, 1, mxREAL);
        for (int64_t w = 0; w < W; ++w) {
            const int64_t Pw = off[(size_t)w + 1] - off[(size_t)w];
            mxGetPr(plhs[k])[w] = k == 2 ? (double)n_succ[(size_t)w] : k == 3 ? (double)max_inl[(size_t)w]
                                  : (Pw > 0 ? 100.0 * (double)max_inl[(size_t)w] / (double)Pw : 0.0);
        }
    }
    return true;
}

bool cmd_get_matches(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 4 || !mxIsDouble(prhs[1]) || !mxIsDouble(prhs[2]) || mxIsComplex(prhs[1]) || mxIsComplex(prhs[2]) || !mxIsStruct(prhs[3]) ||
        mxGetN(prhs[1]) != mxGetN(prhs[2])) {
        g_fail = "get_matches: need (descSurface N1xD double, descModel N2xD double, par struct)";
        return false;
    }
    pcreg_match_opts o;
    pcreg_match_opts_default(&o);
    o.unnormalize = field_or(prhs[3], "UNNORMALIZE", 0.0) != 0;             // getMatches.m:22
    o.norm_factor = field_or(prhs[3], "norm_factor", o.norm_factor);
    o.change_metric = field_or(prhs[3], "CHANGE_METRIC", 0.0) != 0;         // :35
    o.metric_factor = field_or(prhs[3], "metric_factor", o.metric_factor);
    o.match_threshold = field_or(prhs[3], "MatchThreshold", 1.0);           // matchFeatures' own defaults when absent
    o.max_ratio = field_or(prhs[3], "MaxRatio", 0.6);
    o.unique = field_or(prhs[3], "Unique", 0.0) != 0;
    o.metric = PCREG_METRIC_SSD;
    {
        const mxArray* f = mxGetField(prhs[3], 0, "Metric");
        char name[16] = "";
        if (f && mxIsChar(f) && mxGetString(f, name, sizeof name) == 0) {
            if (!strcmp(name, "SAD") || !strcmp(name, "sad")) o.metric = PCREG_METRIC_SAD;
            else if (!strcmp(name, "SSD") || !strcmp(name, "ssd")) o.metric = PCREG_METRIC_SSD;
            else { g_fail = "get_matches: par.Metric must be 'SAD' or 'SSD'"; return false; }
        }
    }
    const int64_t n1 = (int64_t)mxGetM(prhs[1]), n2 = (int64_t)mxGetM(prhs[2]), dim = (int64_t)mxGetN(prhs[1]);
    int64_t np = 0;
    int rc;
    {
        std::vector<int32_t> pairs((size_t)(n1 > 0 ? n1 : 1) * 2);
        std::vector<double> mm((size_t)(n1 > 0 ? n1 : 1));
        rc = pcreg_get_matches(mxGetPr(prhs[1]), n1, n1 > 0 ? n1 : 1, mxGetPr(prhs[2]), n2, n2 > 0 ? n2 : 1, dim, &o, pairs.data(), mm.data(), &np);
        if (rc == PCREG_OK) {
            plhs[0] = mxCreateNumericMatrix((mwSize)np, 2, mxUINT32_CLASS, mxREAL);      // indexPairs is uint32 in matchFeatures
            uint32_t* out = (uint32_t*)mxGetData(plhs[0]);
            for (int64_t p = 0; p < np; ++p) { out[p] = (uint32_t)pairs[(size_t)(2 * p)] + 1u; out[np + p] = (uint32_t)pairs[(size_t)(2 * p + 1)] + 1u; }
            if (nlhs > 1) {
                plhs[1] = mxCreateDoubleMatrix((mwSize)np, 1, mxREAL);
                for (int64_t p = 0; p < np; ++p) mxGetPr(plhs[1])[p] = mm[(size_t)p];
            }
        }
    }
    if (rc != PCREG_OK) { g_fail = pcreg_last_error(); return false; }
    return true;
}

bool cmd_icp(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    pcreg_model* m = nrhs > 1 ? handle_of(prhs[1]) : nullptr;
    if (!m || nrhs < 5 || !is_pts(prhs[2]) || !mxIsDouble(prhs[3]) || mxGetNumberOfElements(prhs[3]) % 16 != 0) {
        g_fail = "icp: need (handle, src Nx3, T0 4x4xH double, opts struct[, w_src])";
        return false;
    }
    const pcreg_icp_opts o = icp_opts_of(prhs[4]);
    const int64_t ns = (int64_t)mxGetM(prhs[2]);
    const int64_t H = (int64_t)(mxGetNumberOfElements(prhs[3]) / 16);
    const double* w = (nrhs > 5 && mxIsDouble(prhs[5]) && (int64_t)mxGetNumberOfElements(prhs[5]) == ns) ? mxGetPr(prhs[5]) : nullptr;
    mxArray* T = mxCreateDoubleMatrix(16, (mwSize)H, mxREAL);            // reshaped to 4x4xH by the .m shim
    mxArray* rmse = mxCreateDoubleMatrix((mwSize)H, 1, mxREAL);
    mxArray* nu = mxCreateNumericMatrix((mwSize)H, 1, mxINT32_CLASS, mxREAL);
    mxArray* st = mxCreateNumericMatrix((mwSize)H, 1, mxINT32_CLASS, mxREAL);
    mxArray* idx = (nlhs > 5) ? mxCreateNumericMatrix((mwSize)ns, (mwSize)H, mxINT32_CLASS, mxREAL) : nullptr;
    int64_t best = -1;
    const int rc = pcreg_icp_batch(m, mxGetData(prhs[2]), mxIsDouble(prhs[2]), ns, ns, w, mxGetPr(prhs[3]), H, &o, mxGetPr(T), mxGetPr(rmse),
                                   (int32_t*)mxGetData(nu), (int32_t*)mxGetData(st), idx ? (int32_t*)mxGetData(idx) : nullptr, nullptr, &best);
    if (rc != PCREG_OK) {
        g_fail = pcreg_last_error();
        mxDestroyArray(T); mxDestroyArray(rmse); mxDestroyArray(nu); mxDestroyArray(st); if (idx) mxDestroyArray(idx);
        return false;
    }
    if (idx) { int32_t* p = (int32_t*)mxGetData(idx); for (int64_t i = 0; i < ns * H; ++i) p[i] += 1; }
    plhs[0] = T;
    if (nlhs > 1) plhs[1] = rmse; else mxDestroyArray(rmse);
    if (nlhs > 2) plhs[2] = nu; else mxDestroyArray(nu);
    if (nlhs > 3) plhs[3] = st; else mxDestroyArray(st);
    if (nlhs > 4) plhs[4] = mxCreateDoubleScalar((double)best + 1.0);
    if (nlhs > 5) plhs[5] = idx;
    return true;
}

}  // namespace

extern "C" void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    g_fail.clear();
    bool ok = false;
    {
        char cmd[64] = "";
        if (nrhs < 1 || !mxIsChar(prhs[0]) || mxGetString(prhs[0], cmd, sizeof cmd) != 0) {
            g_fail = "pcreg_mex: first argument must be a command string";
        } else if (!strcmp(cmd, "init")) {
            ok = ensure_init(nrhs > 1 ? prhs[1] : nullptr);
            if (ok && nlhs > 0) plhs[0] = empty();
        } else if (!ensure_init(nullptr)) {
            ok = false;
        } else if (!strcmp(cmd, "model_create")) ok = cmd_model_create(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "model_destroy")) { pcreg_model_destroy(nrhs > 1 ? handle_of(prhs[1]) : nullptr); ok = true; if (nlhs > 0) plhs[0] = empty(); }
        else if (!strcmp(cmd, "nn_search")) ok = cmd_nn_search(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "quick_tf")) ok = cmd_quick_tf(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "local_points")) ok = cmd_local_points(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "spatial_histogram")) ok = cmd_spatial_histogram(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "align")) ok = cmd_align(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "estimate_transform")) ok = cmd_estimate_transform(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "ransac")) ok = cmd_ransac(nlhs, plhs, nrhs, prhs, false);
        else if (!strcmp(cmd, "ransac_seeded")) ok = cmd_ransac(nlhs, plhs, nrhs, prhs, true);
        else if (!strcmp(cmd, "ransac_batch")) ok = cmd_ransac_batch(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "get_matches")) ok = cmd_get_matches(nlhs, plhs, nrhs, prhs);
        else if (!strcmp(cmd, "icp")) ok = cmd_icp(nlhs, plhs, nrhs, prhs);
        else g_fail = std::string("pcreg_mex: unknown command '") + cmd + "'";
    }
    // every C++ object of the frame above is destroyed; only now may MATLAB long-jump
    if (!ok) mexErrMsgIdAndTxt("pcreg:error", "%s", g_fail.c_str());
}
