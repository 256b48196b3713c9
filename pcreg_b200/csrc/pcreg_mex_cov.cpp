// pcreg_mex_cov.cpp -- MEX gateway of the pose covariance and predicted target registration error (pcreg_icp_covariance).  Pure
// marshaling, same conventions as pcreg_mex.cpp (whose 'model_create' makes the handle and initialises the library) and
// pcreg_mex_windows.cpp (the windows layout).
//
// Build (on a host with MATLAB):  mex -R2018a pcreg_mex_cov.cpp -I../../include -L.. -lpcreg_b200
//
//   pcreg_mex_cov(handle, src (N x 3, the windows' rows one after the other), src_offsets ((W+1), 0-based), T (4x4xH, grouped by
//                 window), hyp_offsets ((W+1), 0-based), opts (struct)[, ref (3 or []), targets (K x 3 or []), w_src (N or [])])
//     -> cov (36 x H: each column a 6x6, unknowns (omega, tau), about ref), sigma2 (H), rmse (H), n_used, status (H, int32),
//        tre (H x K), info (36 x H)
#include <string>
#include <vector>

#include "mex.h"
#include "../../include/pcreg.h"
#include "pcreg_mex_util.h"

namespace {

std::string g_fail;                // set instead of throwing; reported after the frame unwinds

bool icp_cov(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    pcreg_model* m = nrhs > 0 ? handle_of(prhs[0]) : nullptr;
    if (!m || nrhs < 6 || !is_pts(prhs[1]) || !mxIsDouble(prhs[2]) || !mxIsDouble(prhs[3]) || mxGetNumberOfElements(prhs[3]) % 16 != 0 ||
        !mxIsDouble(prhs[4]) || mxGetNumberOfElements(prhs[2]) < 2 || mxGetNumberOfElements(prhs[4]) != mxGetNumberOfElements(prhs[2])) {
        g_fail = "pcreg_mex_cov: need (handle, src Nx3, src_offsets (W+1), T 4x4xH double, hyp_offsets (W+1), opts struct[, ref, targets, w_src])";
        return false;
    }
    const pcreg_icp_opts o = icp_opts_of(prhs[5]);
    const int64_t N = (int64_t)mxGetM(prhs[1]);
    const int64_t W = (int64_t)mxGetNumberOfElements(prhs[2]) - 1;
    const int64_t H = (int64_t)(mxGetNumberOfElements(prhs[3]) / 16);
    std::vector<int64_t> soff((size_t)W + 1), hoff((size_t)W + 1);
    for (int64_t w = 0; w <= W; ++w) { soff[(size_t)w] = (int64_t)mxGetPr(prhs[2])[w]; hoff[(size_t)w] = (int64_t)mxGetPr(prhs[4])[w]; }
    if (soff[(size_t)W] != N || hoff[(size_t)W] != H) { g_fail = "pcreg_mex_cov: the offsets must end at size(src,1) / the number of poses"; return false; }
    const mxArray* a_ref = nrhs > 6 ? prhs[6] : nullptr;
    const mxArray* a_tg = nrhs > 7 ? prhs[7] : nullptr;
    const mxArray* a_w = nrhs > 8 ? prhs[8] : nullptr;
    if ((a_ref && !mxIsEmpty(a_ref) && (!mxIsDouble(a_ref) || mxGetNumberOfElements(a_ref) != 3)) ||
        (a_tg && !mxIsEmpty(a_tg) && (!mxIsDouble(a_tg) || mxGetN(a_tg) != 3)) ||
        (a_w && !mxIsEmpty(a_w) && (!mxIsDouble(a_w) || (int64_t)mxGetNumberOfElements(a_w) != N))) {
        g_fail = "pcreg_mex_cov: ref must be 3 doubles, targets K x 3 double, w_src N doubles (or [])";
        return false;
    }
    const double* ref = (a_ref && !mxIsEmpty(a_ref)) ? mxGetPr(a_ref) : nullptr;
    const int64_t K = (a_tg && !mxIsEmpty(a_tg)) ? (int64_t)mxGetM(a_tg) : 0;
    const double* wsrc = (a_w && !mxIsEmpty(a_w)) ? mxGetPr(a_w) : nullptr;
    mxArray* cov = mxCreateDoubleMatrix(36, (mwSize)H, mxREAL);
    mxArray* s2 = mxCreateDoubleMatrix((mwSize)H, 1, mxREAL);
    mxArray* rmse = mxCreateDoubleMatrix((mwSize)H, 1, mxREAL);
    mxArray* nu = mxCreateNumericMatrix((mwSize)H, 1, mxINT32_CLASS, mxREAL);
    mxArray* st = mxCreateNumericMatrix((mwSize)H, 1, mxINT32_CLASS, mxREAL);
    mxArray* info = (nlhs > 6) ? mxCreateDoubleMatrix(36, (mwSize)H, mxREAL) : nullptr;
    std::vector<double> tre_hk((size_t)(H * K));                   // [H][K] from the library, H x K column-major for MATLAB
    const int rc = pcreg_icp_covariance(m, mxGetData(prhs[1]), mxIsDouble(prhs[1]), N > 0 ? N : 1, soff.data(), wsrc, hoff.data(), W,
                                        mxGetPr(prhs[3]), &o, ref, K ? mxGetPr(a_tg) : nullptr, K, mxGetPr(cov), info ? mxGetPr(info) : nullptr,
                                        mxGetPr(s2), mxGetPr(rmse), (int32_t*)mxGetData(nu), (int32_t*)mxGetData(st),
                                        K ? tre_hk.data() : nullptr);
    if (rc != PCREG_OK) {
        g_fail = pcreg_last_error();
        mxDestroyArray(cov); mxDestroyArray(s2); mxDestroyArray(rmse); mxDestroyArray(nu); mxDestroyArray(st); if (info) mxDestroyArray(info);
        return false;
    }
    plhs[0] = cov;
    if (nlhs > 1) plhs[1] = s2; else mxDestroyArray(s2);
    if (nlhs > 2) plhs[2] = rmse; else mxDestroyArray(rmse);
    if (nlhs > 3) plhs[3] = nu; else mxDestroyArray(nu);
    if (nlhs > 4) plhs[4] = st; else mxDestroyArray(st);
    if (nlhs > 5) {
        plhs[5] = mxCreateDoubleMatrix((mwSize)H, (mwSize)K, mxREAL);
        for (int64_t h = 0; h < H; ++h)
            for (int64_t k = 0; k < K; ++k) mxGetPr(plhs[5])[k * H + h] = tre_hk[(size_t)(h * K + k)];
    }
    if (nlhs > 6) plhs[6] = info;
    return true;
}

}  // namespace

extern "C" void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    g_fail.clear();
    const bool ok = icp_cov(nlhs, plhs, nrhs, prhs);
    // every C++ object of the frame above is destroyed; only now may MATLAB long-jump
    if (!ok) mexErrMsgIdAndTxt("pcreg:error", "%s", g_fail.c_str());
}
