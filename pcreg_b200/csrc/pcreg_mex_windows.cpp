// pcreg_mex_windows.cpp -- MEX gateway of the ICP over many matching windows in one call (pcreg_icp_batch_windows).  Pure
// marshaling, same conventions as pcreg_mex.cpp (whose 'model_create' makes the handle and initialises the library).
//
// Build (on a host with MATLAB):  mex -R2018a pcreg_mex_windows.cpp -I../../include -L.. -lpcreg_b200
//
//   pcreg_mex_windows(handle, src (N x 3, the windows' rows one after the other), src_offsets ((W+1), 0-based),
//                     T0 (4x4xH, grouped by window), hyp_offsets ((W+1), 0-based), opts (struct)[, w_src (N)])
//     -> T (16 x H), rmse (H), n_used, status, best (W, 1-based within the window, 0 where it has no hypothesis),
//        idx (sum_w H_w N_w x 1, window-major, 1-based within the window)
// Point-to-point without a stop, the scope of pcreg_mex('icp', ...).
#include <string>
#include <vector>

#include "mex.h"
#include "../../include/pcreg.h"
#include "pcreg_mex_util.h"

namespace {

std::string g_fail;                // set instead of throwing; reported after the frame unwinds

bool icp_windows(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    pcreg_model* m = nrhs > 0 ? handle_of(prhs[0]) : nullptr;
    if (!m || nrhs < 6 || !is_pts(prhs[1]) || !mxIsDouble(prhs[2]) || !mxIsDouble(prhs[3]) || mxGetNumberOfElements(prhs[3]) % 16 != 0 ||
        !mxIsDouble(prhs[4]) || mxGetNumberOfElements(prhs[2]) < 2 || mxGetNumberOfElements(prhs[4]) != mxGetNumberOfElements(prhs[2])) {
        g_fail = "pcreg_mex_windows: need (handle, src Nx3, src_offsets (W+1), T0 4x4xH double, hyp_offsets (W+1), opts struct[, w_src])";
        return false;
    }
    const pcreg_icp_opts o = icp_opts_of(prhs[5]);
    const int64_t N = (int64_t)mxGetM(prhs[1]);
    const int64_t W = (int64_t)mxGetNumberOfElements(prhs[2]) - 1;
    const int64_t H = (int64_t)(mxGetNumberOfElements(prhs[3]) / 16);
    std::vector<int64_t> soff((size_t)W + 1), hoff((size_t)W + 1), best((size_t)W);
    for (int64_t w = 0; w <= W; ++w) { soff[(size_t)w] = (int64_t)mxGetPr(prhs[2])[w]; hoff[(size_t)w] = (int64_t)mxGetPr(prhs[4])[w]; }
    if (soff[(size_t)W] != N || hoff[(size_t)W] != H) { g_fail = "pcreg_mex_windows: the offsets must end at size(src,1) / the number of poses"; return false; }
    int64_t nidx = 0;
    for (int64_t w = 0; w < W; ++w) nidx += (hoff[(size_t)w + 1] - hoff[(size_t)w]) * (soff[(size_t)w + 1] - soff[(size_t)w]);
    const double* wsrc = (nrhs > 6 && mxIsDouble(prhs[6]) && (int64_t)mxGetNumberOfElements(prhs[6]) == N) ? mxGetPr(prhs[6]) : nullptr;
    mxArray* T = mxCreateDoubleMatrix(16, (mwSize)H, mxREAL);            // reshaped per window by the .m shim
    mxArray* rmse = mxCreateDoubleMatrix((mwSize)H, 1, mxREAL);
    mxArray* nu = mxCreateNumericMatrix((mwSize)H, 1, mxINT32_CLASS, mxREAL);
    mxArray* st = mxCreateNumericMatrix((mwSize)H, 1, mxINT32_CLASS, mxREAL);
    mxArray* idx = (nlhs > 5) ? mxCreateNumericMatrix((mwSize)nidx, 1, mxINT32_CLASS, mxREAL) : nullptr;
    const int rc = pcreg_icp_batch_windows(m, mxGetData(prhs[1]), mxIsDouble(prhs[1]), N > 0 ? N : 1, soff.data(), wsrc, nullptr, 0.0, hoff.data(), W,
                                           mxGetPr(prhs[3]), &o, PCREG_ICP_POINT_TO_POINT, nullptr, mxGetPr(T), mxGetPr(rmse),
                                           (int32_t*)mxGetData(nu), (int32_t*)mxGetData(st), idx ? (int32_t*)mxGetData(idx) : nullptr, nullptr,
                                           best.data(), nullptr, nullptr);
    if (rc != PCREG_OK) {
        g_fail = pcreg_last_error();
        mxDestroyArray(T); mxDestroyArray(rmse); mxDestroyArray(nu); mxDestroyArray(st); if (idx) mxDestroyArray(idx);
        return false;
    }
    if (idx) { int32_t* p = (int32_t*)mxGetData(idx); for (int64_t i = 0; i < nidx; ++i) p[i] += 1; }
    plhs[0] = T;
    if (nlhs > 1) plhs[1] = rmse; else mxDestroyArray(rmse);
    if (nlhs > 2) plhs[2] = nu; else mxDestroyArray(nu);
    if (nlhs > 3) plhs[3] = st; else mxDestroyArray(st);
    if (nlhs > 4) {
        plhs[4] = mxCreateDoubleMatrix((mwSize)W, 1, mxREAL);
        for (int64_t w = 0; w < W; ++w) mxGetPr(plhs[4])[w] = (double)best[(size_t)w] + 1.0;
    }
    if (nlhs > 5) plhs[5] = idx;
    return true;
}

}  // namespace

extern "C" void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    g_fail.clear();
    const bool ok = icp_windows(nlhs, plhs, nrhs, prhs);
    // every C++ object of the frame above is destroyed; only now may MATLAB long-jump
    if (!ok) mexErrMsgIdAndTxt("pcreg:error", "%s", g_fail.c_str());
}
