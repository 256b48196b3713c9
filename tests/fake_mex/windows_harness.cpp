// windows_harness.cpp -- runs pcreg_b200/csrc/pcreg_mex_windows.cpp WITHOUT MATLAB and WITHOUT a GPU, on the fake mx runtime and
// the C-ABI stubs of gateway_harness.cpp (included; its own driver is renamed and not run) plus a stub of pcreg_icp_batch_windows.
// TEST INFRASTRUCTURE (tests/test_mex_gateway_windows.py).
//
// Build + run:  g++ -std=c++17 -I tests/fake_mex tests/fake_mex/windows_harness.cpp pcreg_b200/csrc/pcreg_mex_windows.cpp -o h && ./h
#define main gateway_harness_main
#include "gateway_harness.cpp"
#undef main

static struct {
    pcreg_icp_opts o{}; std::vector<int64_t> soff, hoff; int metric = -1; int64_t ld = 0;
    bool has_w = false, has_idx = false, has_stop = true, has_nrm = true;
} W;

extern "C" int pcreg_icp_batch_windows(const pcreg_model* m, const void*, int, int64_t ld, const int64_t* src_off, const double* w, const void* src_nrm,
                                       double, const int64_t* hyp_off, int64_t nwin, const double* T0, const pcreg_icp_opts* o, int metric,
                                       const pcreg_icp_stop* stop, double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx,
                                       double*, int64_t* best, int32_t*, int32_t*) {
    MAYBE_FAIL();
    if (m != HANDLE) return PCREG_ERR_STATE;
    W.o = *o; W.has_w = w != nullptr; W.has_idx = idx != nullptr;
    W.soff.assign(src_off, src_off + nwin + 1); W.hoff.assign(hyp_off, hyp_off + nwin + 1);
    W.metric = metric; W.ld = ld; W.has_stop = stop != nullptr; W.has_nrm = src_nrm != nullptr;
    int64_t i = 0;
    for (int64_t k = 0; k < nwin; ++k) {
        const int64_t ns = src_off[k + 1] - src_off[k];
        best[k] = hyp_off[k + 1] > hyp_off[k] ? hyp_off[k + 1] - hyp_off[k] - 1 : -1;      // the window's last hypothesis
        for (int64_t h = hyp_off[k]; h < hyp_off[k + 1]; ++h) {
            for (int c = 0; c < 16; ++c) T16[h * 16 + c] = T0[h * 16 + c] + 1.0;
            rmse[h] = 0.1 * (double)(h + 1); n_used[h] = (int32_t)(ns - (h - hyp_off[k])); status[h] = (int32_t)k;
            if (idx) for (int64_t r = 0; r < ns; ++r) idx[i++] = (int32_t)r;           // 0-based within the window
        }
    }
    return PCREG_OK;
}

int main() {
    mxArray* handle = u64((uint64_t)(uintptr_t)HANDLE);
    mxArray* opts = strct({{"mode", dbl(1, 1, {1})}, {"iters", dbl(1, 1, {20})}});
    std::vector<double> t0(48);
    for (int i = 0; i < 48; ++i) t0[i] = i;
    // three windows: 2 rows / 2 poses, 3 rows / no pose, 1 row / 1 pose
    mxArray* soff = dbl(4, 1, {0, 2, 5, 6});
    mxArray* hoff = dbl(4, 1, {0, 2, 2, 3});
    { Out o = call(6, {handle, dbl(6, 3), soff, dbl(16, 3, t0), hoff, opts, dbl(6, 1, {1, 1, 1, 1, 1, 1})});
      CHECK(o.err.empty() && W.o.mode == PCREG_ICP_KNN && W.o.iters == 20 && W.o.nn == PCREG_NN_BRUTE && W.o.k_frac == 0.85);
      CHECK(W.metric == PCREG_ICP_POINT_TO_POINT && !W.has_stop && !W.has_nrm && W.has_w && W.has_idx && W.ld == 6);
      CHECK(W.soff == std::vector<int64_t>({0, 2, 5, 6}) && W.hoff == std::vector<int64_t>({0, 2, 2, 3}));
      CHECK(o.a[0]->m == 16 && o.a[0]->n == 3 && mxGetPr(o.a[0])[33] == 34.0 && fabs(mxGetPr(o.a[1])[2] - 0.3) < 1e-15);
      CHECK(o.a[2]->cls == mxINT32_CLASS && ((int32_t*)mxGetData(o.a[2]))[1] == 1 && ((int32_t*)mxGetData(o.a[3]))[2] == 2);
      // best: 1-based within the window, 0 for the window without hypotheses
      CHECK(o.a[4]->m == 3 && mxGetPr(o.a[4])[0] == 2.0 && mxGetPr(o.a[4])[1] == 0.0 && mxGetPr(o.a[4])[2] == 1.0);
      // idx: window 0's two 2-row blocks, then window 2's 1-row block, 1-based
      const int32_t* ix = o.a[5] ? (const int32_t*)mxGetData(o.a[5]) : nullptr;
      CHECK(ix && o.a[5]->m == 5 && o.a[5]->n == 1 && ix[0] == 1 && ix[1] == 2 && ix[2] == 1 && ix[3] == 2 && ix[4] == 1);
      release(o); }
    { Out o = call(1, {handle, dbl(6, 3), soff, dbl(16, 3, t0), hoff, opts});
      CHECK(o.err.empty() && !W.has_w && !W.has_idx && o.a[0]->n == 3); release(o); }
    { Out o = call(1, {handle, dbl(6, 3), dbl(4, 1, {0, 2, 5, 7}), dbl(16, 3, t0), hoff, opts});
      CHECK(o.err.find("offsets must end") != std::string::npos); release(o); }
    { Out o = call(1, {handle, dbl(6, 3), dbl(3, 1, {0, 2, 6}), dbl(16, 3, t0), hoff, opts});
      CHECK(o.err.find("pcreg_mex_windows: need") != std::string::npos); release(o); }
    { Out o = call(1, {dbl(1, 1, {3}), dbl(6, 3), soff, dbl(16, 3, t0), hoff, opts});
      CHECK(o.err.find("pcreg_mex_windows: need") != std::string::npos); release(o); }
    { const int live0 = g_live; R.fail_next = 1;
      Out o = call(6, {handle, dbl(6, 3), soff, dbl(16, 3, t0), hoff, opts});
      CHECK(o.err.find("stub: device fell over") != std::string::npos && g_live == live0); release(o); }
    CHECK(g_live == 0);                           // every array the gateway created was returned to us or destroyed
    for (mxArray* a : g_inputs) delete a;
    printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "OK", g_checks, g_failed);
    return g_failed ? 1 : 0;
}
