// cov_harness.cpp -- runs pcreg_b200/csrc/pcreg_mex_cov.cpp WITHOUT MATLAB and WITHOUT a GPU, on the fake mx runtime and the C-ABI
// stubs of gateway_harness.cpp (included; its own driver is renamed and not run) plus a stub of pcreg_icp_covariance.
// TEST INFRASTRUCTURE (tests/test_mex_gateway_cov.py).
//
// Build + run:  g++ -std=c++17 -I tests/fake_mex tests/fake_mex/cov_harness.cpp pcreg_b200/csrc/pcreg_mex_cov.cpp -o h && ./h
#define main gateway_harness_main
#include "gateway_harness.cpp"
#undef main

static struct {
    pcreg_icp_opts o{}; std::vector<int64_t> soff, hoff; int64_t ld = 0, ntarget = -1;
    bool has_w = false, has_ref = false, has_info = false, has_tre = false; double ref0 = 0.0, tg_last = 0.0;
} V;

extern "C" int pcreg_icp_covariance(const pcreg_model* m, const void*, int, int64_t ld, const int64_t* src_off, const double* w,
                                    const int64_t* hyp_off, int64_t nwin, const double*, const pcreg_icp_opts* o, const double* ref,
                                    const double* targets, int64_t ntarget, double* cov36, double* info36, double* sigma2, double* rmse,
                                    int32_t* n_used, int32_t* status, double* tre) {
    MAYBE_FAIL();
    if (m != HANDLE) return PCREG_ERR_STATE;
    V.o = *o; V.ld = ld; V.has_w = w != nullptr; V.has_ref = ref != nullptr; V.ref0 = ref ? ref[0] : 0.0;
    V.soff.assign(src_off, src_off + nwin + 1); V.hoff.assign(hyp_off, hyp_off + nwin + 1);
    V.ntarget = ntarget; V.has_info = info36 != nullptr; V.has_tre = tre != nullptr;
    V.tg_last = ntarget ? targets[3 * ntarget - 1] : 0.0;
    for (int64_t h = 0; h < hyp_off[nwin]; ++h) {
        for (int k = 0; k < 36; ++k) { cov36[h * 36 + k] = 100.0 * h + k; if (info36) info36[h * 36 + k] = -(double)k; }
        sigma2[h] = 0.5 * (double)(h + 1); rmse[h] = 0.1 * (double)(h + 1); n_used[h] = (int32_t)(10 + h); status[h] = (int32_t)(h % 2);
        for (int64_t k = 0; k < ntarget; ++k) tre[h * ntarget + k] = 10.0 * (double)h + (double)k;     // [H][K]
    }
    return PCREG_OK;
}

int main() {
    mxArray* handle = u64((uint64_t)(uintptr_t)HANDLE);
    mxArray* opts = strct({{"mode", dbl(1, 1, {2})}, {"iters", dbl(1, 1, {20})}, {"nn", dbl(1, 1, {1})}});
    std::vector<double> t(48);
    for (int i = 0; i < 48; ++i) t[i] = i;
    mxArray* soff = dbl(3, 1, {0, 4, 6});
    mxArray* hoff = dbl(3, 1, {0, 2, 3});
    // targets: K = 2 rows, column-major 2 x 3
    { Out o = call(7, {handle, dbl(6, 3), soff, dbl(16, 3, t), hoff, opts, dbl(3, 1, {7, 8, 9}), dbl(2, 3, {1, 2, 3, 4, 5, 6}), dbl(6, 1, {1, 1, 1, 1, 1, 1})});
      CHECK(o.err.empty() && V.o.mode == PCREG_ICP_WEIGHTED && V.o.nn == PCREG_NN_GRID && V.ld == 6 && V.has_w && V.has_ref && V.ref0 == 7.0);
      CHECK(V.soff == std::vector<int64_t>({0, 4, 6}) && V.hoff == std::vector<int64_t>({0, 2, 3}) && V.ntarget == 2 && V.tg_last == 6.0);
      CHECK(V.has_info && V.has_tre);
      CHECK(o.a[0]->m == 36 && o.a[0]->n == 3 && mxGetPr(o.a[0])[36 + 5] == 105.0);
      CHECK(fabs(mxGetPr(o.a[1])[2] - 1.5) < 1e-15 && fabs(mxGetPr(o.a[2])[1] - 0.2) < 1e-15);
      CHECK(o.a[3]->cls == mxINT32_CLASS && ((int32_t*)mxGetData(o.a[3]))[2] == 12 && ((int32_t*)mxGetData(o.a[4]))[1] == 1);
      // tre: H x K column-major from the library's [H][K]
      CHECK(o.a[5]->m == 3 && o.a[5]->n == 2 && mxGetPr(o.a[5])[3 + 2] == 21.0 && mxGetPr(o.a[5])[1] == 10.0);
      CHECK(o.a[6]->m == 36 && mxGetPr(o.a[6])[36 + 4] == -4.0);
      release(o); }
    { Out o = call(1, {handle, dbl(6, 3), soff, dbl(16, 3, t), hoff, opts});
      CHECK(o.err.empty() && !V.has_w && !V.has_ref && V.ntarget == 0 && !V.has_info && !V.has_tre && o.a[0]->n == 3); release(o); }
    { Out o = call(1, {handle, dbl(6, 3), soff, dbl(16, 3, t), hoff, opts, dbl(2, 1, {1, 2})});
      CHECK(o.err.find("ref must be 3 doubles") != std::string::npos); release(o); }
    { Out o = call(1, {handle, dbl(6, 3), dbl(3, 1, {0, 4, 7}), dbl(16, 3, t), hoff, opts});
      CHECK(o.err.find("offsets must end") != std::string::npos); release(o); }
    { Out o = call(1, {dbl(1, 1, {3}), dbl(6, 3), soff, dbl(16, 3, t), hoff, opts});
      CHECK(o.err.find("pcreg_mex_cov: need") != std::string::npos); release(o); }
    { const int live0 = g_live; R.fail_next = 1;
      Out o = call(7, {handle, dbl(6, 3), soff, dbl(16, 3, t), hoff, opts});
      CHECK(o.err.find("stub: device fell over") != std::string::npos && g_live == live0); release(o); }
    CHECK(g_live == 0);                           // every array the gateway created was returned to us or destroyed
    for (mxArray* a : g_inputs) delete a;
    printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "OK", g_checks, g_failed);
    return g_failed ? 1 : 0;
}
