// Host-only C ABI over pcreg_b200/csrc/pcreg_math.cuh for the CPU test suite (no GPU needed).
#include "../../pcreg_b200/csrc/pcreg_math.cuh"

extern "C" {
void hm_svd3(const double* A, double* U, double* S, double* V) { pcreg::svd3(A, U, S, V); }
void hm_eigsym3(const double* A, double* w, double* V, int dir) { pcreg::eigsym3(A, w, V); if (dir) pcreg::eigsort3(w, V, dir); }
// sums: sw, sq[3], sm[3], sqm[9], swd2 (17 doubles); pivots [3] each; dT row-major 16
void hm_kabsch_from_sums(const double* s, const double* pq, const double* pm, int refl, double* dT) {
    pcreg::KabschSums k;
    k.sw = s[0];
    for (int i = 0; i < 3; ++i) { k.sq[i] = s[1 + i]; k.sm[i] = s[4 + i]; }
    for (int i = 0; i < 9; ++i) k.sqm[i] = s[7 + i];
    k.swd2 = s[16];
    pcreg::kabsch_from_sums(k, pq, pm, refl != 0, dT);
}
// the same with the ICP update's rank rule (pcreg_math.cuh: ICP_RANK2_TAU)
void hm_kabsch_from_sums_icp(const double* s, const double* pq, const double* pm, int refl, double* dT) {
    pcreg::KabschSums k;
    k.sw = s[0];
    for (int i = 0; i < 3; ++i) { k.sq[i] = s[1 + i]; k.sm[i] = s[4 + i]; }
    for (int i = 0; i < 9; ++i) k.sqm[i] = s[7 + i];
    k.swd2 = s[16];
    pcreg::kabsch_from_sums(k, pq, pm, refl != 0, dT, true);
}
double hm_icp_rank2_tau() { return pcreg::ICP_RANK2_TAU; }
void hm_mul4(const double* A, const double* B, double* C) { pcreg::mul4(A, B, C); }
double hm_spacing(double x) { return pcreg::spacing(x); }
int hm_rank_from_sv(const double* s, long long n) { return pcreg::rank_from_sv(s, n); }
double hm_det3(const double* A) { return pcreg::det3(A); }
}
