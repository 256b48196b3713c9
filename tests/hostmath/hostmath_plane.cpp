// Host-only C ABI over the point-to-plane step of pcreg_b200/csrc/pcreg_math.cuh for the CPU test suite (no GPU needed);
// linked into the same library as hostmath.cpp.
#include "../../pcreg_b200/csrc/pcreg_math.cuh"

extern "C" {
// Au = 21 upper-triangle entries (row-major) of a symmetric 6x6; returns 1 and x, or 0 (degenerate, x untouched)
int hm_ldlt6_solve(const double* Au, const double* g, double* x) { return pcreg::ldlt6_solve(Au, g, x) ? 1 : 0; }
void hm_rodrigues(const double* w, double* R) { pcreg::rodrigues(w, R); }
}
