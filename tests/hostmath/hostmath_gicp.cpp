// Host-only C ABI over the plane-to-plane accumulation of pcreg_b200/csrc/pcreg_math.cuh for the CPU test suite (no GPU needed);
// linked into the same library as hostmath.cpp.
#include "../../pcreg_b200/csrc/pcreg_math.cuh"

extern "C" {
// s: the 29 sums (accumulated into); qt, mt: point and model point relative to the pivot; nq, nm: source normal (carried by the
// pose) and model normal
void hm_gicp_accumulate(double* s, double w, double d, const double* qt, const double* mt, const double* nq, const double* nm, double eps) {
    pcreg::gicp_accumulate(s, w, d, qt, mt, nq, nm, eps);
}
}
