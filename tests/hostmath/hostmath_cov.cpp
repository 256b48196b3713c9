// Host-only C ABI over the pose covariance of pcreg_b200/csrc/pcreg_math.cuh for the CPU test suite (no GPU needed); linked into the
// same library as hostmath.cpp.
#include "../../pcreg_b200/csrc/pcreg_math.cuh"

extern "C" {
// s: the 29 sums of a covariance pass; info may be null.  Returns the status (0, or 1: cov NaN).
int hm_pose_cov_from_sums(const double* s, long long n_used, const double* pivot, const double* ref, double* cov, double* info,
                          double* sigma2) {
    return pcreg::pose_cov_from_sums(s, n_used, pivot, ref, cov, info, sigma2);
}
double hm_pose_cov_tre(const double* cov, const double* ref, const double* x) { return pcreg::pose_cov_tre(cov, ref, x); }
}
