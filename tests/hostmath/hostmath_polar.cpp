// Host-only C ABI over the ICP update's polar path of pcreg_b200/csrc/pcreg_math.cuh (tests/test_icp_polar_cpu.py).
#include "../../pcreg_b200/csrc/pcreg_math.cuh"

extern "C" {
// step count of polar3 (0: not converged), the path kabsch_rotation took (0: svd3) and the certificate's constants
int hm_polar3(const double* A, double* Q) { return pcreg::polar3(A, Q); }
int hm_kabsch_rotation(const double* H, double f2, int refl, int icp, double* R) { return pcreg::kabsch_rotation(H, f2, refl != 0, icp != 0, R); }
double hm_icp_polar_det_c() { return pcreg::ICP_POLAR_DET_C; }
double hm_icp_polar_noise_f() { return pcreg::ICP_POLAR_NOISE_F; }
}
