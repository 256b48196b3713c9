// Host-only C ABI over the pose extrapolation of pcreg_b200/csrc/pcreg_math.cuh for the CPU test suite (no GPU needed); linked into
// the same library as hostmath.cpp.
#include "../../pcreg_b200/csrc/pcreg_math.cuh"

extern "C" {
// T: row-major 4x4 (rotation block read / written); q: (w, x, y, z)
void hm_rot_to_quat(const double* T, double* q) { pcreg::rot_to_quat(T, q); }
void hm_quat_to_rot(const double* q, double* T) { pcreg::quat_to_rot(q, T); }
// qprev null: the canonical sign of the first state
void hm_pose_state(const double* T, const double* c, const double* qprev, double* x) { pcreg::pose_state(T, c, qprev, x); }
double hm_line_zero(const double* v, const double* D) { return pcreg::extrap_line_zero(v, D); }
double hm_parabola_vertex(const double* v, const double* D) { return pcreg::extrap_parabola_vertex(v, D); }
int hm_extrap_branch(double v1, double v2, double vmax, double* dv) { return pcreg::extrap_branch(v1, v2, vmax, dv); }
// s: the 17 sums taken at Tc relative to pivot p
double hm_sums_mse_at(const double* s, const double* p, const double* Tc, const double* T) { return pcreg::sums_mse_at(s, p, Tc, T); }
// st: [EXTRAP_STATE], trace: [EXTRAP_NTRACE]
int hm_extrap_step(double angle_deg, double vmax_scale, const double* s, const double* p, const double* c, const double* Tc, double* Tn,
                   int u, double* st, double* trace) {
    return pcreg::extrap_step(angle_deg, vmax_scale, s, p, c, Tc, Tn, u, st, trace);
}
int hm_extrap_state_len() { return pcreg::EXTRAP_STATE; }
}
