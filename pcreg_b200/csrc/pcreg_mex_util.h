// pcreg_mex_util.h -- argument helpers shared by the MEX gateways (pcreg_mex.cpp, pcreg_mex_windows.cpp, pcreg_mex_cov.cpp).
#pragma once
#include <stdint.h>

#include "mex.h"
#include "../../include/pcreg.h"

inline bool is_pts(const mxArray* a) { return a && (mxIsDouble(a) || mxIsSingle(a)) && !mxIsComplex(a) && mxGetN(a) == 3; }
inline double field_or(const mxArray* s, const char* name, double dflt) {
    if (!s || !mxIsStruct(s)) return dflt;
    const mxArray* f = mxGetField(s, 0, name);
    return (f && !mxIsEmpty(f)) ? mxGetScalar(f) : dflt;
}
// the model handle travels as a uint64 scalar
inline pcreg_model* handle_of(const mxArray* a) {
    if (!a || mxGetClassID(a) != mxUINT64_CLASS || mxGetNumberOfElements(a) != 1) return nullptr;
    return (pcreg_model*)(uintptr_t)(*(const uint64_t*)mxGetData(a));
}
// the ICP options struct (fields mode, iters, k_frac, R_w, thDist2, nn, reflection_fix) over the library defaults
inline pcreg_icp_opts icp_opts_of(const mxArray* s) {
    pcreg_icp_opts o;
    pcreg_icp_opts_default(&o);
    o.mode = (int)field_or(s, "mode", o.mode);
    o.iters = (int)field_or(s, "iters", o.iters);
    o.k_frac = field_or(s, "k_frac", o.k_frac);
    o.R_w = field_or(s, "R_w", o.R_w);
    o.thDist2 = field_or(s, "thDist2", o.thDist2);
    o.nn = (int)field_or(s, "nn", o.nn);
    o.reflection_fix = (int)field_or(s, "reflection_fix", 0);
    return o;
}
