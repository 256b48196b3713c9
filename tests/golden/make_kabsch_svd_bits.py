"""Writes tests/golden/kabsch_svd_bits.json: the ICP update's dT (kabsch_from_sums with the ICP rank rule) on updates that must
keep taking svd3 -- rank 2 (planar correspondences), rank <= 1 (collinear, coincident: H at rounding-noise level, three weighted
collinear points), S[2] / S[0] between the rank rule's tau and the polar certificate's bound, and reflection_fix = 1 with
det H < 0 -- as the svd3-only update computed them (the host build of pcreg_math.cuh at commit 75a3772, before polar3).
Inputs (the 17 sums, the pivot) and outputs are stored as float.hex, so the comparison is bit for bit.

    python tests/golden/make_kabsch_svd_bits.py path/to/libhostmath.so
"""
import ctypes as C
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import icp_degenerate as D  # noqa: E402

dp = C.POINTER(C.c_double)


def cases():
    out = []
    for seed in range(4):
        for tilted in (False, True):
            for inplane in (False, True):
                out.append(("planar", D.flat_pair(100 + seed, tilted=tilted, inplane_noise=inplane)))
        out.append(("planar-offset-1e3", D.flat_pair(110 + seed, offset=1e3)))
        out.append(("collinear", D.collinear_pair(120 + seed)))
        out.append(("coincident", D.coincident_pair(130 + seed)))
        out.append(("three-weighted", D.three_weighted_pair(140 + seed)))
        out.append(("between-tau-and-certificate", D.curved_pair(150 + seed, 2e-3, seed % 2 == 1)))
        out.append(("mirrored", D.curved_pair(160 + seed, 1.0, True)))
    return out


def main(lib_path):
    hm = C.CDLL(lib_path)
    hm.hm_kabsch_from_sums_icp.argtypes = [dp, dp, dp, C.c_int, dp]
    rows = []
    for kind, (m, q, w, p) in cases():
        s = np.ascontiguousarray(D.sums17(q, m, w, p))
        p = np.ascontiguousarray(p, dtype=np.float64)
        for refl in ((1,) if kind == "mirrored" else (0, 1)):
            dT = np.empty(16)
            hm.hm_kabsch_from_sums_icp(s.ctypes.data_as(dp), p.ctypes.data_as(dp), p.ctypes.data_as(dp), refl, dT.ctypes.data_as(dp))
            rows.append(dict(kind=kind, refl=refl, sums=[float(v).hex() for v in s], pivot=[float(v).hex() for v in p],
                             dT=[float(v).hex() for v in dT]))
    with open(os.path.join(HERE, "kabsch_svd_bits.json"), "w") as f:
        json.dump(rows, f, indent=0)
    print(len(rows), "updates")


if __name__ == "__main__":
    main(sys.argv[1])
