"""The ICP pose extrapolation without a GPU: the host build of its arithmetic (pcreg_b200/csrc/pcreg_math.cuh: rot_to_quat,
quat_to_rot, pose_state, the two fits, the branch table, sums_mse_at, extrap_step) against numpy / scipy, the ctypes layout of
pcreg_icp_extrap, and the FP64 reference (tests/icp_extrap_reference.py): without the step it is the oracle's loop, it is causal,
and on a seeded problem it is measured against the 50-update loop without extrapolation."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from icp_extrap_reference import BRANCH_NONE, BRANCH_V1, BRANCH_V2, BRANCH_VMAX, branch, icp_single_extrap, pose_state  # noqa: E402
from oracle.icp import _weighted_kabsch  # noqa: E402
from oracle.nn import KDTreeNN  # noqa: E402
from oracle.primitives import quickTF  # noqa: E402
from pcreg_b200 import synth  # noqa: E402
from pcreg_b200.build import build_hostmath  # noqa: E402

dp = C.POINTER(C.c_double)


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hm():
    lib = C.CDLL(build_hostmath())
    for n, args, res in (("hm_rot_to_quat", [dp, dp], None), ("hm_quat_to_rot", [dp, dp], None), ("hm_pose_state", [dp, dp, dp, dp], None),
                         ("hm_line_zero", [dp, dp], C.c_double), ("hm_parabola_vertex", [dp, dp], C.c_double),
                         ("hm_extrap_branch", [C.c_double, C.c_double, C.c_double, dp], C.c_int),
                         ("hm_sums_mse_at", [dp, dp, dp, dp], C.c_double),
                         ("hm_extrap_step", [C.c_double, C.c_double, dp, dp, dp, dp, dp, C.c_int, dp, dp], C.c_int),
                         ("hm_extrap_state_len", [], C.c_int)):
        getattr(lib, n).argtypes = args
        getattr(lib, n).restype = res
    return lib


def _T(R, t):
    T = np.eye(4)
    T[:3, :3] = R
    T[3, :3] = t
    return T


def test_quaternion_round_trip_and_sign(hm):
    g = np.random.default_rng(5)
    Rs = list(Rotation.random(200, random_state=7).as_matrix())
    # every Shepperd branch: near-identity, and half-turns about each axis (trace -1, one diagonal entry 1)
    Rs += [np.eye(3), Rotation.from_rotvec([1e-9, 0, 0]).as_matrix()] + [Rotation.from_rotvec(np.pi * np.eye(3)[k]).as_matrix() for k in range(3)]
    for R in Rs:
        T = _T(R, g.normal(0, 50, 3))
        q = np.zeros(4)
        hm.hm_rot_to_quat(_p(T), _p(q))
        assert abs(np.linalg.norm(q) - 1.0) < 1e-14
        x, y, z, w = Rotation.from_matrix(R).as_quat()
        assert min(np.abs(q - [w, x, y, z]).max(), np.abs(q + [w, x, y, z]).max()) < 1e-13
        T2 = np.zeros(16)
        hm.hm_quat_to_rot(_p(q), _p(T2))
        assert np.abs(T2.reshape(4, 4)[:3, :3] - R).max() < 1e-14
    c = np.array([40.0, -3.0, 12.0])
    # first state: w >= 0, at w = 0 the first nonzero component positive; later ones follow the previous quaternion
    for R in (Rotation.from_rotvec([0, 0, 3.0]).as_matrix(), Rotation.from_rotvec(np.pi * np.array([0.0, -1.0, 0.0])).as_matrix()):
        T = _T(R, [1.0, 2.0, 3.0])
        x = np.zeros(7)
        hm.hm_pose_state(_p(T), _p(c), None, _p(x))
        assert x[0] > 0 or (x[0] == 0 and x[np.nonzero(x[:4])[0][0]] > 0)
        np.testing.assert_allclose(x, pose_state(T, c), atol=1e-13)
        np.testing.assert_allclose(x[4:], c @ R + [1.0, 2.0, 3.0], rtol=1e-15)
        qp = -x[:4]
        y = np.zeros(7)
        hm.hm_pose_state(_p(T), _p(c), _p(qp), _p(y))
        assert y[:4] @ qp >= 0 and np.array_equal(y[:4], -x[:4])


def test_fits_match_polyfit(hm):
    g = np.random.default_rng(11)
    for _ in range(200):
        n1, n2 = g.uniform(1e-4, 1.0, 2)
        v = np.array([0.0, -n1, -n1 - n2])
        D = g.uniform(0.01, 1.0, 3)
        a1, b1 = np.polyfit(v, D, 1)
        a2, b2, _ = np.polyfit(v, D, 2)
        assert hm.hm_line_zero(_p(v), _p(D)) == pytest.approx(-b1 / a1, rel=1e-12, abs=1e-12 * n1)
        assert hm.hm_parabola_vertex(_p(v), _p(D)) == pytest.approx(-b2 / (2 * a2), rel=1e-12, abs=1e-12 * n1)


@pytest.mark.parametrize("v1,v2,vmax,want", [
    (2.0, 1.0, 3.0, BRANCH_V2), (4.0, 1.0, 3.0, BRANCH_V2),                         # 0 < v2 < v1 < vmax, 0 < v2 < vmax < v1
    (1.0, 2.0, 3.0, BRANCH_V1), (1.0, 4.0, 3.0, BRANCH_V1), (1.0, -2.0, 3.0, BRANCH_V1),
    (4.0, 5.0, 3.0, BRANCH_VMAX),
    (1.0, 1.0, 3.0, BRANCH_NONE), (3.0, 1.0, 3.0, BRANCH_NONE), (1.0, 3.0, 3.0, BRANCH_NONE),   # ties fail every strict compare
    (3.0, 4.0, 3.0, BRANCH_NONE), (0.0, 1.0, 3.0, BRANCH_NONE), (-1.0, 2.0, 3.0, BRANCH_NONE), (-1.0, -2.0, 3.0, BRANCH_NONE),
    (4.0, -1.0, 3.0, BRANCH_NONE), (1.0, 0.0, 3.0, BRANCH_NONE),
    (math.nan, 1.0, 3.0, BRANCH_NONE), (1.0, math.nan, 3.0, BRANCH_NONE), (math.inf, 4.0, 3.0, BRANCH_VMAX),
    (math.inf, math.inf, 3.0, BRANCH_VMAX), (-math.inf, 1.0, 3.0, BRANCH_NONE), (1.0, -math.inf, 3.0, BRANCH_V1),
    (1.0, math.inf, 3.0, BRANCH_V1), (math.inf, 1.0, 3.0, BRANCH_V2),
])
def test_branch_table(hm, v1, v2, vmax, want):
    dv = C.c_double(-1.0)
    got = hm.hm_extrap_branch(v1, v2, vmax, C.byref(dv))
    assert got == want and branch(v1, v2, vmax)[1] == want
    assert dv.value == {BRANCH_NONE: 0.0, BRANCH_V2: v2, BRANCH_V1: v1, BRANCH_VMAX: vmax}[want]


def _sums(q, m, w, p):
    qt, mt = q - p, m - p
    s = np.zeros(17)
    s[0] = w.sum()
    s[1:4] = w @ qt
    s[4:7] = w @ mt
    s[7:16] = (qt * w[:, None]).T.dot(mt).ravel()
    s[16] = w @ ((m - q) ** 2).sum(axis=1)
    return s


def test_closed_form_error_far_from_the_pivot(hm):
    """d(T) from the 17 sums equals the point-by-point sum for a patch 40 mm from the pivot, poses near and far from the data."""
    g = np.random.default_rng(3)
    p = np.zeros(3)
    for k in range(20):
        src = g.normal(0, 8, (500, 3)) + [40.0, 5.0, -3.0]
        Tc = _T(Rotation.from_rotvec(g.normal(0, 0.3, 3)).as_matrix(), g.normal(0, 5, 3))
        q = src @ Tc[:3, :3] + Tc[3, :3]
        m = q + g.normal(0, 0.05, q.shape)
        w = g.uniform(0, 1, q.shape[0]) * (g.uniform(size=q.shape[0]) > 0.2)
        s = _sums(q, m, w, p)
        for ang in (1e-4, 1e-2, 0.5):
            T = Tc @ _T(Rotation.from_rotvec(g.normal(0, ang, 3)).as_matrix(), g.normal(0, ang, 3))
            direct = float((w * ((m - (src @ T[:3, :3] + T[3, :3])) ** 2).sum(axis=1)).sum() / w.sum())
            got = hm.hm_sums_mse_at(_p(s), _p(p), _p(np.ascontiguousarray(Tc.ravel())), _p(np.ascontiguousarray(T.ravel())))
            assert got == pytest.approx(direct, rel=1e-9), (k, ang)


def test_struct_layout_and_defaults():
    from pcreg_b200 import _lib as L
    from pcreg_b200.build import build_library
    assert C.sizeof(L.IcpExtrap) == 16 and L.IcpExtrap.angle_deg.offset == 0 and L.IcpExtrap.vmax_scale.offset == 8
    lib = C.CDLL(build_library())
    lib.pcreg_icp_extrap_default.argtypes = [C.POINTER(L.IcpExtrap)]
    e = L.IcpExtrap(0.0, 0.0)
    lib.pcreg_icp_extrap_default(C.byref(e))
    assert (e.angle_deg, e.vmax_scale) == (10.0, 25.0)
    from pcreg_b200.api import icp_extrap
    d = icp_extrap()
    assert (d.angle_deg, d.vmax_scale) == (10.0, 25.0)


@pytest.fixture(scope="module")
def prob():
    """A smooth patch well inside the model with 6 poses up to 8 deg / 2 mm off: point-to-point creeps along it."""
    model = synth.make_model(20_000, 100).astype(np.float64)
    src, T_gt, c = synth.make_source(model, 400, 0.3, 101)
    T0 = synth.pose_grid(T_gt, c, 3, (2, 1, 1), 8.0, 2.0, 102)
    return model, src.astype(np.float64), T0, T_gt


def test_disabled_step_is_the_oracle(prob):
    model, src, T0, _ = prob
    nn = KDTreeNN(model)
    for h in range(2):
        ref = oracle.icp_single(model, src, T0[h], mode=oracle.ICP_KNN, iters=8, k_frac=0.85, nn=nn, return_hist=True)
        out = icp_single_extrap(model, src, T0[h], extrapolate=False, mode=oracle.ICP_KNN, iters=8, k_frac=0.85, nn=nn)
        assert np.array_equal(out["T"], ref["T"]) and np.array_equal(out["idx"], ref["idx"]) and out["rmse"] == ref["rmse"]
        assert np.array_equal(out["rmse_hist"], ref["rmse_hist"], equal_nan=True) and out["n_extrap"] == 0


def test_prefix_property(prob):
    """The rule is causal: a run of k updates is the first k updates of a longer one."""
    model, src, T0, _ = prob
    long = icp_single_extrap(model, src, T0[0], mode=oracle.ICP_KNN, iters=12)
    assert long["n_extrap"] > 0
    for k in (3, 5, 9):
        short = icp_single_extrap(model, src, T0[0], mode=oracle.ICP_KNN, iters=k)
        assert np.array_equal(short["T"], long["trace"][k - 1]["T"])
        assert [t["branch"] for t in short["trace"]] == [t["branch"] for t in long["trace"][:k]]
        assert np.array_equal(short["rmse_hist"][:k], long["rmse_hist"][:k])


def test_host_step_follows_the_reference(hm, prob):
    """extrap_step (the kernels' arithmetic, host build) replayed on the reference's own correspondences takes the same decisions."""
    model, src, T0, _ = prob
    out = icp_single_extrap(model, src, T0[1], mode=oracle.ICP_PLAIN, iters=10)
    c = src.mean(axis=0)
    p = np.zeros(3)
    st = np.zeros(hm.hm_extrap_state_len())
    tr = np.zeros(5)
    nn = KDTreeNN(model)
    T = np.array(T0[1], dtype=np.float64)
    seen = 0
    for t in out["trace"]:
        q = quickTF(src, T)
        j, _ = nn.query(q)
        w = np.ones(q.shape[0])
        K = T @ _weighted_kabsch(model[j], q, w, False)
        Tn = np.ascontiguousarray(K.ravel())
        br = hm.hm_extrap_step(10.0, 25.0, _p(_sums(q, model[j], w, p)), _p(p), _p(c), _p(np.ascontiguousarray(T.ravel())), _p(Tn),
                               t["u"], _p(st), _p(tr))
        if t["margin"] > 1e-6:
            assert br == t["branch"], t
            seen += br != BRANCH_NONE
        np.testing.assert_allclose(Tn.reshape(4, 4), t["T"], atol=1e-9)
        T = t["T"]
    assert seen >= 1


def test_seeded_case_against_fifty_plain_updates(prob):
    """Measured, not tuned: on this seeded problem, the update at which the extrapolating loop first reaches the rmse the loop
    without extrapolation has after 50 updates (to 1e-9 relative), per pose.  What it shows: 3 of the 6 poses reach it, after 11,
    31 and 34 updates.  Of the other 3, two settle 0.04-0.05 mm away in a neighbouring minimum whose rmse is 1e-4 higher, and
    one is thrown by a jump into a worse basin (rmse 0.53 against 0.40, 3.5 mm off).  The assertion records that some pose gets
    there in fewer updates, nothing more."""
    model, src, T0, _ = prob
    first = []
    for h in range(T0.shape[0]):
        base = icp_single_extrap(model, src, T0[h], extrapolate=False, mode=oracle.ICP_KNN, iters=50)
        ex = icp_single_extrap(model, src, T0[h], mode=oracle.ICP_KNN, iters=50)
        target = base["rmse"] * (1 + 1e-9)
        hit = np.nonzero(ex["rmse_hist"] <= target)[0]
        first.append(int(hit[0]) if hit.size else None)
    reached = [f for f in first if f is not None]
    print("updates to reach the 50-update rmse with extrapolation:", first)
    assert len(reached) >= 1 and all(f < 50 for f in reached), first
