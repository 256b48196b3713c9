"""The pose covariance and the predicted target registration error without a GPU: the host build of pose_cov_from_sums /
pose_cov_tre (pcreg_b200/csrc/pcreg_math.cuh) against numpy, its degenerate rule, the change of reference point, and the FP64
reference (tests/icp_cov_reference.py) on exact shapes whose free motions are known."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from icp_cov_reference import cov_from_sums, cylinder_shape, plane_shape, pose_covariance, sphere_shape, tre_of  # noqa: E402
from pcreg_b200.build import build_hostmath  # noqa: E402

dp = C.POINTER(C.c_double)


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hm():
    lib = C.CDLL(build_hostmath())
    lib.hm_pose_cov_from_sums.argtypes = [dp, C.c_longlong, dp, dp, dp, dp, dp]
    lib.hm_pose_cov_from_sums.restype = C.c_int
    lib.hm_pose_cov_tre.argtypes = [dp, dp, dp]
    lib.hm_pose_cov_tre.restype = C.c_double
    return lib


def _sums(A, B, S):
    s = np.zeros(29)
    s[0] = S
    s[1:22] = A[np.triu_indices(6)]
    s[22] = B
    return s


def _host(hm, s, n_used, pivot, ref):
    cov, info, s2 = np.empty(36), np.empty(36), np.empty(1)
    st = hm.hm_pose_cov_from_sums(_p(s), n_used, _p(np.asarray(pivot, dtype=np.float64)), _p(np.asarray(ref, dtype=np.float64)),
                                  _p(cov), _p(info), _p(s2))
    return cov.reshape(6, 6), info.reshape(6, 6), s2[0], st


def _problem(g, n=400):
    """Sums of n random correspondences about a pivot p (patch 20 mm wide, 150 mm from the origin, random normals)."""
    p = g.uniform(-150, 150, 3)
    qt = g.normal(0, 10, (n, 3))
    nrm = g.normal(size=(n, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    w = g.uniform(0.2, 1.5, n)
    a = np.hstack([np.cross(qt, nrm), nrm])
    b = g.normal(0, 0.3, n)
    return (w[:, None] * a).T @ a, float((w * b * b).sum()), float(w.sum()), n, p, qt, nrm, w


def test_covariance_matches_numpy_inverse(hm):
    g = np.random.default_rng(0)
    for _ in range(50):
        A, B, S, n, p, *_ = _problem(g)
        ref = g.uniform(-200, 200, 3)
        cov, info, s2, st = _host(hm, _sums(A, B, S), n, p, ref)
        cr, ir, s2r, str_ = cov_from_sums(A, B, S, n, p, ref)
        assert st == 0 and str_ == 0
        assert abs(s2 - s2r) <= 1e-14 * s2r
        assert np.max(np.abs(cov - cr)) <= 1e-12 * np.max(np.abs(cr))
        assert np.max(np.abs(info - ir)) <= 1e-12 * np.max(np.abs(ir))
        assert np.array_equal(cov, cov.T)


def test_singular_and_near_singular_give_status_1(hm):
    g = np.random.default_rng(1)
    A, B, S, n, p, qt, nrm, w = _problem(g)
    for flat in (np.tile([0.0, 0.0, 1.0], (n, 1)), None):
        if flat is not None:                       # every normal along z: rank 3
            a = np.hstack([np.cross(qt, flat), flat])
        else:                                      # one direction scaled down to 1e-7 of the others: a pivot below 1e-12 max A_kk
            a = np.hstack([np.cross(qt, nrm), nrm]) @ np.diag([1, 1, 1, 1, 1, 1e-7])
        As = (w[:, None] * a).T @ a
        cov, info, s2, st = _host(hm, _sums(As, B, S), n, p, np.zeros(3))
        assert st == 1 and np.all(np.isnan(cov)) and np.isfinite(s2) and np.all(np.isfinite(info))
    for n_used in (0, 6):
        cov, info, s2, st = _host(hm, _sums(A, B, S), n_used, p, np.zeros(3))
        assert st == 1 and np.all(np.isnan(cov)) and np.isnan(s2)
        assert np.all(np.isnan(info)) == (n_used == 0)
    cov, _, s2, st = _host(hm, _sums(A, B, 0.0), n, p, np.zeros(3))
    assert st == 1 and np.isnan(s2)


def test_reference_point_change_equals_direct_sums_at_that_point(hm):
    """Sums about the pivot moved to ref = the sums taken about ref directly (a = ((q - ref) x n, n))."""
    g = np.random.default_rng(2)
    for _ in range(20):
        A, B, S, n, p, qt, nrm, w = _problem(g)
        ref = g.uniform(-200, 200, 3)
        q_ref = qt + p - ref
        a = np.hstack([np.cross(q_ref, nrm), nrm])
        A_ref = (w[:, None] * a).T @ a
        cov, info, _, _ = _host(hm, _sums(A, B, S), n, p, ref)
        cov_d, info_d, _, _ = _host(hm, _sums(A_ref, B, S), n, ref, ref)
        assert np.max(np.abs(cov - cov_d)) <= 1e-9 * np.max(np.abs(cov_d))
        assert np.max(np.abs(info - info_d)) <= 1e-9 * np.max(np.abs(info_d))


def test_tre_does_not_depend_on_ref(hm):
    g = np.random.default_rng(3)
    for _ in range(20):
        A, B, S, n, p, *_ = _problem(g)
        xs = g.uniform(-200, 200, (5, 3))
        tres = []
        for ref in (np.zeros(3), p, g.uniform(-300, 300, 3)):
            cov, _, _, _ = _host(hm, _sums(A, B, S), n, p, ref)
            tres.append([hm.hm_pose_cov_tre(_p(cov.ravel().copy()), _p(ref), _p(x.copy())) for x in xs])
            assert np.allclose(tres[-1], tre_of(cov, ref, xs), rtol=1e-12, atol=0)
        assert np.max(np.abs(np.array(tres) - tres[0]) / np.array(tres[0])) <= 1e-12


def _null_space(info, tol=1e-10):
    w, V = np.linalg.eigh(info)
    return V[:, w <= tol * w.max()]


def _in_span(N, v):
    v = v / np.linalg.norm(v)
    return np.linalg.norm(v - N @ (N.T @ v)) < 1e-6


@pytest.mark.parametrize("shape,free", [("plane", 3), ("cylinder", 2), ("sphere", 3)])
def test_exact_shapes_leave_their_analytic_free_motions(shape, free):
    """Noise-free source on the model itself (T = I): info's null space is exactly the shape's symmetry motions, and the pass reports
    status 1.  A motion about an axis through c with direction u is (omega, tau) = (u, u x (ref - c))."""
    pts, nrm = {"plane": plane_shape, "cylinder": cylinder_shape, "sphere": sphere_shape}[shape]()
    ref = np.array([1.5, -2.0, 0.5])
    r = pose_covariance(pts, nrm, pts, np.eye(4)[None], ref=ref)
    assert r["status"][0] == 1 and r["n_used"][0] == pts.shape[0]
    N = _null_space(r["info"][0])
    assert N.shape[1] == free
    e = np.eye(3)
    rot = lambda u: np.hstack([u, np.cross(u, ref)])                        # axis through the origin (every shape's centre)
    tr = lambda u: np.hstack([np.zeros(3), u])
    motions = {"plane": [tr(e[0]), tr(e[1]), rot(e[2])], "cylinder": [tr(e[2]), rot(e[2])], "sphere": [rot(e[0]), rot(e[1]), rot(e[2])]}
    for v in motions[shape]:
        assert _in_span(N, v)


def test_constrained_shape_has_full_rank_and_finite_covariance():
    """A noisy patch of an ellipsoid-like bump constrains all six directions: status 0, cov symmetric positive definite."""
    g = np.random.default_rng(4)
    pts, nrm = sphere_shape(3000, 8.0, 5)
    pts = pts * np.array([1.0, 0.8, 0.6])
    nrm = nrm / np.array([1.0, 0.8, 0.6])
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    src = pts[pts[:, 2] > 1.0] + g.normal(0, 0.05, (int((pts[:, 2] > 1.0).sum()), 3))
    r = pose_covariance(pts, nrm, src, np.eye(4)[None], targets=[[0, 0, 5.0], [3, 3, 3]])
    assert r["status"][0] == 0 and np.all(np.linalg.eigvalsh(r["cov"][0]) > 0)
    assert np.all(np.isfinite(r["tre"][0])) and np.all(r["tre"][0] > 0)


def test_abi_declares_the_covariance_entries():
    with open(os.path.join(ROOT, "include", "pcreg.h")) as f:
        hdr = f.read()
    for name in ("pcreg_icp_covariance", "pcreg_icp_covariance_dev"):
        assert re.search(r"\bint\s+%s\s*\(" % name, hdr)
    from pcreg_b200 import _lib
    assert {"pcreg_icp_covariance", "pcreg_icp_covariance_dev"} <= set(_lib.SIGNATURES)


def test_pose_error_recovers_a_small_perturbation():
    """T = T_gt followed by x -> x + omega x (x - ref) + tau (exact rotation): pose_error returns (omega, tau) to second order."""
    from icp_cov_reference import pose_error
    from pcreg_b200 import synth
    g = np.random.default_rng(6)
    T_gt = synth.make_T(synth.rot_xyz(g.uniform(0, 6, 3)), g.uniform(-50, 50, 3))
    ref = g.uniform(-100, 100, 3)
    om, tau = g.normal(0, 1e-5, 3), g.normal(0, 1e-3, 3)
    R = synth.rot_axis_angle(om, np.linalg.norm(om))       # column-vector rotation by omega
    P = synth.make_T(R.T, ref - ref @ R.T + tau)           # row-vector: x R' = R x
    e = pose_error(T_gt @ P, T_gt, ref)
    assert np.allclose(e, np.hstack([om, tau]), rtol=0, atol=1e-8)
