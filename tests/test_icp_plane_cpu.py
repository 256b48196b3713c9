"""The point-to-plane ICP metric and the model normals without a GPU: the FP64 reference (tests/icp_plane_reference.py) converges
on a smooth model, its degeneracy rule fires on a flat patch, the host build of the LDL' solve and Rodrigues
(pcreg_b200/csrc/pcreg_math.cuh) agrees with numpy, and the C-ABI constants / signatures are declared."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from icp_plane_reference import (ellipsoid_problem, icp_single_plane, knn_exact, ldlt_solve, normals_reference,  # noqa: E402
                                 rodrigues)
from oracle.nn import d2_exact  # noqa: E402
from pcreg_b200.build import build_hostmath  # noqa: E402

dp = C.POINTER(C.c_double)


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hm():
    lib = C.CDLL(build_hostmath())
    lib.hm_ldlt6_solve.argtypes = [dp, dp, dp]
    lib.hm_ldlt6_solve.restype = C.c_int
    lib.hm_rodrigues.argtypes = [dp, dp]
    return lib


def _pose_error(T, T_gt):
    return np.linalg.norm(T[:3, :3] - T_gt[:3, :3], "fro"), np.linalg.norm(T[3, :3] - T_gt[3, :3])


def test_reference_reaches_the_truth_on_a_smooth_model_in_few_updates():
    """Noiseless ellipsoid with analytic normals, start 5 deg / 2 mm from T_gt: within 1e-6 after at most 10 updates, where
    point-to-point is still far from it."""
    model, nrm, src, T_gt, T0 = ellipsoid_problem()
    r = icp_single_plane(model, nrm, src, T0, iters=10)
    assert r["status"] == 0
    errs = [max(_pose_error(T, T_gt)) for T in r["T_hist"]]
    assert errs[0] > 0.05
    assert min(errs) <= 1e-6, errs
    import oracle
    p2p = oracle.icp_single(model, src, T0, iters=10)
    assert max(_pose_error(p2p["T"], T_gt)) > 1e-4


def test_degeneracy_rule_fires_on_a_flat_patch():
    """On a plane the in-plane translation and the rotation about the normal are unconstrained: a pivot of A vanishes."""
    g = np.random.default_rng(3)
    xy = g.uniform(-20, 20, (3000, 2))
    model = np.column_stack([xy, np.zeros(3000)])
    nrm = np.tile([0.0, 0.0, 1.0], (3000, 1))
    src = model[:200] + [0.0, 0.0, 0.5]
    r = icp_single_plane(model, nrm, src, np.eye(4), iters=5)
    assert r["status"] == 1 and r["n_iter"] == 0
    assert np.array_equal(r["T"], np.eye(4))


def _random_spd(g, n=6):
    B = g.normal(size=(n, n))
    return B @ B.T + n * np.eye(n) * 10.0 ** g.uniform(-3, 1)


def _upper(A):
    return np.ascontiguousarray(A[np.triu_indices(6)])


def test_ldlt6_solve_matches_numpy(hm):
    g = np.random.default_rng(11)
    for _ in range(200):
        A = _random_spd(g)
        b = g.normal(size=6)
        x = np.empty(6)
        assert hm.hm_ldlt6_solve(_p(_upper(A)), _p(b), _p(x)) == 1
        xr = np.linalg.solve(A, b)
        assert np.allclose(x, xr, rtol=1e-10, atol=1e-12 * np.abs(xr).max())
        assert np.allclose(ldlt_solve(A, b), xr, rtol=1e-10, atol=1e-12 * np.abs(xr).max())
    # rank-deficient (a flat patch: no constraint along some direction) and zero matrices are degenerate
    for A in (np.diag([1.0, 2.0, 3.0, 4.0, 5.0, 0.0]), np.zeros((6, 6)), np.outer(np.arange(1.0, 7.0), np.arange(1.0, 7.0))):
        x = np.full(6, 7.0)
        assert hm.hm_ldlt6_solve(_p(_upper(A)), _p(np.ones(6)), _p(x)) == 0
        assert np.all(x == 7.0)
        assert ldlt_solve(A, np.ones(6)) is None
    # the threshold: a pivot of exactly 1e-12 max A_kk is degenerate, just above it is not
    A = np.diag([1.0, 1.0, 1.0, 1.0, 1.0, 1e-12])
    assert hm.hm_ldlt6_solve(_p(_upper(A)), _p(np.ones(6)), _p(np.empty(6))) == 0
    A[5, 5] = np.nextafter(1e-12, 1.0)
    assert hm.hm_ldlt6_solve(_p(_upper(A)), _p(np.ones(6)), _p(np.empty(6))) == 1


def test_rodrigues_matches_numpy(hm):
    from scipy.linalg import expm
    g = np.random.default_rng(12)
    for scale in (0.0, 1e-9, 1e-4, 0.1, 1.0, 3.0):
        w = g.normal(size=3) * scale
        R = np.empty((3, 3))
        hm.hm_rodrigues(_p(np.ascontiguousarray(w)), _p(R))
        K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
        assert np.allclose(R, expm(K), rtol=0, atol=1e-14)
        assert np.allclose(R, rodrigues(w), rtol=0, atol=1e-15)
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-14)
    R = np.empty((3, 3))
    hm.hm_rodrigues(_p(np.zeros(3)), _p(R))
    assert np.array_equal(R, np.eye(3))


def test_reference_normals_and_neighbourhoods():
    """knn_exact is the brute-force (d2, index) order; the reference normals of the ellipsoid are close to the analytic ones
    and point outward (no viewpoint) or toward a viewpoint."""
    model, nrm_true, _, _, _ = ellipsoid_problem(n_model=3000)
    nb = knn_exact(model, 6)
    for i in range(0, 3000, 97):
        d = d2_exact(model, model[i])
        assert np.array_equal(nb[i], np.lexsort((np.arange(3000), d))[:6])
    n, w = normals_reference(model, 6)
    assert np.all(w[:, 0] <= w[:, 1])
    assert np.median(np.abs((n * nrm_true).sum(axis=1))) > 0.99
    assert np.all((n * model).sum(axis=1) >= 0)                  # pivot = bbox centre = origin here
    vp = np.array([0.0, 0.0, 500.0])
    nv, _ = normals_reference(model, 6, viewpoint=vp)
    assert np.all(((vp - model) * nv).sum(axis=1) >= 0)
    assert np.allclose(np.abs((nv * n).sum(axis=1)), 1.0)


def test_abi_declares_metric_and_normals():
    from pcreg_b200 import _lib
    with open(os.path.join(ROOT, "include", "pcreg.h")) as f:
        h = f.read()
    assert re.search(r"#define PCREG_ICP_POINT_TO_POINT 0\b", h) and re.search(r"#define PCREG_ICP_POINT_TO_PLANE 1\b", h)
    import pcreg_b200
    assert (pcreg_b200.ICP_POINT_TO_POINT, pcreg_b200.ICP_POINT_TO_PLANE) == (0, 1)
    for name in ("pcreg_model_set_normals", "pcreg_model_compute_normals", "pcreg_model_get_normals", "pcreg_icp_batch_metric",
                 "pcreg_icp_batch_metric_dev"):
        assert name in _lib.SIGNATURES
    # the metric and the stop sit between opts and the outputs; the host entry has 20 arguments, the device entry 19
    res, args = _lib.SIGNATURES["pcreg_icp_batch_metric"]
    assert len(args) == 20 and args[9] is C.c_int and args[10] == C.POINTER(_lib.IcpStop)
    res, args = _lib.SIGNATURES["pcreg_icp_batch_metric_dev"]
    assert len(args) == 19 and args[7] is C.c_int and args[8] == C.POINTER(_lib.IcpStop)
    # the existing option structs keep their layout
    assert C.sizeof(_lib.IcpOpts) == 40 and C.sizeof(_lib.IcpStop) == 24
    from pcreg_b200.build import build_library
    build_library()
    assert _lib.load().pcreg_abi_version() == 2
