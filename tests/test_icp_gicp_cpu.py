"""The plane-to-plane (generalized ICP) metric without a GPU: the host build of its per-correspondence accumulation
(pcreg_b200/csrc/pcreg_math.cuh: gicp_accumulate) equals numpy's J' M J / J' M e and ignores the sign of the normals bit for bit,
eps = 1 is the linearised point-to-point step, and the FP64 reference (tests/icp_gicp_reference.py) converges on a smooth model and
stops after k updates exactly where a k-update run ends."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from icp_gicp_reference import (ellipsoid_gicp_problem, gicp_sums, gicp_update, icp_single_gicp, skew,  # noqa: E402
                                unit_rows)
from icp_plane_reference import ldlt_solve, model_pivot, plane_update  # noqa: E402
from pcreg_b200.build import build_hostmath  # noqa: E402

dp = C.POINTER(C.c_double)
NS = 29


def _p(a):
    return a.ctypes.data_as(dp)


@pytest.fixture(scope="module")
def hm():
    lib = C.CDLL(build_hostmath())
    lib.hm_gicp_accumulate.argtypes = [dp, C.c_double, C.c_double, dp, dp, dp, dp, C.c_double]
    lib.hm_gicp_accumulate.restype = None
    return lib


def _host_sums(hm, qt, mt, nq, nm, w, d, eps):
    s = np.zeros(NS)
    for i in range(qt.shape[0]):
        hm.hm_gicp_accumulate(_p(s), float(w[i]), float(d[i]), _p(np.ascontiguousarray(qt[i])), _p(np.ascontiguousarray(mt[i])),
                              _p(np.ascontiguousarray(nq[i])), _p(np.ascontiguousarray(nm[i])), float(eps))
    return s


def _random_case(g, n):
    qt = g.normal(size=(n, 3)) * 30.0
    mt = qt + g.normal(size=(n, 3))
    nq = unit_rows(g.normal(size=(n, 3)))
    nm = unit_rows(g.normal(size=(n, 3)))
    w = g.uniform(0.0, 2.0, n)
    w[::7] = 0.0
    d = g.uniform(0.0, 4.0, n)
    return qt, mt, nq, nm, w, d


@pytest.mark.parametrize("eps", [1e-3, 0.05, 0.5, 1.0])
def test_host_accumulation_matches_numpy(hm, eps):
    g = np.random.default_rng(21)
    for n in (1, 7, 300):
        qt, mt, nq, nm, w, d = _random_case(g, n)
        s = _host_sums(hm, qt, mt, nq, nm, w, d, eps)
        A, gv = gicp_sums(qt, mt, nq, nm, w, eps)
        assert s[0] == pytest.approx(w.sum(), rel=1e-14) and s[28] == pytest.approx((w * d).sum(), rel=1e-14)
        scale = np.abs(A).max()
        np.testing.assert_allclose(s[1:22], A[np.triu_indices(6)], rtol=1e-9, atol=1e-12 * scale)
        np.testing.assert_allclose(s[22:28], gv, rtol=1e-9, atol=1e-12 * np.abs(gv).max())


def test_host_accumulation_reduces_to_point_to_plane_with_one_plane(hm):
    """The reduction stated in include/pcreg.h: with the information matrix replaced by the rank-one M = n n', J' M J = a a' and
    J' M e = a b for the point-to-plane a = (q~ x n, n) and b = n . e."""
    g = np.random.default_rng(22)
    qt, mt, _, nm, w, _ = _random_case(g, 50)
    Jt = np.concatenate([skew(qt), np.broadcast_to(np.eye(3), (50, 3, 3))], axis=1)
    M = np.einsum("ni,nj->nij", nm, nm)
    A = np.einsum("n,nik,nkl,njl->ij", w, Jt, M, Jt)
    a = np.hstack([np.cross(qt, nm), nm])
    np.testing.assert_allclose(A, (w[:, None] * a).T @ a, rtol=1e-12, atol=1e-9)
    b = ((mt - qt) * nm).sum(axis=1)
    np.testing.assert_allclose(np.einsum("n,nik,nkl,nl->i", w, Jt, M, mt - qt), (w[:, None] * a).T @ b, rtol=1e-12, atol=1e-9)


def test_sign_of_the_normals_changes_no_bit(hm):
    g = np.random.default_rng(23)
    qt, mt, nq, nm, w, d = _random_case(g, 200)
    ref = _host_sums(hm, qt, mt, nq, nm, w, d, 1e-3)
    for _ in range(4):
        fq = np.where(g.random(200) < 0.5, -1.0, 1.0)[:, None]
        fm = np.where(g.random(200) < 0.5, -1.0, 1.0)[:, None]
        out = _host_sums(hm, qt, mt, nq * fq, nm * fm, w, d, 1e-3)
        assert np.array_equal(out, ref)


def test_eps_one_is_the_linearised_point_to_point_step(hm):
    """eps = 1: M = I / 2, so the step solves (sum w J'J) x = sum w J'e, the Gauss-Newton step of sum w |e - J x|^2."""
    g = np.random.default_rng(24)
    qt, mt, nq, nm, w, d = _random_case(g, 400)
    s = _host_sums(hm, qt, mt, nq, nm, w, d, 1.0)
    J = np.concatenate([-skew(qt), np.broadcast_to(np.eye(3), (400, 3, 3))], axis=2)            # [n, 3, 6]: J x = w x q~ + t
    JtJ = np.einsum("n,nki,nkj->ij", w, J, J)
    Jte = np.einsum("n,nki,nk->i", w, J, mt - qt)
    np.testing.assert_allclose(s[1:22], 0.5 * JtJ[np.triu_indices(6)], rtol=1e-12, atol=1e-12 * np.abs(JtJ).max())
    np.testing.assert_allclose(s[22:28], 0.5 * Jte, rtol=1e-12, atol=1e-12 * np.abs(Jte).max())
    # the reference update with eps = 1 is the least-squares solution of the linearised point-to-point problem
    pivot = np.array([1.0, -2.0, 3.0])
    q, m = qt + pivot, mt + pivot
    dT = gicp_update(m, q, nq, nm, w, 400, pivot, 1.0)
    x = np.linalg.lstsq(np.sqrt(w)[:, None, None].repeat(3, 1).reshape(-1, 1) * J.reshape(-1, 6),
                        (np.sqrt(w)[:, None] * (mt - qt)).reshape(-1), rcond=None)[0]
    np.testing.assert_allclose(ldlt_solve(JtJ, Jte), x, rtol=1e-9, atol=1e-12)
    dT2 = gicp_update(m, q, nq, nm, w * 7.0, 400, pivot, 1.0)           # a uniform weight scale does not move the step
    np.testing.assert_allclose(dT, dT2, rtol=0, atol=1e-12)
    assert not np.allclose(dT, gicp_update(m, q, nq, nm, w, 400, pivot, 1e-3), atol=1e-9)


def test_reference_reaches_the_truth_on_a_smooth_model():
    """Noiseless ellipsoid, analytic normals on both sides, start 5 deg / 2 mm off, eps = 1e-3: within 1e-6 after at most 10
    updates, as point-to-plane does."""
    model, nrm, src, sn, T_gt, T0 = ellipsoid_gicp_problem()
    r = icp_single_gicp(model, nrm, src, sn, T0, eps=1e-3, iters=10)
    assert r["status"] == 0
    errs = [max(np.linalg.norm(T[:3, :3] - T_gt[:3, :3], "fro"), np.linalg.norm(T[3, :3] - T_gt[3, :3])) for T in r["T_hist"]]
    assert errs[0] > 0.05
    assert min(errs) <= 1e-6, errs


def test_reference_stop_at_k_equals_a_fixed_k_run():
    model, nrm, src, sn, T_gt, T0 = ellipsoid_gicp_problem(n_model=8000, n_src=300)
    r = icp_single_gicp(model, nrm, src, sn, T0, iters=20, mode=1, tolerance=(0.01, 0.5))
    assert r["converged"] == 1 and 3 <= r["n_iter"] < 20
    k = r["n_iter"]
    f = icp_single_gicp(model, nrm, src, sn, T0, iters=k, mode=1)
    assert np.array_equal(r["T"], f["T"]) and r["rmse"] == f["rmse"] and np.array_equal(r["idx"], f["idx"])
    assert np.array_equal(r["rmse_hist"][:k + 1], f["rmse_hist"])
    assert np.all(r["rmse_hist"][k:] == r["rmse"])


def test_reference_degenerate_flat_patch():
    """Both surfaces one plane: point-to-plane is degenerate there (a pivot of its LDL' solve vanishes), plane-to-plane keeps the
    in-plane directions at eps stiffness and is not; fewer than 6 usable correspondences is degenerate for both."""
    g = np.random.default_rng(3)
    xy = g.uniform(-20, 20, (3000, 2))
    model = np.column_stack([xy, np.zeros(3000)])
    nrm = np.tile([0.0, 0.0, 1.0], (3000, 1))
    src = model[:200] + [0.0, 0.0, 0.5]
    pivot = model_pivot(model)
    w = np.ones(200)
    # M = diag(1/2, 1/2, 1/(2 eps)): the in-plane directions are eps times as stiff as the normal one, weak but not degenerate
    assert gicp_update(model[:200], src, nrm[:200], nrm[:200], w, 200, pivot, 1e-3) is not None
    assert plane_update(model[:200], src, nrm[:200], w, 200, pivot) is None
    # fewer than 6 usable correspondences
    assert gicp_update(model[:5], src[:5], nrm[:5], nrm[:5], w[:5], 5, pivot, 1e-3) is None


def test_abi_declares_gicp():
    from pcreg_b200 import _lib
    with open(os.path.join(ROOT, "include", "pcreg.h")) as f:
        h = f.read()
    assert re.search(r"int\s+pcreg_icp_batch_gicp\(", h) and re.search(r"int\s+pcreg_icp_batch_gicp_dev\(", h)
    res, args = _lib.SIGNATURES["pcreg_icp_batch_gicp"]
    assert len(args) == 21 and args[6] is C.c_void_p and args[7] is C.c_double and args[11] == C.POINTER(_lib.IcpStop)
    res, args = _lib.SIGNATURES["pcreg_icp_batch_gicp_dev"]
    assert len(args) == 20 and args[5] is C.c_double and args[9] == C.POINTER(_lib.IcpStop)
    import pcreg_b200
    assert callable(pcreg_b200.cloud_normals)


def test_model_keeps_its_methods_and_cloud_normals_is_a_module_function():
    """cloud_normals sits next to Model in api.py; Model must keep every method, __del__ included (an undestroyed Model frees
    its device buffers through it)."""
    from pcreg_b200 import api
    for name in ("__init__", "handle", "grid_info", "voxel_info", "nn_search", "set_normals", "compute_normals", "normals",
                 "destroy", "__del__"):
        assert name in api.Model.__dict__, name
    assert api.cloud_normals.__qualname__ == "cloud_normals"
