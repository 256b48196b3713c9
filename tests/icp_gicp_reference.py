"""FP64 reference of the plane-to-plane (generalized ICP) metric (include/pcreg.h: pcreg_icp_batch_gicp).  TEST INFRASTRUCTURE ONLY.

The loop is tests/icp_plane_reference.py's (oracle/icp.py's NN step, weights and compose; the same LDL' solve, degeneracy rule and
Rodrigues update); only the sums differ: per correspondence C = 2I - (1 - eps)(n_m n_m' + n_q n_q') with n_q = n_s R,
M = inv(C), e = m~ - q~, J' = [[q~]x; I], A = sum w J' M J and g = sum w J' M e.  The optional tolerance stop is
tests/icp_stop_reference.py's rule.
"""
from __future__ import annotations

import numpy as np

from icp_plane_reference import _rot, ellipsoid_problem, ldlt_solve, model_pivot, rodrigues  # noqa: F401
from icp_stop_reference import update_motion, window_means
from oracle.icp import _weights
from oracle.nn import KDTreeNN, d2_exact, nn_brute
from oracle.primitives import quickTF


def skew(v):
    """[v]x for a batch [n, 3] -> [n, 3, 3] ([v]x u = v x u)."""
    v = np.asarray(v, dtype=np.float64)
    z = np.zeros(v.shape[:-1])
    return np.stack([np.stack([z, -v[..., 2], v[..., 1]], -1), np.stack([v[..., 2], z, -v[..., 0]], -1),
                     np.stack([-v[..., 1], v[..., 0], z], -1)], -2)


def gicp_information(nq, nm, eps):
    """M = inv(2I - (1 - eps)(nm nm' + nq nq')) for a batch [n, 3] -> [n, 3, 3]."""
    C = 2.0 * np.eye(3) - (1.0 - eps) * (np.einsum("ni,nj->nij", nm, nm) + np.einsum("ni,nj->nij", nq, nq))
    return np.linalg.inv(C)


def gicp_sums(qt, mt, nq, nm, w, eps):
    """A = sum w J' M J (6 x 6) and g = sum w J' M e (6) with J' = [[qt]x; I], e = mt - qt."""
    M = gicp_information(nq, nm, eps)
    Jt = np.concatenate([skew(qt), np.broadcast_to(np.eye(3), (qt.shape[0], 3, 3))], axis=1)      # [n, 6, 3]
    JtM = w[:, None, None] * (Jt @ M)
    A = np.einsum("nik,njk->ij", JtM, Jt)
    g = np.einsum("nik,nk->i", JtM, mt - qt)
    return A, g


def gicp_update(mj, q, nq, nm, w, n_used, pivot, eps):
    """dT of one plane-to-plane step, or None (degenerate); the solve and update are the point-to-plane ones."""
    if n_used < 6 or not w.sum() > 0:
        return None
    A, g = gicp_sums(q - pivot, mj - pivot, nq, nm, w, eps)
    x = ldlt_solve(A, g)
    if x is None:
        return None
    dR = rodrigues(x[:3]).T
    dT = np.eye(4)
    dT[:3, :3] = dR
    dT[3, :3] = pivot - pivot @ dR + x[3:]
    return dT


def icp_single_gicp(model, normals, src, src_normals, T0, eps=1e-3, mode=0, iters=50, k_frac=0.85, R_w=3.5, thDist2=0.0,
                    w_src=None, nn=None, tolerance=None, window=3):
    """One hypothesis -> dict(T, rmse, n_used, idx, status, rmse_hist, n_iter, converged, T_hist).  src_normals must be unit rows."""
    model = np.asarray(model, dtype=np.float64)
    normals = np.asarray(normals, dtype=np.float64)
    src = np.asarray(src, dtype=np.float64)
    sn = np.asarray(src_normals, dtype=np.float64)
    pivot = model_pivot(model)
    T = np.array(T0, dtype=np.float64).reshape(4, 4).copy()
    if nn is None:
        nn = KDTreeNN(model)
    status, n_iter, converged = 0, iters, 0
    hist, motion, T_hist = [], [], [T.copy()]
    for it in range(iters):
        q = quickTF(src, T)
        j, _ = nn.query(q)
        d2 = d2_exact(model[j], q)
        w, n_used = _weights(d2, mode, k_frac, R_w, thDist2, w_src)
        sw = w.sum()
        hist.append(np.sqrt((w * d2).sum() / sw) if sw > 0 else np.nan)
        dT = gicp_update(model[j], q, sn @ T[:3, :3], normals[j], w, n_used, pivot, eps)
        if dT is None:
            status, n_iter = 1, it
            break
        Tn = T @ dT
        motion.append(update_motion(T, Tn))
        T = Tn
        T_hist.append(T.copy())
        if tolerance is not None and len(motion) >= window:
            mt, mr = window_means(motion, window)
            if mt < tolerance[0] and mr < tolerance[1]:
                n_iter, converged = it + 1, 1
                break
    q = quickTF(src, T)
    j, _ = nn.query(q)
    d2 = d2_exact(model[j], q)
    w, n_used = _weights(d2, mode, k_frac, R_w, thDist2, w_src)
    sw = w.sum()
    rmse = float(np.sqrt((w * d2).sum() / sw)) if sw > 0 else float("nan")
    hist = np.asarray(hist + [rmse] * (iters + 1 - len(hist)))
    return dict(T=T, rmse=rmse, n_used=n_used, idx=np.asarray(j, dtype=np.int32), status=status, rmse_hist=hist, n_iter=n_iter,
                converged=converged, T_hist=T_hist)


def icp_batch_gicp(model, normals, src, src_normals, T0s, brute=False, **kw):
    """H hypotheses; winner = first-index arg-min of rmse (NaN never wins), as oracle.icp_batch."""
    T0s = np.asarray(T0s, dtype=np.float64).reshape(-1, 4, 4)
    model = np.asarray(model, dtype=np.float64)
    if brute:
        class _B:
            def query(self, q): return nn_brute(model, q)
        nn = _B()
    else:
        nn = KDTreeNN(model)
    res = [icp_single_gicp(model, normals, src, src_normals, T0s[h], nn=nn, **kw) for h in range(T0s.shape[0])]
    rm = np.array([r["rmse"] for r in res])
    out = dict(T=np.stack([r["T"] for r in res]), rmse=rm, best=int(np.nanargmin(rm)) if np.any(~np.isnan(rm)) else -1, results=res)
    for k in ("n_used", "status", "n_iter", "converged"):
        out[k] = np.array([r[k] for r in res], dtype=np.int32)
    out["idx"] = np.stack([r["idx"] for r in res])
    out["rmse_hist"] = np.stack([r["rmse_hist"] for r in res])
    return out


def unit_rows(n):
    """Rows normalised as the library does: n / sqrt((nx*nx + ny*ny) + nz*nz)."""
    n = np.asarray(n, dtype=np.float64)
    return n / np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])[:, None]


def ellipsoid_gicp_problem(n_model=40_000, n_src=1000, seed=7, deg=5.0, mm=2.0):
    """tests/icp_plane_reference.py's ellipsoid problem plus the source normals: the analytic model normals of the picked points,
    carried by T_gt^-1 as the points are.  -> (model, model normals, src, src normals, T_gt, T0)."""
    model, nrm, src, T_gt, T0 = ellipsoid_problem(n_model, n_src, seed, deg, mm)
    sel = np.argsort(d2_exact(model, model[0]), kind="stable")[:8 * n_src:8]           # the picks of ellipsoid_problem
    Ri = T_gt[:3, :3].T
    assert np.allclose(quickTF(model[sel], np.linalg.inv(T_gt)), src, rtol=0, atol=1e-9)
    return model, nrm, src, nrm[sel] @ Ri, T_gt, T0
