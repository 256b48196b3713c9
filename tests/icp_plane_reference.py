"""FP64 reference of the model normals and the point-to-plane ICP metric (include/pcreg.h: pcreg_model_compute_normals,
pcreg_icp_batch_metric).  TEST INFRASTRUCTURE ONLY.

Normals: the k nearest model points of every model point in (d2, index) order -- d2 as oracle.nn.d2_exact computes it -- their
unweighted covariance about the mean, numpy.linalg.eigh's eigenvector of the smallest eigenvalue, the library's orientation rule.
The ICP loop is oracle/icp.py's icp_single (same NN step, weights and compose; its helpers are reused) with the point-to-plane
update: a = (q~ x n, n), b = (m~ - q~) . n about the model's pivot, A x = g by LDL' without pivoting (degenerate when a pivot is
at or below 1e-12 max A_kk, with fewer than 6 usable correspondences or no weight), Rodrigues, T <- T dT.  The optional tolerance
stop is tests/icp_stop_reference.py's rule.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

from icp_stop_reference import update_motion, window_means
from oracle.icp import _weights
from oracle.nn import KDTreeNN, d2_exact, nn_brute
from oracle.primitives import quickTF


def model_pivot(model):
    model = np.asarray(model, dtype=np.float64)
    return 0.5 * (model.min(axis=0) + model.max(axis=0))


def knn_exact(model, k):
    """[n, k] indices of the k nearest model points of every model point, (d2, index) order, the point itself included.
    Candidates come from a kd-tree (k + 8 of them) and are re-ranked with the exact d2; a point whose candidate list cannot
    prove its k-th neighbour (the last candidate not strictly farther) is searched by brute force."""
    model = np.asarray(model, dtype=np.float64)
    n = model.shape[0]
    kc = min(n, k + 8)
    _, cand = cKDTree(model).query(model, kc)
    cand = np.asarray(cand).reshape(n, kc)
    d2 = d2_exact(model[cand], model[:, None, :])
    o = np.lexsort((cand, d2), axis=-1)
    out = np.take_along_axis(cand, o[:, :k], axis=1).astype(np.int64)
    kth = np.take_along_axis(d2, o[:, k - 1:k], axis=1)[:, 0]
    for i in np.nonzero(~(kth < d2.max(axis=1)))[0] if kc < n else []:
        out[i] = np.lexsort((np.arange(n), d2_exact(model, model[i])))[:k]
    return out


def normals_reference(model, k=6, viewpoint=None):
    """-> (normals [n, 3], eigenvalues [n, 3] ascending) by the rule of pcreg_model_compute_normals."""
    model = np.asarray(model, dtype=np.float64)
    nb = knn_exact(model, k)
    X = model[nb]                                              # [n, k, 3]
    Xc = X - X.mean(axis=1, keepdims=True)
    C = np.einsum("nki,nkj->nij", Xc, Xc)
    w, V = np.linalg.eigh(C)
    nrm = V[:, :, 0]
    nrm = nrm / np.linalg.norm(nrm, axis=1, keepdims=True)
    if viewpoint is not None:
        dot = ((np.asarray(viewpoint, dtype=np.float64) - model) * nrm).sum(axis=1)
    else:
        dot = ((model - model_pivot(model)) * nrm).sum(axis=1)
    nrm[dot < 0] *= -1.0
    return nrm, w


def ldlt_solve(A, g):
    """A x = g by A = L D L' without pivoting; None when some D_k <= 1e-12 max_k A_kk."""
    n = A.shape[0]
    tiny = 1e-12 * max(0.0, float(np.max(np.diag(A))))
    L = np.eye(n)
    D = np.zeros(n)
    for j in range(n):
        d = A[j, j] - np.sum(L[j, :j] ** 2 * D[:j])
        if not d > tiny:
            return None
        D[j] = d
        for i in range(j + 1, n):
            L[i, j] = (A[i, j] - np.sum(L[i, :j] * L[j, :j] * D[:j])) / d
    y = np.linalg.solve(L, g)
    return np.linalg.solve(L.T, y / D)


def rodrigues(w):
    t = float(np.linalg.norm(w))
    if not t > 0:
        return np.eye(3)
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    return np.eye(3) + np.sin(t) / t * K + (1 - np.cos(t)) / (t * t) * (K @ K)


def plane_update(mj, q, nj, w, n_used, pivot):
    """dT of one point-to-plane step, or None (degenerate)."""
    if n_used < 6 or not w.sum() > 0:
        return None
    qt, mt = q - pivot, mj - pivot
    a = np.hstack([np.cross(qt, nj), nj])
    b = ((mt - qt) * nj).sum(axis=1)
    wa = w[:, None] * a
    x = ldlt_solve(wa.T @ a, wa.T @ b)
    if x is None:
        return None
    dR = rodrigues(x[:3]).T
    dT = np.eye(4)
    dT[:3, :3] = dR
    dT[3, :3] = pivot - pivot @ dR + x[3:]
    return dT


def icp_single_plane(model, normals, src, T0, mode=0, iters=50, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src=None, nn=None,
                     tolerance=None, window=3):
    """One hypothesis -> dict(T, rmse, n_used, idx, status, rmse_hist, n_iter, converged, T_hist)."""
    model = np.asarray(model, dtype=np.float64)
    normals = np.asarray(normals, dtype=np.float64)
    src = np.asarray(src, dtype=np.float64)
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
        dT = plane_update(model[j], q, normals[j], w, n_used, pivot)
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


def icp_batch_plane(model, normals, src, T0s, brute=False, **kw):
    """H hypotheses; winner = first-index arg-min of rmse (NaN never wins), as oracle.icp_batch."""
    T0s = np.asarray(T0s, dtype=np.float64).reshape(-1, 4, 4)
    model = np.asarray(model, dtype=np.float64)
    if brute:
        class _B:
            def query(self, q): return nn_brute(model, q)
        nn = _B()
    else:
        nn = KDTreeNN(model)
    res = [icp_single_plane(model, normals, src, T0s[h], nn=nn, **kw) for h in range(T0s.shape[0])]
    rm = np.array([r["rmse"] for r in res])
    out = dict(T=np.stack([r["T"] for r in res]), rmse=rm, best=int(np.nanargmin(rm)) if np.any(~np.isnan(rm)) else -1, results=res)
    for k in ("n_used", "status", "n_iter", "converged"):
        out[k] = np.array([r[k] for r in res], dtype=np.int32)
    out["idx"] = np.stack([r["idx"] for r in res])
    out["rmse_hist"] = np.stack([r["rmse_hist"] for r in res])
    return out


def ellipsoid_problem(n_model=40_000, n_src=1000, seed=7, deg=5.0, mm=2.0):
    """A dense, noiseless, smooth model (an ellipsoid, semi-axes 60 / 45 / 35 mm) with its analytic unit normals, a source patch
    (every 8th of the 8 n_src model points nearest to one of them, about a fifth of the surface) moved by the inverse of T_gt,
    and a start pose deg degrees / mm millimetres from T_gt."""
    g = np.random.default_rng(seed)
    ax = np.array([60.0, 45.0, 35.0])
    d = g.standard_normal((n_model, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    model = d * ax
    nrm = model / ax ** 2
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    c = model[0]
    sel = np.argsort(d2_exact(model, c), kind="stable")[:8 * n_src:8]
    R_gt = _rot([0.2, 0.9, -0.4], np.deg2rad(20.0))
    T_gt = np.eye(4)
    T_gt[:3, :3] = R_gt
    T_gt[3, :3] = [5.0, -3.0, 8.0]
    Ti = np.eye(4)
    Ti[:3, :3] = R_gt.T
    Ti[3, :3] = -T_gt[3, :3] @ R_gt.T
    src = quickTF(model[sel], Ti)
    P = np.eye(4)
    Rp = _rot([1.0, -0.5, 0.3], np.deg2rad(deg))
    P[:3, :3] = Rp
    P[3, :3] = c - c @ Rp + mm * np.array([0.6, -0.48, 0.64])
    return model, nrm, src, T_gt, T_gt @ P


def _rot(axis, angle):
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)
