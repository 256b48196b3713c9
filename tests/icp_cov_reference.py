"""FP64 reference of the pose covariance and the predicted target registration error (include/pcreg.h: pcreg_icp_covariance).
TEST INFRASTRUCTURE ONLY.

The scoring pass is oracle/icp.py's final pass (exact NN, d2_exact, _weights); the sums are the point-to-plane ones of
tests/icp_plane_reference.py about the model's pivot, with B = sum w b^2; the degenerate rule is its ldlt_solve's.  The covariance is
numpy.linalg.inv of A moved to `ref` by M = [[I, 0], [-[ref - p]x, I]]."""
from __future__ import annotations

import numpy as np

from icp_plane_reference import ldlt_solve, model_pivot
from oracle.icp import _weights
from oracle.nn import KDTreeNN, d2_exact
from oracle.primitives import quickTF


def skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def cov_from_sums(A, B, S, n_used, pivot, ref):
    """-> (cov [6,6], info [6,6], sigma2, status) by the rule of pcreg_icp_covariance."""
    M = np.eye(6)
    M[3:, :3] = -skew(np.asarray(ref, dtype=np.float64) - pivot)
    Mi = np.linalg.inv(M)
    info = Mi.T @ A @ Mi if n_used > 0 else np.full((6, 6), np.nan)
    ok = n_used > 6 and S > 0
    sigma2 = (B / S) * n_used / (n_used - 6) if ok else np.nan
    if not ok or ldlt_solve(A, np.zeros(6)) is None:
        return np.full((6, 6), np.nan), info, sigma2, 1
    return sigma2 * M @ np.linalg.inv(A) @ M.T, info, sigma2, 0


def tre_of(cov, ref, targets):
    """sqrt(trace(J_k cov J_k')) with J_k = [-[x_k - ref]x, I] for every target x_k."""
    out = []
    for x in np.asarray(targets, dtype=np.float64).reshape(-1, 3):
        J = np.hstack([-skew(x - np.asarray(ref, dtype=np.float64)), np.eye(3)])
        out.append(np.sqrt(np.trace(J @ cov @ J.T)))
    return np.asarray(out)


def pose_covariance(model, normals, src, Ts, mode=0, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src=None, ref=None, targets=None, nn=None):
    """H poses -> dict(cov [H,6,6], info [H,6,6], sigma2, rmse, n_used, status [H], tre [H,K], idx [H,ns])."""
    model = np.asarray(model, dtype=np.float64)
    normals = np.asarray(normals, dtype=np.float64)
    src = np.asarray(src, dtype=np.float64)
    pivot = model_pivot(model)
    ref = np.zeros(3) if ref is None else np.asarray(ref, dtype=np.float64)
    targets = np.zeros((0, 3)) if targets is None else np.asarray(targets, dtype=np.float64).reshape(-1, 3)
    if nn is None:
        nn = KDTreeNN(model)
    out = {k: [] for k in ("cov", "info", "sigma2", "rmse", "n_used", "status", "tre", "idx")}
    for T in np.asarray(Ts, dtype=np.float64).reshape(-1, 4, 4):
        q = quickTF(src, T)
        j, _ = nn.query(q)
        d2 = d2_exact(model[j], q)
        w, n_used = _weights(d2, mode, k_frac, R_w, thDist2, w_src)
        S = w.sum()
        qt, mt, nj = q - pivot, model[j] - pivot, normals[j]
        a = np.hstack([np.cross(qt, nj), nj])
        b = ((mt - qt) * nj).sum(axis=1)
        A = (w[:, None] * a).T @ a
        cov, info, s2, st = cov_from_sums(A, float((w * b * b).sum()), S, n_used, pivot, ref)
        for k, v in (("cov", cov), ("info", info), ("sigma2", s2), ("rmse", np.sqrt((w * d2).sum() / S) if S > 0 else np.nan),
                     ("n_used", n_used), ("status", st), ("tre", tre_of(cov, ref, targets)), ("idx", np.asarray(j, dtype=np.int32))):
            out[k].append(v)
    return {k: np.asarray(v) for k, v in out.items()}


# ---- exact shapes with analytic normals (noise-free, the source ON the model: every residual b is zero) ----
def plane_shape(n=40):
    g = np.linspace(-10, 10, n)
    X, Y = np.meshgrid(g, g)
    pts = np.stack([X.ravel(), Y.ravel(), np.zeros(X.size)], axis=1)
    return pts, np.tile([0.0, 0.0, 1.0], (pts.shape[0], 1))


def cylinder_shape(n_around=64, n_axis=40, r=8.0):
    t = np.linspace(0, 2 * np.pi, n_around, endpoint=False)
    z = np.linspace(-10, 10, n_axis)
    T, Z = np.meshgrid(t, z)
    nrm = np.stack([np.cos(T.ravel()), np.sin(T.ravel()), np.zeros(T.size)], axis=1)
    return np.hstack([r * nrm[:, :2], Z.ravel()[:, None]]), nrm


def sphere_shape(n=2000, r=8.0, seed=0):
    d = np.random.default_rng(seed).standard_normal((n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return r * d, d


# ---- calibration: predicted against empirical pose scatter ----
def pose_error(T, T_gt, ref):
    """(omega, tau) about ref of the pose error D = T_gt^-1 T (row-vector poses): to first order T moves the model-frame point x of T_gt
    to x + omega x (x - ref) + tau."""
    D = np.linalg.inv(T_gt) @ T
    Rd, td = D[:3, :3], D[3, :3]
    K = 0.5 * (Rd.T - Rd)                       # [omega]x to first order
    om = np.array([K[2, 1], K[0, 2], K[1, 0]])
    return np.hstack([om, td + np.cross(om, ref)])


def calibration_ratios(cov_pred, errors):
    """Empirical / predicted std along the principal directions of the mean predicted covariance (largest first)."""
    C = np.mean(cov_pred, axis=0)
    E = np.cov(np.asarray(errors).T)
    w, V = np.linalg.eigh(C)
    V = V[:, ::-1]
    pred = np.sqrt(np.einsum("ij,jk,ki->i", V.T, C, V))
    emp = np.sqrt(np.einsum("ij,jk,ki->i", V.T, E, V))
    return emp / pred, pred
