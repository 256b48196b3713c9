"""FP64 reference of the ICP pose extrapolation (include/pcreg.h: pcreg_icp_extrap).  TEST INFRASTRUCTURE ONLY.

The loop is oracle/icp.py's icp_single (same NN step, weights, rigid fit and compose; its helpers are reused) with Besl & McKay's
accelerated step (1992, section IV) added, restated independently of the library's code: the quaternion comes from scipy, the
error d(T) is evaluated point by point, and the two fits are numpy.polyfit.  Parity with pcregistericp's 'Extrapolate' is UNPINNED.
  c = the source centroid; x(T) = (qR, c R + t), qR = (w, x, y, z) with w >= 0 for T_0 (first nonzero component positive at w = 0)
  and qR . qR_prev >= 0 afterwards.  Update u: K_u = T_{u-1} dT, Delta_u = x(K_u) - x_{u-1}, n_u = |Delta_u|, theta_u = the angle
  between Delta_{u-1} and Delta_u in degrees.  With u >= 3 and theta_u, theta_{u-1} < angle_deg: v = (0, -n_u, -n_u - n_{u-1}),
  D = (d(K_u), d_{u-1}, d_{u-2}); v1 = zero of the least-squares line, v2 = vertex of the parabola, vmax = vmax_scale n_u; the
  branch table picks dv; with dv > 0 the pose is built from x(K_u) + dv Delta_u / n_u (quaternion renormalised).
"""
from __future__ import annotations

import math

import numpy as np
from scipy.spatial.transform import Rotation

from icp_stop_reference import update_motion, window_means
from oracle.icp import _weighted_kabsch, _weights
from oracle.nn import KDTreeNN, d2_exact
from oracle.primitives import quickTF

BRANCH_NONE, BRANCH_V2, BRANCH_V1, BRANCH_VMAX = 0, 1, 2, 3


def pose_state(T, c, qprev=None):
    """x(T) in R^7: the quaternion (w, x, y, z) of the rotation block (read as a rotation matrix) and the centroid's image c R + t."""
    x, y, z, w = Rotation.from_matrix(T[:3, :3]).as_quat()
    q = np.array([w, x, y, z])
    if qprev is not None:
        if q @ qprev < 0:
            q = -q
    else:
        nz = q[np.nonzero(q)[0][0]]
        if nz < 0:
            q = -q
    return np.concatenate([q, c @ T[:3, :3] + T[3, :3]])


def pose_of_state(x, c):
    q = x[:4] / np.linalg.norm(x[:4])
    T = np.eye(4)
    T[:3, :3] = Rotation.from_quat([q[1], q[2], q[3], q[0]]).as_matrix()
    T[3, :3] = x[4:] - c @ T[:3, :3]
    return T


def branch(v1, v2, vmax):
    """(dv, branch) of the step table (strict compares; NaN fails each)."""
    if (0 < v2 < v1 < vmax) or (0 < v2 < vmax < v1):
        return v2, BRANCH_V2
    if (0 < v1 < v2 < vmax) or (0 < v1 < vmax < v2) or (v2 < 0 and 0 < v1 < vmax):
        return v1, BRANCH_V1
    if v1 > vmax and v2 > vmax:
        return vmax, BRANCH_VMAX
    return 0.0, BRANCH_NONE


def _rel_gap(a, b):
    return abs(a - b) / max(abs(a), abs(b), 1e-300)


def decision_margin(th, th_prev, angle_deg, v1, v2, vmax):
    """Smallest relative gap between two values the decision compares (a decision closer than rounding is not reproducible)."""
    gaps = [_rel_gap(t, angle_deg) for t in (th, th_prev) if t == t]
    if th < angle_deg and th_prev < angle_deg:
        vals = [v for v in (v1, v2, vmax) if math.isfinite(v)]
        gaps += [_rel_gap(a, b) for i, a in enumerate(vals) for b in vals[i + 1:]]
        gaps += [abs(v) / max(abs(vmax), 1e-300) for v in (v1, v2) if math.isfinite(v)]      # the compares with 0
    return min(gaps) if gaps else math.inf


def icp_single_extrap(model, src, T0, angle_deg=10.0, vmax_scale=25.0, extrapolate=True, tolerance=None, window=3, mode=0, iters=50,
                      k_frac=0.85, R_w=3.5, thDist2=0.0, w_src=None, reflection_fix=False, nn=None, replay=None):
    """One hypothesis -> dict(T, rmse, n_used, idx, status, rmse_hist, n_iter, converged, n_extrap, trace).

    trace: one dict per update (u, theta, v1, v2, vmax, dv, branch, margin, T).  replay: poses T_0..T_K (e.g. the library's own) --
    update u then starts from replay[u - 1] instead of the reference's pose, so its decisions can be compared one by one."""
    model = np.asarray(model, dtype=np.float64)
    src = np.asarray(src, dtype=np.float64)
    T = np.array(T0, dtype=np.float64).reshape(4, 4).copy()
    if nn is None:
        nn = KDTreeNN(model)
    c = src.mean(axis=0)
    if replay is not None:
        iters = len(replay) - 1
    status, n_iter, converged, n_extrap = 0, iters, 0, 0
    hist, motion, trace = [], [], []
    x_prev = pose_state(T, c)
    dl_prev, n_prev, th_prev, d_prev, d_prev2 = None, math.nan, math.nan, math.nan, math.nan
    for it in range(iters):
        if replay is not None:
            T = np.array(replay[it], dtype=np.float64)
        u = it + 1
        q = quickTF(src, T)
        j, _ = nn.query(q)
        mj = model[j]
        d2 = d2_exact(mj, q)
        w, n_used = _weights(d2, mode, k_frac, R_w, thDist2, w_src)
        sw = w.sum()
        hist.append(np.sqrt((w * d2).sum() / sw) if sw > 0 else np.nan)
        if n_used < 3 or not sw > 0:
            status, n_iter = 1, it
            break
        K = T @ _weighted_kabsch(mj, q, w, reflection_fix)
        mse = lambda P: float((w * ((mj - quickTF(src, P)) ** 2).sum(axis=1)).sum() / sw)  # noqa: E731
        Tn = K
        if extrapolate:
            xk = pose_state(K, c, x_prev[:4])
            dl = xk - x_prev
            n = float(np.linalg.norm(dl))
            th = math.nan
            if u >= 2 and n > 0 and n_prev > 0:
                th = math.degrees(math.acos(min(max(float(dl @ dl_prev) / (n * n_prev), -1.0), 1.0)))
            dK = mse(K)
            v1 = v2 = math.nan
            dv, br = 0.0, BRANCH_NONE
            vmax = vmax_scale * n
            if u >= 3 and th < angle_deg and th_prev < angle_deg:
                v = np.array([0.0, -n, -n - n_prev])
                D = np.array([dK, d_prev, d_prev2])
                a1, b1 = np.polyfit(v, D, 1)
                v1 = -b1 / a1 if a1 != 0 else math.nan
                a2, b2, _ = np.polyfit(v, D, 2)
                v2 = -b2 / (2 * a2) if a2 != 0 else math.nan
                dv, br = branch(v1, v2, vmax)
            trace.append(dict(u=u, theta=th, v1=v1, v2=v2, vmax=vmax, dv=dv, branch=br,
                              margin=decision_margin(th, th_prev, angle_deg, v1, v2, vmax) if u >= 3 else math.inf))
            if dv > 0:
                xn = xk + dv * dl / n
                xn[:4] /= np.linalg.norm(xn[:4])
                Tn = pose_of_state(xn, c)
                n_extrap += 1
            else:
                xn = xk
            trace[-1]["T"] = Tn
            x_prev, dl_prev, n_prev, th_prev = xn, dl, n, th
            d_prev2, d_prev = d_prev, mse(Tn)
        motion.append(update_motion(T, Tn))
        T = Tn
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
                converged=converged, n_extrap=n_extrap, trace=trace)
