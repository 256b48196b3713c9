"""FP64 reference of the ICP tolerance stop (include/pcreg.h: pcreg_icp_stop).  TEST INFRASTRUCTURE ONLY.

The loop is oracle/icp.py's icp_single (same NN step, weights, rigid fit and compose; its helpers are reused) with the stop
rule added.  The rule restates the documented 'Tolerance' of MATLAB's pcregistericp -- a translation and a rotation
difference averaged over the most recent iterations -- and its parity with the toolbox is UNPINNED:
  after update u >= window, stop when mean(dt) < tol_t and mean(dr) < tol_r_deg over updates u-window+1 .. u
  (left-to-right FP64 sums divided by window, strict compares); the stopping update is applied.
"""
from __future__ import annotations

import numpy as np

from oracle.icp import _weighted_kabsch, _weights
from oracle.nn import KDTreeNN, d2_exact, nn_brute
from oracle.primitives import quickTF


def update_motion(Tc, Tn):
    """(dt, dr_deg) of the update Tc -> Tn = Tc @ dT: translation-row distance and the angle of dR = Rc' Rn (atan2 form)."""
    dR = Tc[:3, :3].T @ Tn[:3, :3]
    v = 0.5 * np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
    dr = np.degrees(np.arctan2(np.linalg.norm(v), 0.5 * (np.trace(dR) - 1.0)))
    return float(np.linalg.norm(Tn[3, :3] - Tc[3, :3])), float(dr)


def window_means(motion, window):
    """Means of the last `window` (dt, dr) pairs: left-to-right sums divided by window."""
    mt = mr = 0.0
    for dt, dr in motion[-window:]:
        mt += dt
        mr += dr
    return mt / window, mr / window


def icp_single_stop(model, src, T0, tolerance, window=3, mode=0, iters=50, k_frac=0.85, R_w=3.5, thDist2=0.0,
                    w_src=None, reflection_fix=False, nn=None):
    """One hypothesis -> dict(T, rmse, n_used, idx, status, rmse_hist, n_iter, converged, stop_means).

    rmse_hist has iters + 1 columns; from the final pass on, every column holds the final rmse.  stop_means lists the
    (mean_t, mean_r) of every update the rule was evaluated at (so a test can check how close a decision was)."""
    model = np.asarray(model, dtype=np.float64)
    src = np.asarray(src, dtype=np.float64)
    T = np.array(T0, dtype=np.float64).reshape(4, 4).copy()
    if nn is None:
        nn = KDTreeNN(model)
    status, n_iter, converged = 0, iters, 0
    hist, motion, stop_means = [], [], []
    for it in range(iters):
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
        Tn = T @ _weighted_kabsch(mj, q, w, reflection_fix)
        motion.append(update_motion(T, Tn))
        T = Tn
        if len(motion) >= window:
            mt, mr = window_means(motion, window)
            stop_means.append((mt, mr))
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
    return dict(T=T, rmse=rmse, n_used=n_used, idx=np.asarray(j, dtype=np.int32), status=status, rmse_hist=hist,
                n_iter=n_iter, converged=converged, stop_means=stop_means)


def icp_batch_stop(model, src, T0s, tolerance, window=3, brute=False, **kw):
    """H hypotheses; winner = first-index arg-min of rmse (NaN never wins), as oracle.icp_batch."""
    T0s = np.asarray(T0s, dtype=np.float64).reshape(-1, 4, 4)
    model = np.asarray(model, dtype=np.float64)
    if brute:
        class _B:
            def query(self, q): return nn_brute(model, q)
        nn = _B()
    else:
        nn = KDTreeNN(model)
    res = [icp_single_stop(model, src, T0s[h], tolerance, window, nn=nn, **kw) for h in range(T0s.shape[0])]
    rm = np.array([r["rmse"] for r in res])
    best = int(np.nanargmin(rm)) if np.any(~np.isnan(rm)) else -1
    out = dict(T=np.stack([r["T"] for r in res]), rmse=rm, best=best, results=res)
    for k, dt in (("n_used", np.int32), ("status", np.int32), ("n_iter", np.int32), ("converged", np.int32)):
        out[k] = np.array([r[k] for r in res], dtype=dt)
    out["idx"] = np.stack([r["idx"] for r in res])
    out["rmse_hist"] = np.stack([r["rmse_hist"] for r in res])
    return out
