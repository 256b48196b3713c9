"""Oracle of the composed ICP loop (SURVEY.md section 8c).  TEST INFRASTRUCTURE ONLY.

The reference contains no ICP; this is the composition of its primitives that
BASELINE.json's north_star describes:
  pose apply      quickTF.m:5-7
  NN step         MATLAB knnsearch semantics (not in reference; oracle/nn.py) -- PARITY UNPINNED
  rejection       squared-distance compare as ransac.m:49 (dist < thDist keeps)
  trimming (KNN)  keep round(k_frac*n) smallest residuals, stable sort  (AlignPoints_KNN.m:20-26)
  weights         w = max(R_w - r, 0)                                    (AlignPoints_weighted.m:16-18)
  rigid fit       estimateTransform.m:41-71 arranged as estimateTransform(pts1=model_j, pts2=q),
                  weighted centroids + weighted cross-covariance, R = V*U' (no det fix by default); the
                  project's own rule: an H of numerical rank <= 2 gives the proper solution (RANK2_TAU)
  compose         T <- T * dT  (row-vector convention)
  winner          first-index arg-min of rmse (ransac.m:69-73 max() tie rule, mirrored)
FP64 throughout.
"""
from __future__ import annotations

import numpy as np

from .nn import KDTreeNN, d2_exact, nn_brute
from .primitives import matlab_round, quickTF

ICP_PLAIN, ICP_KNN, ICP_WEIGHTED = 0, 1, 2


def _weights(d2, mode, k_frac, R_w, thDist2, w_src):
    """Per-correspondence weights for one hypothesis -> (w, n_used)."""
    n = d2.shape[0]
    keep = np.ones(n, dtype=bool)
    if thDist2 > 0:
        keep &= d2 < thDist2                       # squared compare (ransac.m:49)
    r = np.sqrt(d2)
    w = np.zeros(n, dtype=np.float64)
    if mode == ICP_PLAIN:
        w[keep] = 1.0
    elif mode == ICP_KNN:
        cand = np.nonzero(keep)[0]
        K = int(matlab_round(k_frac * cand.size))  # AlignPoints_KNN.m:21
        order = np.argsort(r[cand], kind="stable") # :24, ties -> lower index
        w[cand[order[:K]]] = 1.0
    elif mode == ICP_WEIGHTED:
        w[keep] = np.maximum(R_w - r[keep], 0.0)   # AlignPoints_weighted.m:16-18
    else:
        raise ValueError("mode")
    if w_src is not None:
        w = w * w_src
    return w, int(np.sum(w > 0))


RANK2_TAU = 1e-8       # include/pcreg.h: pcreg_icp_opts.reflection_fix (pcreg_math.cuh: ICP_RANK2_TAU)


def _weighted_kabsch(m_pts, q_pts, w, reflection_fix):
    """estimateTransform(pts1=m_pts, pts2=q_pts) with weights: returns dT with [q,1]*dT ~ [m,1].

    The ICP update's rank rule: with S[2] <= RANK2_TAU * S[0], or S[0] <= RANK2_TAU * |sum w q m'|_F (H numerically of rank <= 2,
    or rounding noise; the rotation and the reflection then fit equally well) the update is the proper solution whatever
    reflection_fix says."""
    sw = w.sum()
    cd = (w[:, None] * m_pts).sum(axis=0) / sw     # estimateTransform.m:46 (d = pts1 = model side)
    cm = (w[:, None] * q_pts).sum(axis=0) / sw     # :47 (m = pts2 = query side)
    H = ((q_pts - cm) * w[:, None]).T @ (m_pts - cd)   # :58  H = m_c * d_c'
    U, S, Vt = np.linalg.svd(H)                    # :60
    V = Vt.T
    rank2 = S[2] <= RANK2_TAU * S[0] or S[0] <= RANK2_TAU * np.linalg.norm((w[:, None] * q_pts).T @ m_pts)
    if (reflection_fix or rank2) and np.linalg.det(V @ U.T) < 0:
        V = V.copy()
        V[:, 2] = -V[:, 2]
    R = V @ U.T                                    # :62
    t = cd - R @ cm                                # :63
    dT = np.eye(4)
    dT[0:3, 0:3] = R.T
    dT[3, 0:3] = t
    return dT


def icp_single(model, src, T0, mode=ICP_PLAIN, iters=50, k_frac=0.85, R_w=3.5, thDist2=0.0,
               w_src=None, reflection_fix=False, nn=None, return_hist=False):
    """One hypothesis.  Returns dict(T, rmse, n_used, idx, d2, status[, rmse_hist]).

    status: 0 ok; 1 = fewer than 3 usable correspondences at some iteration (T frozen there)."""
    model = np.asarray(model, dtype=np.float64)
    src = np.asarray(src, dtype=np.float64)
    T = np.array(T0, dtype=np.float64).reshape(4, 4).copy()
    if nn is None:
        nn = KDTreeNN(model)
    query = nn.query if hasattr(nn, "query") else (lambda q: nn_brute(model, q))
    status = 0
    hist = []
    for _ in range(iters):
        q = quickTF(src, T)
        j, _ = query(q)
        mj = model[j]
        d2 = d2_exact(mj, q)
        w, n_used = _weights(d2, mode, k_frac, R_w, thDist2, w_src)
        sw = w.sum()
        hist.append(np.sqrt((w * d2).sum() / sw) if sw > 0 else np.nan)
        if n_used < 3 or not sw > 0:
            status = 1
            break
        dT = _weighted_kabsch(mj, q, w, reflection_fix)
        T = T @ dT
    q = quickTF(src, T)
    j, _ = query(q)
    d2 = d2_exact(model[j], q)
    w, n_used = _weights(d2, mode, k_frac, R_w, thDist2, w_src)
    sw = w.sum()
    rmse = float(np.sqrt((w * d2).sum() / sw)) if sw > 0 else float("nan")
    out = dict(T=T, rmse=rmse, n_used=n_used, idx=np.asarray(j, dtype=np.int32), d2=d2, status=status)
    if return_hist:
        hist.append(rmse)
        out["rmse_hist"] = np.asarray(hist)
    return out


def icp_batch(model, src, T0s, brute=False, **kw):
    """H hypotheses; winner = first-index arg-min of rmse over hypotheses (NaN never wins)."""
    T0s = np.asarray(T0s, dtype=np.float64).reshape(-1, 4, 4)
    nn = None if brute else KDTreeNN(np.asarray(model, dtype=np.float64))
    if brute:
        class _B:
            def __init__(self, m): self.m = np.asarray(m, dtype=np.float64)
            def query(self, q): return nn_brute(self.m, q)
        nn = _B(model)
    res = [icp_single(model, src, T0s[h], nn=nn, **kw) for h in range(T0s.shape[0])]
    rm = np.array([r["rmse"] for r in res])
    best = int(np.nanargmin(rm)) if np.any(~np.isnan(rm)) else -1
    return dict(T=np.stack([r["T"] for r in res]), rmse=rm,
                n_used=np.array([r["n_used"] for r in res], dtype=np.int32),
                status=np.array([r["status"] for r in res], dtype=np.int32),
                idx=np.stack([r["idx"] for r in res]), best=best, results=res)
