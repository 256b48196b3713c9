"""The trim selection of the fused ICP kernel on inputs that stress its histogram.

The fused kernel fills the trim histogram while it searches the neighbours, under a range-free bin map whose 16-octave
window is centred on the previous pass's K-th residual (pass 0, and a pass after one whose K-th residual is zero or that
selected nothing: a fixed 1/16-octave map over [2^-64, 2^64)).  The per-pass kernels and the brute-force path use the
linear map over [min, max] of the pass.  The selection is exact under any monotone map, so every path returns the same
bits; each case here runs all three and compares poses, rmse, rmse history, n_used, status and correspondences."""
import numpy as np
import pytest

import oracle
from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

OUT_KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


def _run_paths(P, monkeypatch, model, src, T0, iters, **kw):
    """fused (forced), per-pass and brute force: every output bit for bit.  Returns the fused result."""
    m = P.Model(model, grid=True, voxel_map=1)
    out = {}
    try:
        for path, nn, fused in (("fused", P.NN_GRID, "1"), ("per-pass", P.NN_GRID, "0"), ("brute", P.NN_BRUTE, None)):
            monkeypatch.delenv("PCREG_FUSED", raising=False)
            if fused is not None:
                monkeypatch.setenv("PCREG_FUSED", fused)
            out[path] = P.icp_batch(m, src, T0, mode=P.ICP_KNN, iters=iters, nn=nn, return_idx=True, return_hist=True, **kw)
    finally:
        monkeypatch.delenv("PCREG_FUSED", raising=False)
        m.destroy()
    for path in ("per-pass", "brute"):
        for k in OUT_KEYS:
            assert _eq(out["fused"][k], out[path][k]), (path, k)
        assert out["fused"]["best"] == out[path]["best"], path
    return out["fused"]


def _problem(ns=600, H=6, seed=300, sigma=0.3):
    model = synth.make_model(20_000, seed)
    src, T_gt, c = synth.make_source(model, ns, sigma, seed + 1)
    T0 = synth.pose_grid(T_gt, c, max(1, H // 2), (2, 1, 1), 8.0, 1.0, seed + 2)[:H]
    return model, src, np.asarray(T0)


@pytest.mark.parametrize("scale", [1e-6, 1e6])
def test_scaled_problem(pcreg, monkeypatch, scale):
    """Residuals around 1e-7 or 1e5: the pass-0 window and the centred windows of later passes sit far from unit scale."""
    model, src, T0 = _problem()
    T0s = T0.copy()
    T0s[:, 3, :3] *= scale
    res = _run_paths(pcreg, monkeypatch, model.astype(np.float64) * scale, src * scale, T0s, 10, k_frac=0.85)
    assert np.all(res["status"] == 0)
    assert np.all(res["n_used"] == round(0.85 * src.shape[0]))


def test_residuals_wider_than_the_window(pcreg, monkeypatch):
    """Residuals from 1e-7 to 1e5 (more than 16 octaves each side of the K-th): both clamped end bins hold keys."""
    model = np.asarray(synth.make_model(20_000, 310), dtype=np.float64)
    g = synth.rng(311)
    ns = 800
    pick = g.choice(model.shape[0], ns, replace=False)
    direction = g.standard_normal((ns, 3))
    direction /= np.linalg.norm(direction, axis=1, keepdims=True)
    mag = 10.0 ** g.uniform(-7.0, -1.0, ns)
    mag[g.choice(ns, ns // 10, replace=False)] = 1e5                   # far outliers, walked and trimmed
    src = model[pick] + direction * mag[:, None]
    T0 = np.repeat(np.eye(4)[None], 4, axis=0)
    for h in range(1, 4):
        T0[h, 3, :3] = g.uniform(-0.02, 0.02, 3)
    res = _run_paths(pcreg, monkeypatch, model, src, T0, 8, k_frac=0.85)
    assert np.all(res["n_used"] == round(0.85 * ns))


def test_crowded_boundary_bin_takes_the_radix_fallback(pcreg, monkeypatch):
    """1500 copies of one source point (more than the 1024 candidates of a boundary bin) hold the K-th residual."""
    model, src, T0 = _problem(ns=1500, H=4, seed=320)
    src = np.vstack([src[:1000], np.repeat(src[:1], 1500, axis=0), src[1000:] + 5.0])       # K = 1500 falls on the copies
    res = _run_paths(pcreg, monkeypatch, model, src, T0, 6, k_frac=0.5)
    assert np.all(res["n_used"][res["status"] == 0] == 1500)


def test_tie_at_k_with_tie_order(pcreg, monkeypatch):
    """A few hundred duplicated source points straddle the K-th residual; the source is reordered on the device, so the
    stable rule ranks the ties in the caller's order (tie_order).  Also against the FP64 oracle."""
    model, src, T0 = _problem(ns=300, H=3, seed=330)
    src = np.vstack([src, src, src[:120]])
    res = _run_paths(pcreg, monkeypatch, model, src, T0, 6, k_frac=0.5)
    ref = oracle.icp_batch(model, src, T0, mode=oracle.ICP_KNN, iters=6, k_frac=0.5)
    assert np.array_equal(res["n_used"], ref["n_used"])
    assert np.array_equal(res["status"], ref["status"])
    np.testing.assert_allclose(res["rmse"], ref["rmse"], rtol=1e-7)


def test_window_resets(pcreg, monkeypatch):
    """A hypothesis that keeps nothing (all residuals beyond thDist2: K = 0, pose frozen) beside ones whose K-th residual
    is exactly zero (source = model points at the identity), so later passes fall back to the fixed window, and ordinary
    ones."""
    model = np.asarray(synth.make_model(20_000, 340), dtype=np.float64)
    g = synth.rng(341)
    pick = g.choice(model.shape[0], 700, replace=False)
    src = model[pick].copy()
    src[350:] += g.normal(0.0, 0.3, (350, 3))
    T0 = np.repeat(np.eye(4)[None], 4, axis=0)
    T0[1, 3, :3] = [500.0, 0.0, 0.0]                                    # nothing within thDist2
    T0[2, 3, :3] = [0.3, -0.2, 0.1]
    res = _run_paths(pcreg, monkeypatch, model, src, T0, 8, k_frac=0.4, thDist2=4.0)
    assert res["status"][1] == 1 and res["n_used"][1] == 0 and np.isnan(res["rmse"][1])
    assert res["status"][0] == 0 and res["rmse"][0] < 1e-9
    assert res["status"][2] == 0 and res["n_used"][2] > 0
