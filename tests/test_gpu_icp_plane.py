"""The point-to-plane ICP metric and the model normals on the GPU (include/pcreg.h: pcreg_model_set_normals / _compute_normals /
_get_normals, pcreg_icp_batch_metric{,_dev}).

POINT_TO_POINT through the metric entry changes no bit of pcreg_icp_batch{,_stop}; POINT_TO_PLANE gives the same bits on the fused,
per-pass, brute-force and map-less grid paths, matches the FP64 reference (tests/icp_plane_reference.py) fed with the library's
own normals, composes with the tolerance stop (a stop after k updates equals an iters = k run) and does not depend on the device
count; the device normals match the reference's k nearest neighbours + eigenvector rule."""
import ctypes as C

import numpy as np
import pytest

from icp_plane_reference import ellipsoid_problem, icp_batch_plane, model_pivot, normals_reference
from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

ITERS = 12
TOL = (0.01, 0.5)
OUT_KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")
P2P, PLANE = 0, 1


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


@pytest.fixture(scope="module")
def prob():
    """12 poses up to 12 deg / 2 mm from the truth of a 600-point patch on a 20 000-point model."""
    model = synth.make_model(20_000, 100)
    src, T_gt, c = synth.make_source(model, 600, 0.3, 101)
    T0 = synth.pose_grid(T_gt, c, 3, (2, 2, 1), 12.0, 2.0, 102)
    return model, src, T0


@pytest.fixture()
def models(pcreg, prob):
    """Per test (the device-count test re-initialises the library, which invalidates model handles); normals computed on each."""
    model = prob[0]
    ms = dict(vox=pcreg.Model(model, grid=True, voxel_map=1), novox=pcreg.Model(model, grid=True, voxel_map=-1))
    for m in ms.values():
        m.compute_normals(6)
    yield ms
    for m in ms.values():
        m.destroy()


PATHS = {
    "fused": ("vox", "grid", {"PCREG_FUSED": "1"}),
    "per-pass": ("vox", "grid", {"PCREG_FUSED": "0"}),
    "per-pass-lanes": ("vox", "grid", {"PCREG_FUSED": "0", "PCREG_LANES": "2", "PCREG_MAX_CHUNK_HYP": "2"}),
    "brute": ("vox", "brute", {}),
    "grid-novox": ("novox", "grid", {}),
}

MODES = {
    "plain": lambda P, src: dict(mode=P.ICP_PLAIN, thDist2=9.0),
    "knn": lambda P, src: dict(mode=P.ICP_KNN, k_frac=0.85),
    "weighted": lambda P, src: dict(mode=P.ICP_WEIGHTED, R_w=3.5, w_src=synth.rng(77).uniform(0.5, 1.0, src.shape[0])),
}


def _setenv(monkeypatch, env):
    for k in ("PCREG_FUSED", "PCREG_LANES", "PCREG_MAX_CHUNK_HYP"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _run(P, m, src, T0, nn, iters=ITERS, **kw):
    kw.setdefault("mode", P.ICP_KNN)
    return P.icp_batch(m, src, T0, iters=iters, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE, return_idx=True,
                       return_hist=True, **kw)


def _run_metric(P, m, src, T0, nn, metric, iters=ITERS, tolerance=None, mode=None, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src=None):
    """pcreg_icp_batch_metric called directly (the Python wrapper routes POINT_TO_POINT to the existing entries)."""
    from pcreg_b200 import _lib as L
    mode = P.ICP_KNN if mode is None else mode
    T0 = np.asarray(T0).reshape(-1, 4, 4)
    H, ns = T0.shape[0], src.shape[0]
    a = np.asfortranarray(src, dtype=np.float64)
    T0a = np.ascontiguousarray(np.transpose(T0, (0, 2, 1))).reshape(H, 16)
    w = None if w_src is None else np.ascontiguousarray(w_src, dtype=np.float64)
    o = P.icp_opts(mode, iters, k_frac, R_w, thDist2, P.NN_GRID if nn == "grid" else P.NN_BRUTE)
    stop = P.icp_stop(*tolerance, 3) if tolerance is not None else None
    T = np.empty((H, 16))
    rmse = np.empty(H)
    n_used, status, n_iter, conv = (np.empty(H, dtype=np.int32) for _ in range(4))
    idx = np.empty((H, ns), dtype=np.int32)
    hist = np.empty((H, iters + 1))
    best = C.c_int64()
    f64 = lambda x: None if x is None else x.ctypes.data_as(L.c_f64p)  # noqa: E731
    i32 = lambda x: x.ctypes.data_as(L.c_i32p)  # noqa: E731
    rc = L.lib().pcreg_icp_batch_metric(m.handle, a.ctypes.data_as(C.c_void_p), 1, ns, ns, f64(w), f64(T0a), H, C.byref(o), metric,
                                        C.byref(stop) if stop is not None else None, f64(T), f64(rmse), i32(n_used), i32(status),
                                        i32(idx), f64(hist), C.byref(best), i32(n_iter), i32(conv))
    out = dict(rc=rc, T=np.ascontiguousarray(np.transpose(T.reshape(H, 4, 4), (0, 2, 1))), rmse=rmse, n_used=n_used, status=status,
               idx=idx, rmse_hist=hist, best=best.value)
    if tolerance is not None:
        out.update(n_iter=n_iter, converged=conv)
    return out


@pytest.mark.parametrize("stop", [None, TOL], ids=["fixed", "stop"])
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("mode", list(MODES))
def test_point_to_point_metric_is_bit_identical(pcreg, prob, models, monkeypatch, path, mode, stop):
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    kw = MODES[mode](pcreg, src)
    ref = _run(pcreg, models[mk], src, T0, nn, tolerance=stop, **kw)
    out = _run_metric(pcreg, models[mk], src, T0, nn, P2P, tolerance=stop, **kw)
    assert out["rc"] == 0
    for k in OUT_KEYS + (("n_iter", "converged") if stop else ()):
        assert _eq(out[k], ref[k]), (path, mode, k)
    assert out["best"] == ref["best"]


@pytest.mark.parametrize("mode", list(MODES))
def test_point_to_plane_paths_agree_bit_for_bit(pcreg, prob, models, monkeypatch, mode):
    _, src, T0 = prob
    kw = MODES[mode](pcreg, src)
    res = {}
    for path, (mk, nn, env) in PATHS.items():
        _setenv(monkeypatch, env)
        res[path] = _run(pcreg, models[mk], src, T0, nn, metric="point_to_plane", **kw)
    ref = res["fused"]
    assert np.all(ref["status"] == 0)
    for path, out in res.items():
        for k in OUT_KEYS:
            assert _eq(out[k], ref[k]), (path, mode, k)
        assert out["best"] == ref["best"]
    # the normals of the two models are the same bits
    assert _eq(models["vox"].normals(), models["novox"].normals())
    # the plane metric actually changes the result
    p2p = _run(pcreg, models["vox"], src, T0, "grid", **kw)
    assert not _eq(p2p["T"], ref["T"])


@pytest.mark.parametrize("path", ["fused", "brute"])
def test_point_to_plane_matches_the_reference(pcreg, prob, models, monkeypatch, path):
    model, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    nrm = models[mk].normals()                 # the ICP is checked on the library's own normals
    ref = icp_batch_plane(model, nrm, src, T0, mode=1, iters=ITERS, k_frac=0.85)
    out = _run(pcreg, models[mk], src, T0, nn, metric="point_to_plane")
    assert np.array_equal(out["status"], ref["status"]) and np.array_equal(out["n_used"], ref["n_used"])
    assert np.array_equal(out["idx"], ref["idx"])
    for h in range(T0.shape[0]):
        assert np.linalg.norm(out["T"][h][:3, :3] - ref["T"][h][:3, :3], "fro") <= 1e-6
        to = ref["T"][h][3, :3]
        assert np.linalg.norm(out["T"][h][3, :3] - to) <= 1e-6 * max(np.linalg.norm(to), 1e-12)
        assert abs(out["rmse"][h] - ref["rmse"][h]) <= 1e-7 * ref["rmse"][h]
    np.testing.assert_allclose(out["rmse_hist"], ref["rmse_hist"], rtol=1e-7)
    assert out["best"] == ref["best"]


@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_point_to_plane_with_stop_equals_fixed_iteration_run(pcreg, prob, models, monkeypatch, path):
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    iters = 20
    out = _run(pcreg, models[mk], src, T0, nn, iters=iters, metric="point_to_plane", tolerance=TOL)
    stopped = out["n_iter"][out["converged"] == 1]
    assert len(stopped) >= 3 and np.all(stopped < iters), out["n_iter"]
    for k in np.unique(out["n_iter"]):
        g = np.nonzero(out["n_iter"] == k)[0]
        ref = _run(pcreg, models[mk], src, T0[g], nn, iters=int(k), metric="point_to_plane")
        for key in ("T", "rmse", "n_used", "status", "idx"):
            assert _eq(out[key][g], ref[key]), (k, key)
        assert _eq(out["rmse_hist"][g, :k + 1], ref["rmse_hist"]), k
        assert _eq(out["rmse_hist"][g, k:], np.repeat(out["rmse"][g, None], iters + 1 - k, axis=1)), k


def _check_normals(pcreg, model, k, viewpoint):
    m = pcreg.Model(model, grid=True)
    try:
        m.compute_normals(k, viewpoint)
        n = m.normals()
    finally:
        m.destroy()
    nr, w = normals_reference(model, k, viewpoint)
    x = np.asarray(model, dtype=np.float64)
    assert np.allclose(np.linalg.norm(n, axis=1), 1.0, rtol=0, atol=1e-15)
    sep = (w[:, 1] - w[:, 0]) > 1e-6 * w[:, 1]
    assert sep.mean() > 0.99
    assert np.all(np.abs((n * nr).sum(axis=1))[sep] >= 1 - 1e-9)
    # the orientation rule (a tolerance for normals that are numerically tangent to the direction)
    d = (np.asarray(viewpoint) - x) if viewpoint is not None else (x - model_pivot(x))
    dot = (n * d).sum(axis=1)
    assert np.all(dot >= -1e-9 * np.linalg.norm(d, axis=1))
    return n


@pytest.mark.parametrize("n", [20_000, 200_000])
def test_compute_normals_matches_the_reference(pcreg, n):
    model = synth.make_model(n, 31 + n)
    n0 = _check_normals(pcreg, model, 6, None)
    vp = np.asarray(model, dtype=np.float64).mean(axis=0) + [0.0, 0.0, 400.0]
    n1 = _check_normals(pcreg, model, 6, vp)
    assert np.allclose(np.abs((n0 * n1).sum(axis=1)), 1.0, rtol=0, atol=1e-12)
    if n == 20_000:
        _check_normals(pcreg, model, 3, None)
        _check_normals(pcreg, model, 64, None)


def test_set_normals_round_trip(pcreg, prob):
    model = prob[0]
    m = pcreg.Model(model)
    try:
        g = synth.rng(5)
        raw = g.normal(size=(model.shape[0], 3)) * g.uniform(0.1, 10.0, (model.shape[0], 1))
        m.set_normals(raw)
        want = raw / np.sqrt((raw[:, 0] * raw[:, 0] + raw[:, 1] * raw[:, 1]) + raw[:, 2] * raw[:, 2])[:, None]
        np.testing.assert_allclose(m.normals(), want, rtol=1e-15, atol=0)
        r32 = raw.astype(np.float32)
        m.set_normals(r32)
        r = r32.astype(np.float64)
        want = r / np.sqrt((r[:, 0] * r[:, 0] + r[:, 1] * r[:, 1]) + r[:, 2] * r[:, 2])[:, None]
        np.testing.assert_allclose(m.normals(), want, rtol=1e-15, atol=0)
    finally:
        m.destroy()


@pytest.fixture()
def multi(pcreg, monkeypatch):
    monkeypatch.setenv("PCREG_ALLOW_DUP_DEVICES", "1")
    yield pcreg
    pcreg.init(0)


def test_results_do_not_depend_on_device_count(multi, prob):
    P = multi
    model, src, T0 = prob
    cases = [dict(nn="grid"), dict(nn="brute"), dict(nn="grid", tolerance=TOL)]
    ref = None
    for devs in ([0], [0, 0], [0, 0, 0]):
        P.init(devs)
        m = P.Model(model, grid=True)
        try:
            m.compute_normals(6)
            got = [m.normals()] + [_run(P, m, src, T0, metric="point_to_plane", **kw) for kw in cases]
        finally:
            m.destroy()
        if ref is None:
            ref = got
            continue
        assert _eq(got[0], ref[0]), devs
        for kw, a, r in zip(cases, got[1:], ref[1:]):
            for k in OUT_KEYS + (("n_iter", "converged") if "tolerance" in kw else ()):
                assert _eq(a[k], r[k]), (devs, kw, k)
            assert a["best"] == r["best"]


def test_errors_and_flat_patch(pcreg, prob):
    from pcreg_b200 import _lib as L
    lib = L.lib()
    model, src, T0 = prob
    m = pcreg.Model(model, grid=True)
    nogrid = pcreg.Model(model)
    try:
        # point-to-plane without normals: PCREG_ERR_STATE; no normals to read back either
        assert _run_metric(pcreg, m, src, T0[:2], "grid", PLANE)["rc"] == -4
        assert _run_metric(pcreg, m, src, T0[:2], "brute", PLANE)["rc"] == -4
        assert lib.pcreg_model_get_normals(m.handle, np.empty(3 * model.shape[0]).ctypes.data_as(L.c_f64p)) == -4
        with pytest.raises(pcreg.PcregError):
            _run(pcreg, m, src, T0[:2], "grid", metric="point_to_plane")
        # an unknown metric
        assert _run_metric(pcreg, m, src, T0[:2], "grid", 2)["rc"] == -1
        assert _run_metric(pcreg, m, src, T0[:2], "grid", -1)["rc"] == -1
        with pytest.raises(ValueError):
            _run(pcreg, m, src, T0[:2], "grid", metric="plane_to_plane")
        # compute_normals: no grid, k out of range
        assert lib.pcreg_model_compute_normals(nogrid.handle, 6, None) == -1
        for k in (2, 65, 0, -1):
            assert lib.pcreg_model_compute_normals(m.handle, k, None) == -1
        # set_normals: a zero or non-finite row
        ok = np.tile([0.0, 0.0, 1.0], (model.shape[0], 1))
        for bad in (0.0, np.nan, np.inf):
            n = ok.copy()
            n[17] = [bad, 0.0, 0.0] if bad != 0.0 else [0.0, 0.0, 0.0]
            a = np.asfortranarray(n)
            assert lib.pcreg_model_set_normals(m.handle, a.ctypes.data_as(C.c_void_p), 1, model.shape[0]) == -1
        assert lib.pcreg_model_get_normals(m.handle, np.empty(3 * model.shape[0]).ctypes.data_as(L.c_f64p)) == -4
    finally:
        m.destroy()
        nogrid.destroy()
    # a flat patch: point-to-point fits it, point-to-plane leaves in-plane motion unconstrained -> degenerate
    g = synth.rng(9)
    flat = np.column_stack([g.uniform(-20, 20, (4000, 2)), np.zeros(4000)])
    fsrc = flat[:300] + [0.3, -0.2, 0.5]
    m = pcreg.Model(flat, grid=True)
    try:
        m.set_normals(np.tile([0.0, 0.0, 1.0], (4000, 1)))
        T0f = np.stack([np.eye(4)] * 2)
        for nn in ("grid", "brute"):
            p = _run(pcreg, m, fsrc, T0f, nn, iters=4, mode=pcreg.ICP_PLAIN, metric="point_to_plane")
            assert np.all(p["status"] == 1) and _eq(p["T"], T0f), nn
            q = _run(pcreg, m, fsrc, T0f, nn, iters=4, mode=pcreg.ICP_PLAIN)
            assert np.all(q["status"] == 0), nn
    finally:
        m.destroy()


@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_point_to_plane_reaches_the_truth_on_a_smooth_model(pcreg, monkeypatch, path):
    model, nrm, src, T_gt, T0 = ellipsoid_problem()
    _setenv(monkeypatch, PATHS[path][2])
    m = pcreg.Model(model, grid=True, voxel_map=1)
    try:
        m.set_normals(nrm)
        out = _run(pcreg, m, src, T0[None], "grid", iters=10, mode=pcreg.ICP_PLAIN, metric="point_to_plane")
    finally:
        m.destroy()
    assert out["status"][0] == 0
    T = out["T"][0]
    assert np.linalg.norm(T[:3, :3] - T_gt[:3, :3], "fro") <= 1e-6
    assert np.linalg.norm(T[3, :3] - T_gt[3, :3]) <= 1e-6
