"""The plane-to-plane (generalized ICP) metric on the GPU (include/pcreg.h: pcreg_icp_batch_gicp{,_dev}) and cloud_normals.

Every path (fused, per-pass, per-pass in two lanes with small chunks, brute force, map-less grid) gives the same bits; the result
matches the FP64 reference (tests/icp_gicp_reference.py) fed with the library's own normals, reaches the truth on a smooth model,
composes with the tolerance stop (a stop after k updates equals an iters = k run), ignores the sign of every normal bit for bit,
does not depend on the device count, and the device entry returns the host entry's bits."""
import ctypes as C

import numpy as np
import pytest

from icp_gicp_reference import ellipsoid_gicp_problem, icp_batch_gicp, unit_rows
from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

ITERS = 12
TOL = (0.01, 0.5)
EPS = 1e-3
OUT_KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


@pytest.fixture(scope="module")
def prob(pcreg):
    """12 poses up to 12 deg / 2 mm from the truth of a 600-point noisy patch on a 20 000-point model; source normals from
    cloud_normals(src, 8)."""
    model = synth.make_model(20_000, 100)
    src, T_gt, c = synth.make_source(model, 600, 0.3, 101)
    T0 = synth.pose_grid(T_gt, c, 3, (2, 2, 1), 12.0, 2.0, 102)
    return model, src, T0, pcreg.cloud_normals(src, 8)


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


def _run(P, m, src, T0, nn, sn, iters=ITERS, **kw):
    kw.setdefault("mode", P.ICP_KNN)
    return P.icp_batch(m, src, T0, iters=iters, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE, return_idx=True, return_hist=True,
                       metric="plane_to_plane", src_normals=sn, **kw)


def _run_raw(P, m, src, T0, sn, eps=EPS, stop=None, iters=4):
    """pcreg_icp_batch_gicp called directly (sn may be None); returns the status code."""
    from pcreg_b200 import _lib as L
    T0 = np.asarray(T0).reshape(-1, 4, 4)
    H, ns = T0.shape[0], src.shape[0]
    a = np.asfortranarray(src, dtype=np.float64)
    n = None if sn is None else np.asfortranarray(sn, dtype=np.float64)
    T0a = np.ascontiguousarray(np.transpose(T0, (0, 2, 1))).reshape(H, 16)
    o = P.icp_opts(P.ICP_KNN, iters, 0.85, 3.5, 0.0, P.NN_GRID)
    T = np.empty((H, 16))
    rmse = np.empty(H)
    return L.lib().pcreg_icp_batch_gicp(m.handle, a.ctypes.data_as(C.c_void_p), 1, ns, ns, None,
                                        None if n is None else n.ctypes.data_as(C.c_void_p), float(eps),
                                        T0a.ctypes.data_as(L.c_f64p), H, C.byref(o), C.byref(stop) if stop is not None else None,
                                        T.ctypes.data_as(L.c_f64p), rmse.ctypes.data_as(L.c_f64p), None, None, None, None, None,
                                        None, None)


@pytest.mark.parametrize("stop", [None, TOL], ids=["fixed", "stop"])
@pytest.mark.parametrize("mode", list(MODES))
def test_paths_agree_bit_for_bit(pcreg, prob, models, monkeypatch, mode, stop):
    _, src, T0, sn = prob
    kw = MODES[mode](pcreg, src)
    res = {}
    for path, (mk, nn, env) in PATHS.items():
        _setenv(monkeypatch, env)
        res[path] = _run(pcreg, models[mk], src, T0, nn, sn, tolerance=stop, **kw)
    ref = res["fused"]
    assert np.all(ref["status"] == 0)
    for path, out in res.items():
        for k in OUT_KEYS + (("n_iter", "converged") if stop else ()):
            assert _eq(out[k], ref[k]), (path, mode, k)
        assert out["best"] == ref["best"]
    # the metric changes the result: neither point-to-plane nor eps = 1 gives these poses
    _setenv(monkeypatch, PATHS["fused"][2])
    plane = pcreg.icp_batch(models["vox"], src, T0, iters=ITERS, nn=pcreg.NN_GRID, metric="point_to_plane", tolerance=stop, **kw)
    assert not _eq(plane["T"], ref["T"])
    one = _run(pcreg, models["vox"], src, T0, "grid", sn, tolerance=stop, gicp_eps=1.0, **kw)
    assert not _eq(one["T"], ref["T"])


@pytest.mark.parametrize("path", ["fused", "brute"])
def test_matches_the_reference(pcreg, prob, models, monkeypatch, path):
    model, src, T0, sn = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    nrm = models[mk].normals()                 # checked on the library's own normals
    ref = icp_batch_gicp(model, nrm, src, unit_rows(sn), T0, eps=EPS, mode=1, iters=ITERS, k_frac=0.85)
    out = _run(pcreg, models[mk], src, T0, nn, sn)
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
def test_stop_equals_fixed_iteration_run(pcreg, prob, models, monkeypatch, path):
    _, src, T0, sn = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    iters = 20
    out = _run(pcreg, models[mk], src, T0, nn, sn, iters=iters, tolerance=TOL)
    stopped = out["n_iter"][out["converged"] == 1]
    assert len(stopped) >= 3 and np.all(stopped < iters), out["n_iter"]
    for k in np.unique(out["n_iter"]):
        g = np.nonzero(out["n_iter"] == k)[0]
        ref = _run(pcreg, models[mk], src, T0[g], nn, sn, iters=int(k))
        for key in ("T", "rmse", "n_used", "status", "idx"):
            assert _eq(out[key][g], ref[key]), (k, key)
        assert _eq(out["rmse_hist"][g, :k + 1], ref["rmse_hist"]), k
        assert _eq(out["rmse_hist"][g, k:], np.repeat(out["rmse"][g, None], iters + 1 - k, axis=1)), k


UPDATES = 10


@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_reaches_the_truth_on_a_smooth_model(pcreg, monkeypatch, path):
    """Noiseless ellipsoid, analytic normals on both sides, start 5 deg / 2 mm off, eps = 1e-3: within 1e-6 of T_gt after
    UPDATES updates."""
    model, nrm, src, sn, T_gt, T0 = ellipsoid_gicp_problem()
    _setenv(monkeypatch, PATHS[path][2])
    m = pcreg.Model(model, grid=True, voxel_map=1)
    try:
        m.set_normals(nrm)
        out = _run(pcreg, m, src, T0[None], "grid", sn, iters=UPDATES, mode=pcreg.ICP_PLAIN)
    finally:
        m.destroy()
    assert out["status"][0] == 0
    T = out["T"][0]
    assert np.linalg.norm(T[:3, :3] - T_gt[:3, :3], "fro") <= 1e-6
    assert np.linalg.norm(T[3, :3] - T_gt[3, :3]) <= 1e-6


@pytest.mark.parametrize("path", ["fused", "per-pass", "brute"])
def test_sign_of_the_normals_changes_no_bit(pcreg, prob, monkeypatch, path):
    model, src, T0, sn = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    g = synth.rng(41)
    base = pcreg.Model(model, grid=True, voxel_map=1)
    flip = pcreg.Model(model, grid=True, voxel_map=1)
    try:
        base.compute_normals(6)
        nrm = base.normals()
        fm = np.where(g.random(nrm.shape[0]) < 0.5, -1.0, 1.0)[:, None]
        fs = np.where(g.random(sn.shape[0]) < 0.5, -1.0, 1.0)[:, None]
        base.set_normals(nrm)                 # both models' normals pass through the same normalisation
        flip.set_normals(nrm * fm)
        ref = _run(pcreg, base, src, T0, nn, sn)
        out = _run(pcreg, flip, src, T0, nn, sn * fs)
    finally:
        base.destroy()
        flip.destroy()
    for k in OUT_KEYS:
        assert _eq(out[k], ref[k]), k
    assert out["best"] == ref["best"]


@pytest.mark.parametrize("stop", [None, TOL], ids=["fixed", "stop"])
@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_device_entry_equals_host_entry(pcreg, prob, models, monkeypatch, path, stop):
    import torch
    from pcreg_b200 import torch_ops
    _, src, T0, sn = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    ref = _run(pcreg, models[mk], src, T0, nn, sn, tolerance=stop)
    dev = torch.device("cuda", 0)
    H, ns = T0.shape[0], src.shape[0]
    bufs = torch_ops.IcpDeviceBuffers(H, ns, ITERS, dev, want_idx=True, want_hist=True, want_n_iter=stop is not None)
    opts = pcreg.icp_opts(pcreg.ICP_KNN, ITERS, 0.85, 3.5, 0.0, pcreg.NN_GRID)
    torch_ops.icp_batch_device(models[mk], torch_ops.src_to_abi_t(torch.from_numpy(src).to(dev)), None,
                               torch_ops.T_to_abi_t(torch.from_numpy(np.asarray(T0)).to(dev)), opts, bufs,
                               stop=pcreg.icp_stop(*stop) if stop else None, metric="plane_to_plane",
                               src_normals=torch.from_numpy(np.ascontiguousarray(sn)).to(dev))
    torch.cuda.synchronize()
    got = dict(T=torch_ops.T_from_abi_t(bufs.T).cpu().numpy(), rmse=bufs.rmse.cpu().numpy(), n_used=bufs.n_used.cpu().numpy(),
               status=bufs.status.cpu().numpy(), idx=bufs.idx.cpu().numpy(), rmse_hist=bufs.hist.cpu().numpy())
    for k in OUT_KEYS:
        assert _eq(got[k], ref[k]), k
    assert int(bufs.best.item()) == ref["best"]
    if stop:
        assert _eq(bufs.n_iter.cpu().numpy(), ref["n_iter"]) and _eq(bufs.converged.cpu().numpy(), ref["converged"])


@pytest.fixture()
def multi(pcreg, monkeypatch):
    monkeypatch.setenv("PCREG_ALLOW_DUP_DEVICES", "1")
    yield pcreg
    pcreg.init(0)


def test_results_do_not_depend_on_device_count(multi, prob):
    P = multi
    model, src, T0, sn = prob
    cases = [dict(nn="grid"), dict(nn="brute"), dict(nn="grid", tolerance=TOL)]
    ref = None
    for devs in ([0], [0, 0], [0, 0, 0]):
        P.init(devs)
        m = P.Model(model, grid=True)
        try:
            m.compute_normals(6)
            got = [_run(P, m, src, T0, sn=sn, **kw) for kw in cases]
        finally:
            m.destroy()
        if ref is None:
            ref = got
            continue
        for kw, a, r in zip(cases, got, ref):
            for k in OUT_KEYS + (("n_iter", "converged") if "tolerance" in kw else ()):
                assert _eq(a[k], r[k]), (devs, kw, k)
            assert a["best"] == r["best"]


def test_errors_and_degenerate(pcreg, prob):
    import torch
    from pcreg_b200 import torch_ops
    model, src, T0, sn = prob
    m = pcreg.Model(model, grid=True)
    try:
        # no model normals: PCREG_ERR_STATE
        assert _run_raw(pcreg, m, src, T0[:2], sn) == -4
        with pytest.raises(pcreg.PcregError):
            _run(pcreg, m, src, T0[:2], "grid", sn)
        m.compute_normals(6)
        assert _run_raw(pcreg, m, src, T0[:2], sn) == 0
        # source normals: NULL, a zero row, a NaN row
        assert _run_raw(pcreg, m, src, T0[:2], None) == -1
        for bad in ([0.0, 0.0, 0.0], [np.nan, 0.0, 1.0], [np.inf, 0.0, 0.0]):
            n = sn.copy()
            n[123] = bad
            assert _run_raw(pcreg, m, src, T0[:2], n) == -1, bad
        # eps outside (0, 1] or not finite
        for eps in (0.0, -1.0, 1.5, np.nan, np.inf):
            assert _run_raw(pcreg, m, src, T0[:2], sn, eps=eps) == -1, eps
        assert _run_raw(pcreg, m, src, T0[:2], sn, eps=1.0) == 0
        # a bad stop
        for stop in (pcreg.icp_stop(-1.0, 0.5), pcreg.icp_stop(np.nan, 0.5), pcreg.icp_stop(0.01, 0.5, 0), pcreg.icp_stop(0.01, 0.5, 17)):
            assert _run_raw(pcreg, m, src, T0[:2], sn, stop=stop) == -1
        # the Python layer asks for the source normals instead of computing them
        with pytest.raises(ValueError):
            pcreg.icp_batch(m, src, T0[:2], metric="plane_to_plane")
        # the device entry validates on the device
        dev = torch.device("cuda", 0)
        bufs = torch_ops.IcpDeviceBuffers(2, src.shape[0], 4, dev)
        opts = pcreg.icp_opts(pcreg.ICP_KNN, 4, 0.85, 3.5, 0.0, pcreg.NN_GRID)
        args = (m, torch_ops.src_to_abi_t(torch.from_numpy(src).to(dev)), None,
                torch_ops.T_to_abi_t(torch.from_numpy(np.asarray(T0[:2])).to(dev)), opts, bufs)
        n = sn.copy()
        n[5] = 0.0
        with pytest.raises(pcreg.PcregError):
            torch_ops.icp_batch_device(*args, metric="plane_to_plane", src_normals=torch.from_numpy(n).to(dev))
        with pytest.raises(pcreg.PcregError):
            torch_ops.icp_batch_device(*args, metric="plane_to_plane", src_normals=torch.from_numpy(sn).to(dev), gicp_eps=0.0)
        torch_ops.icp_batch_device(*args, metric="plane_to_plane", src_normals=torch.from_numpy(np.ascontiguousarray(sn)).to(dev))
        # fewer than 6 usable correspondences: status 1, pose frozen
        T0f = np.asarray(T0[:2])
        few = _run(pcreg, m, src[:5], T0f, "grid", sn[:5], iters=3, mode=pcreg.ICP_PLAIN)
        assert np.all(few["status"] == 1) and _eq(few["T"], T0f)
    finally:
        m.destroy()


@pytest.mark.parametrize("viewpoint", [None, (0.0, 0.0, 500.0)])
def test_cloud_normals_equals_model_compute_normals(pcreg, prob, viewpoint):
    model = prob[0]
    m = pcreg.Model(model, grid=True)
    try:
        m.compute_normals(6, viewpoint)
        want = m.normals()
    finally:
        m.destroy()
    got = pcreg.cloud_normals(model, 6, viewpoint)
    assert got.shape == want.shape and _eq(got, want)
    # the source normals used above are unit rows with the default orientation (away from the bounding-box centre)
    sn = prob[3]
    assert np.allclose(np.linalg.norm(sn, axis=1), 1.0, rtol=0, atol=1e-15)
