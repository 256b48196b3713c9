"""Batched ICP over many matching windows in one call (include/pcreg.h: pcreg_icp_batch_windows{,_dev}).

The defining property: window w's results equal, bit for bit, what icp_batch returns for (src_w, w_src_w, T0 of w) alone -- T,
rmse, n_used, status, best, idx, rmse_hist, n_iter and converged -- for every mode, metric and ICP path, with or without the
tolerance stop, whatever the device count and whether the call runs as one fused launch or as a loop over the windows."""
import ctypes as C
import math

import numpy as np
import pytest

from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

ITERS = 10
TOL = (0.01, 0.5)
OUT_KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


@pytest.fixture(scope="module")
def prob():
    """Deliberately uneven windows of one model: 3000 points (listed before a smaller one), 40 points (below the sort's 64),
    one without hypotheses, 1500 points, and two overlapping crops of one cloud."""
    model = synth.make_model(20_000, 100)
    srcs, T0s = [], []
    for ns, seed, nh in ((3000, 201, 3), (40, 202, 2), (500, 203, 0), (1500, 204, 2)):
        src, T_gt, c = synth.make_source(model, ns, 0.3, seed)
        srcs.append(src)
        T0s.append(synth.pose_grid(T_gt, c, nh, (1, 1, 1), 8.0, 1.0, seed + 50)[:nh].reshape(-1, 4, 4))
    src, T_gt, c = synth.make_source(model, 1200, 0.3, 205)
    grid = synth.pose_grid(T_gt, c, 2, (2, 1, 1), 8.0, 1.0, 255)
    srcs += [src[:800], src[400:]]
    T0s += [grid[:2], grid[2:]]
    return model, srcs, T0s


@pytest.fixture(scope="module")
def normals(prob):
    from pcreg_b200 import api
    return [api.cloud_normals(s) for s in prob[1]]


@pytest.fixture()
def models(pcreg, prob):
    """Per test: the device-count test re-initialises the library, which invalidates model handles."""
    model = prob[0]
    ms = dict(vox=pcreg.Model(model, grid=True, voxel_map=1), novox=pcreg.Model(model, grid=True, voxel_map=-1))
    for m in ms.values():
        m.compute_normals()
    yield ms
    for m in ms.values():
        m.destroy()


# path -> (model, nn, environment)
PATHS = {
    "fused": ("vox", "grid", {"PCREG_FUSED": "1"}),
    "per-pass": ("vox", "grid", {"PCREG_FUSED": "0"}),
    "brute": ("vox", "brute", {}),
    "grid-novox": ("novox", "grid", {}),
}


def _setenv(monkeypatch, env):
    for k in ("PCREG_FUSED", "PCREG_LANES", "PCREG_MAX_CHUNK_HYP"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


MODES = {
    "plain": lambda P, src: dict(mode=P.ICP_PLAIN, thDist2=9.0),
    "knn": lambda P, src: dict(mode=P.ICP_KNN, k_frac=0.85),
    "weighted": lambda P, src: dict(mode=P.ICP_WEIGHTED, R_w=3.5, w_src=synth.rng(77 + src.shape[0]).uniform(0.5, 1.0, src.shape[0])),
}


def _per_window_kw(P, srcs, mode, metric, nrm):
    """The keywords of icp_batch for each window alone (w_src / src_normals of that window)."""
    out = []
    for k, s in enumerate(srcs):
        kw = MODES[mode](P, s)
        kw["metric"] = metric
        if metric == "plane_to_plane":
            kw["src_normals"] = nrm[k]
        out.append(kw)
    return out


def _windows(P, m, srcs, T0s, nn, kws, **extra):
    """One windowed call with the per-window keywords gathered into lists."""
    kw = {k: v for k, v in kws[0].items() if k not in ("w_src", "src_normals")}
    if "w_src" in kws[0]:
        kw["w_src_list"] = [k["w_src"] for k in kws]
    if "src_normals" in kws[0]:
        kw["src_normals_list"] = [k["src_normals"] for k in kws]
    return P.icp_batch_windows(m, srcs, T0s, iters=ITERS, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE, return_idx=True,
                               return_hist=True, **kw, **extra)


def _check_per_window(P, m, srcs, T0s, nn, kws, got, **extra):
    assert len(got) == len(srcs)
    for w, (s, T0, kw, g) in enumerate(zip(srcs, T0s, kws, got)):
        if T0.shape[0] == 0:
            assert g["best"] == -1 and g["T"].shape == (0, 4, 4) and g["idx"].shape == (0, s.shape[0]), w
            continue
        ref = P.icp_batch(m, s, T0, iters=ITERS, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE, return_idx=True, return_hist=True,
                          **kw, **extra)
        keys = OUT_KEYS + (("n_iter", "converged") if "tolerance" in extra else ())
        for k in keys:
            assert _eq(g[k], ref[k]), (w, k)
        assert g["best"] == ref["best"], w


@pytest.mark.parametrize("tol", [None, TOL], ids=["fixed", "tolerance"])
@pytest.mark.parametrize("metric", ["point_to_point", "point_to_plane", "plane_to_plane"])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("path", list(PATHS))
def test_each_window_equals_its_own_call(pcreg, prob, normals, models, monkeypatch, path, mode, metric, tol):
    _, srcs, T0s = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    kws = _per_window_kw(pcreg, srcs, mode, metric, normals)
    extra = {} if tol is None else dict(tolerance=tol)
    pcreg.set_profiling(True)
    try:
        got = _windows(pcreg, models[mk], srcs, T0s, nn, kws, **extra)
        fused = pcreg.last_profile()["fused"]
    finally:
        pcreg.set_profiling(False)
    assert fused == (1.0 if path == "fused" else 0.0)
    _check_per_window(pcreg, models[mk], srcs, T0s, nn, kws, got, **extra)


def test_profile_of_the_loop_sums_the_windows(pcreg, prob, models, monkeypatch):
    _, srcs, T0s = prob
    _setenv(monkeypatch, {"PCREG_FUSED": "0"})
    kws = _per_window_kw(pcreg, srcs, "knn", "point_to_point", None)
    pcreg.set_profiling(True)
    try:
        _windows(pcreg, models["vox"], srcs, T0s, "grid", kws)
        p = pcreg.last_profile()
        want = dict(nn_launches=0.0, update_launches=0.0, nn_queries=0.0, correspondences=0.0)
        for s, T0 in zip(srcs, T0s):
            if T0.shape[0]:
                pcreg.icp_batch(models["vox"], s, T0, mode=pcreg.ICP_KNN, iters=ITERS, nn=pcreg.NN_GRID)
                q = pcreg.last_profile()
                for k in want:
                    want[k] += q[k]
    finally:
        pcreg.set_profiling(False)
    assert p["fused"] == 0.0 and p["voxel_map"] == 1.0
    for k, v in want.items():
        assert p[k] == v, (k, p[k], v)
    assert want["nn_launches"] == 5 * (ITERS + 1)


def test_window_too_large_for_the_fused_kernel_loops(pcreg, prob, models, monkeypatch):
    """KNN mode keeps 12 bytes per source point in shared memory: a window of 18 000 points cannot run fused, so the whole call
    loops over the windows (even with PCREG_FUSED=1), with the same per-window bits."""
    model, srcs, T0s = prob
    big, T_gt, c = synth.make_source(model, 18_000, 0.3, 301)
    s2 = [srcs[1], big, srcs[3]]
    t2 = [T0s[1], synth.pose_grid(T_gt, c, 2, (1, 1, 1), 5.0, 1.0, 302), T0s[3]]
    kws = _per_window_kw(pcreg, s2, "knn", "point_to_point", None)
    for env in ({}, {"PCREG_FUSED": "1"}):
        _setenv(monkeypatch, env)
        pcreg.set_profiling(True)
        try:
            got = _windows(pcreg, models["vox"], s2, t2, "grid", kws)
            assert pcreg.last_profile()["fused"] == 0.0
        finally:
            pcreg.set_profiling(False)
        _check_per_window(pcreg, models["vox"], s2, t2, "grid", kws, got)


@pytest.fixture()
def multi(pcreg, monkeypatch):
    monkeypatch.setenv("PCREG_ALLOW_DUP_DEVICES", "1")
    yield pcreg
    pcreg.init(0)


def test_results_do_not_depend_on_device_count(multi, prob, normals):
    """11 hypotheses over offsets [0, 3, 5, 5, 7, 9, 11]: 2 slots split window 3, 3 slots split windows 1 and 4."""
    P = multi
    model, srcs, T0s = prob
    cases = [("grid", "knn", "point_to_point", None), ("grid", "weighted", "plane_to_plane", TOL), ("brute", "plain", "point_to_point", TOL)]
    P.init(0)
    m = P.Model(model, grid=True)
    m.compute_normals()
    ref = []
    for nn, mode, metric, tol in cases:
        ref.append(_windows(P, m, srcs, T0s, nn, _per_window_kw(P, srcs, mode, metric, normals), **({} if tol is None else dict(tolerance=tol))))
    m.destroy()
    for devs in ([0, 0], [0, 0, 0]):
        P.init(devs)
        m = P.Model(model, grid=True)
        m.compute_normals()
        for (nn, mode, metric, tol), r in zip(cases, ref):
            extra = {} if tol is None else dict(tolerance=tol)
            a = _windows(P, m, srcs, T0s, nn, _per_window_kw(P, srcs, mode, metric, normals), **extra)
            for w in range(len(srcs)):
                for k in OUT_KEYS + (("n_iter", "converged") if tol else ()):
                    assert _eq(a[w][k], r[w][k]), (devs, nn, w, k)
                assert a[w]["best"] == r[w]["best"]
        m.destroy()


@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_device_entry_equals_host_entry(pcreg, prob, normals, models, monkeypatch, path):
    import torch
    from pcreg_b200 import torch_ops
    _, srcs, T0s = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    m = models[mk]
    kws = _per_window_kw(pcreg, srcs, "weighted", "plane_to_plane", normals)
    host = _windows(pcreg, m, srcs, T0s, nn, kws, tolerance=TOL)
    dev = torch.device("cuda", 0)
    cat = np.concatenate(srcs)
    src_cm = torch_ops.src_to_abi_t(torch.as_tensor(cat, device=dev))
    w = torch.as_tensor(np.concatenate([k["w_src"] for k in kws]), device=dev)
    sn = torch.as_tensor(np.concatenate(normals), device=dev)
    T0 = np.concatenate(T0s)
    T0_abi = torch_ops.T_to_abi_t(torch.as_tensor(T0, device=dev)).reshape(-1, 16).contiguous()
    ns = np.array([s.shape[0] for s in srcs])
    H = np.array([t.shape[0] for t in T0s])
    soff, hoff = np.concatenate([[0], np.cumsum(ns)]), np.concatenate([[0], np.cumsum(H)])
    out = torch_ops.IcpWindowsDeviceBuffers(int(H.sum()), int((H * ns).sum()), len(srcs), ITERS, dev, want_idx=True, want_hist=True,
                                            want_n_iter=True)
    o = pcreg.icp_opts(pcreg.ICP_WEIGHTED, ITERS, R_w=3.5, nn=pcreg.NN_GRID)
    torch_ops.icp_windows_device(m, src_cm, soff, w, T0_abi, hoff, o, out, stop=pcreg.icp_stop(*TOL, 3), metric="plane_to_plane",
                                 src_normals=sn)
    torch.cuda.synchronize()
    T = torch_ops.T_from_abi_t(out.T).cpu().numpy()
    idx = out.idx.cpu().numpy()
    io = np.concatenate([[0], np.cumsum(H * ns)])
    best = out.best.cpu().numpy()
    for k in range(len(srcs)):
        a, b = hoff[k], hoff[k + 1]
        assert np.array_equal(T[a:b], host[k]["T"])
        for key, v in (("rmse", out.rmse), ("n_used", out.n_used), ("status", out.status), ("rmse_hist", out.hist), ("n_iter", out.n_iter),
                       ("converged", out.converged)):
            assert _eq(v.cpu().numpy()[a:b], host[k][key]), (k, key)
        assert np.array_equal(idx[io[k]:io[k + 1]].reshape(b - a, ns[k]), host[k]["idx"]), k
        assert best[k] == host[k]["best"], k


def test_argument_and_state_errors(pcreg, prob, models):
    from pcreg_b200 import _lib as L
    model, srcs, T0s = prob
    lib = L.lib()
    m = models["vox"]
    s = [srcs[0][:200], srcs[3][:100]]
    cat = np.asfortranarray(np.concatenate(s))
    T0 = np.ascontiguousarray(np.transpose(np.concatenate([T0s[0][:1], T0s[3][:1]]), (0, 2, 1))).reshape(2, 16)
    nrm = np.asfortranarray(np.ones_like(cat))
    T = np.empty((2, 16))
    o = pcreg.icp_opts(pcreg.ICP_KNN, 3, nn=pcreg.NN_GRID)
    i64 = lambda x: None if x is None else np.ascontiguousarray(x, dtype=np.int64).ctypes.data_as(L.c_i64p)  # noqa: E731
    f64 = lambda x: x.ctypes.data_as(L.c_f64p)  # noqa: E731

    def call(mm=m, soff=(0, 200, 300), hoff=(0, 1, 2), nwin=2, metric=0, n=None, eps=1e-3, stop=None):
        so, ho = (None if soff is None else np.asarray(soff, dtype=np.int64)), (None if hoff is None else np.asarray(hoff, dtype=np.int64))
        return lib.pcreg_icp_batch_windows(mm.handle, cat.ctypes.data_as(C.c_void_p), 1, cat.shape[0], i64(so), None,
                                           None if n is None else n.ctypes.data_as(C.c_void_p), eps, i64(ho), nwin, f64(T0), C.byref(o),
                                           metric, None if stop is None else C.byref(stop), f64(T), None, None, None, None, None, None,
                                           None, None)

    assert call() == 0 and call(metric=1) == 0 and call(metric=2, n=nrm) == 0
    for kw in (dict(soff=None), dict(hoff=None), dict(soff=(1, 200, 300)), dict(hoff=(1, 1, 2)), dict(soff=(0, 301, 300)),
               dict(hoff=(0, 2, 1)), dict(nwin=0), dict(soff=(0, 300, 300)), dict(metric=3), dict(metric=-1), dict(metric=2),
               dict(metric=2, n=nrm, eps=0.0), dict(metric=2, n=nrm, eps=math.nan), dict(metric=2, n=nrm, eps=1.5),
               dict(stop=pcreg.icp_stop(-1.0, 0.5, 3)), dict(stop=pcreg.icp_stop(0.01, 0.5, 17))):
        assert call(**kw) == -1, kw                                        # PCREG_ERR_ARG
    for bad in (0.0, math.nan, math.inf):
        n2 = nrm.copy(order="F")                                           # the ABI reads it column-major
        n2[250] = bad
        assert call(metric=2, n=n2) == -1, bad
    plain = pcreg.Model(model, grid=True, voxel_map=1)                    # no normals
    try:
        assert call(mm=plain, metric=1) == -4 and call(mm=plain, metric=2, n=nrm) == -4       # PCREG_ERR_STATE
        assert call(mm=plain) == 0
    finally:
        plain.destroy()
    # the single-source metric entry keeps rejecting the plane-to-plane value
    a = np.ascontiguousarray(s[0].T).ravel()
    assert lib.pcreg_icp_batch_metric(m.handle, a.ctypes.data_as(C.c_void_p), 1, 200, 200, None, f64(T0[:1].copy()), 1, C.byref(o), 2, None,
                                      f64(T), None, None, None, None, None, None, None, None) == -1
    with pytest.raises(ValueError):
        pcreg.icp_batch_windows(m, s, [T0s[0][:1], T0s[3][:1]], metric="plane_to_plane")


def test_ransac_then_icp_windows_end_to_end(pcreg):
    """A scene cut into matching windows: pcreg_ransac_batch on each window's putative matches, then one icp_batch_windows call
    polishing a small pose grid around each RANSAC pose against the window's own source cloud.  Every window's best polished pose is
    closer to its ground truth than its RANSAC pose (the test_gpu_pipeline.py criteria)."""
    g = synth.rng(31)
    model = synth.make_model(200_000, 30)
    srcs, truth, centres, p1s, p2s = [], [], [], [], []
    for w in range(5):
        src, T_gt, c = synth.make_source(model, int(g.integers(2000, 4000)), 0.02, 400 + w)
        kp = src[g.choice(src.shape[0], 120, replace=False)]
        p1 = synth.apply_T(kp, T_gt) + g.normal(0.0, 0.15, kp.shape)      # model-side detections of the same spots
        out = g.choice(120, 40, replace=False)
        p1[out] = g.uniform(0, 1, (40, 3)) * synth.BOX
        srcs.append(src); truth.append(T_gt); centres.append(c); p1s.append(p1); p2s.append(kp)
    rs = pcreg.ransac_batch(p1s, p2s, dict(iterNum=2000, thDist=0.2, thInlrRatio=0.1, REFINE=True))
    T0s = [synth.pose_grid(r["T"], c, 2, (2, 1, 1), 1.0, 0.2, 500 + k) for k, (r, c) in enumerate(zip(rs, centres))]
    m = pcreg.Model(model, grid=True)
    try:
        got = pcreg.icp_batch_windows(m, srcs, T0s, mode=pcreg.ICP_KNN, iters=20, nn=pcreg.NN_GRID)
    finally:
        m.destroy()
    for k, (src, T_gt, r, g_) in enumerate(zip(srcs, truth, rs, got)):
        assert r["T"] is not None, k
        Tp = g_["T"][g_["best"]]
        err_ransac = np.linalg.norm(synth.apply_T(src, r["T"]) - synth.apply_T(src, T_gt), axis=1).mean()
        err_icp = np.linalg.norm(synth.apply_T(src, Tp) - synth.apply_T(src, T_gt), axis=1).mean()
        assert err_icp < 0.05 and err_icp < err_ransac, (k, err_ransac, err_icp)
        assert g_["rmse"][g_["best"]] < 0.06, k
