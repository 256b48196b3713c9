"""The ICP pose extrapolation on the GPU (include/pcreg.h: pcreg_icp_extrap, pcreg_icp_batch_extrap{,_dev}).

ex = NULL returns the bits of pcreg_icp_batch / pcreg_icp_batch_windows; with extrapolation every path (fused, per-pass, two lanes,
brute force, map-less grid with lazy trimming) returns the same bits; a hypothesis stopped after k updates is the extrapolating call
with iters = k; the decisions are the FP64 reference's (tests/icp_extrap_reference.py) replayed on the GPU's own poses; each window is
its own one-window call; results do not depend on the device count; bad arguments are rejected."""
import ctypes as C
import math

import numpy as np
import pytest

from icp_extrap_reference import BRANCH_NONE, BRANCH_V1, BRANCH_V2, BRANCH_VMAX, icp_single_extrap
from oracle.nn import KDTreeNN
from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

ITERS = 20
TOL = (0.01, 0.5)
OUT_KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


@pytest.fixture(scope="module")
def prob():
    """12 poses up to 12 deg / 2 mm from the truth; point-to-point creeps along the patch, and the extrapolation takes each branch."""
    model = synth.make_model(20_000, 100)
    src, T_gt, c = synth.make_source(model, 600, 0.3, 101)
    T0 = synth.pose_grid(T_gt, c, 3, (2, 2, 1), 12.0, 2.0, 102)
    return model, src, T0


@pytest.fixture()
def models(pcreg, prob):
    model = prob[0]
    ms = dict(vox=pcreg.Model(model, grid=True, voxel_map=1), novox=pcreg.Model(model, grid=True, voxel_map=-1))
    yield ms
    for m in ms.values():
        m.destroy()


# path -> (model, nn, environment), as the tolerance stop's tests
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


def _run(P, m, src, T0, nn, iters=ITERS, tolerance=None, extrapolate=True, **kw):
    kw.setdefault("mode", P.ICP_KNN)
    return P.icp_batch(m, src, T0, iters=iters, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE, return_idx=True, return_hist=True,
                       tolerance=tolerance, extrapolate=extrapolate, **kw)


def _raw(P, m, src, T0, nn, ex, stop=None, iters=ITERS, mode=None, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src=None, n_extrap=True):
    """pcreg_icp_batch_extrap with one window through ctypes (ex may be None) -> (rc, outputs)."""
    from pcreg_b200 import _lib as L
    f64 = lambda x: x.ctypes.data_as(L.c_f64p) if x is not None else None  # noqa: E731
    i32 = lambda x: x.ctypes.data_as(L.c_i32p) if x is not None else None  # noqa: E731
    ns, H = src.shape[0], T0.shape[0]
    a = np.asfortranarray(np.asarray(src, dtype=np.float64))
    T0a = np.ascontiguousarray(np.transpose(np.asarray(T0, dtype=np.float64), (0, 2, 1))).reshape(H, 16)
    o = P.icp_opts(P.ICP_KNN if mode is None else mode, iters, k_frac, R_w, thDist2, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE)
    soff, hoff = np.array([0, ns], dtype=np.int64), np.array([0, H], dtype=np.int64)
    T = np.empty((H, 16))
    rmse, hist = np.empty(H), np.empty((H, iters + 1))
    n_used, status, idx = np.empty(H, np.int32), np.empty(H, np.int32), np.empty((H, ns), np.int32)
    n_iter, conv, nex = np.empty(H, np.int32), np.empty(H, np.int32), np.full(H, -7, np.int32) if n_extrap else None
    best = np.empty(1, np.int64)
    w = None if w_src is None else np.ascontiguousarray(w_src, dtype=np.float64)
    rc = L.lib().pcreg_icp_batch_extrap(m.handle, a.ctypes.data_as(C.c_void_p), 1, ns, soff.ctypes.data_as(L.c_i64p), f64(w),
                                        hoff.ctypes.data_as(L.c_i64p), 1, f64(T0a), C.byref(o), C.byref(stop) if stop is not None else None,
                                        C.byref(ex) if ex is not None else None, f64(T), f64(rmse), i32(n_used), i32(status), i32(idx),
                                        f64(hist), best.ctypes.data_as(L.c_i64p), i32(n_iter), i32(conv), i32(nex))
    out = dict(T=np.transpose(T.reshape(H, 4, 4), (0, 2, 1)), rmse=rmse, n_used=n_used, status=status, idx=idx, rmse_hist=hist,
               best=int(best[0]), n_iter=n_iter, converged=conv, n_extrap=nex)
    return rc, out


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("mode", list(MODES))
def test_null_ex_returns_the_existing_bits(pcreg, prob, models, monkeypatch, path, mode):
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    kw = MODES[mode](pcreg, src)
    ref = _run(pcreg, models[mk], src, T0, nn, iters=12, extrapolate=False, **kw)
    win = pcreg.icp_batch_windows(models[mk], [src], [T0], iters=12, nn=pcreg.NN_GRID if nn == "grid" else pcreg.NN_BRUTE, return_idx=True,
                                  return_hist=True, w_src_list=None if kw.get("w_src") is None else [kw["w_src"]],
                                  **{k: v for k, v in kw.items() if k != "w_src"})[0]
    rc, out = _raw(pcreg, models[mk], src, T0, nn, None, iters=12, **kw)
    assert rc == 0
    for k in OUT_KEYS:
        assert _eq(out[k], ref[k]) and _eq(out[k], win[k]), (path, mode, k)
    assert out["best"] == ref["best"] == win["best"]
    assert np.all(out["n_extrap"] == -7)                     # written only with ex
    if mode == "knn":                                        # with a stop too: the bits of pcreg_icp_batch_stop
        stop = _run(pcreg, models[mk], src, T0, nn, tolerance=TOL, extrapolate=False, **kw)
        rc, out = _raw(pcreg, models[mk], src, T0, nn, None, stop=pcreg.icp_stop(*TOL), **kw)
        assert rc == 0
        for k in OUT_KEYS + ("n_iter", "converged"):
            assert _eq(out[k], stop[k]), (path, k)


@pytest.mark.parametrize("tol", [None, TOL])
@pytest.mark.parametrize("mode", list(MODES))
def test_every_path_gives_the_same_bits(pcreg, prob, models, monkeypatch, mode, tol):
    _, src, T0 = prob
    kw = MODES[mode](pcreg, src)
    outs = {}
    for path, (mk, nn, env) in PATHS.items():
        _setenv(monkeypatch, env)
        if path == "grid-novox" and mode == "knn":
            pcreg.set_profiling(True)            # lazy trimming is active on this path: it skips searches
            try:
                outs[path] = _run(pcreg, models[mk], src, T0, nn, tolerance=tol, **kw)
                assert pcreg.last_profile()["lazy_skipped_queries"] > 0
            finally:
                pcreg.set_profiling(False)
        else:
            outs[path] = _run(pcreg, models[mk], src, T0, nn, tolerance=tol, **kw)
    ref = outs["fused"]
    assert np.any(ref["n_extrap"] > 0) and np.any(ref["status"] == 0)
    for path, out in outs.items():
        for k in OUT_KEYS + ("n_extrap",) + (("n_iter", "converged") if tol else ()):
            assert _eq(out[k], ref[k]), (path, mode, k)
        assert out["best"] == ref["best"]


@pytest.mark.parametrize("path", ["fused", "per-pass", "brute"])
def test_stop_at_k_equals_the_iters_k_call(pcreg, prob, models, monkeypatch, path):
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    out = _run(pcreg, models[mk], src, T0, nn, tolerance=TOL)
    assert np.any(out["converged"] == 1) and np.any(out["n_extrap"] > 0)
    for k in np.unique(out["n_iter"]):
        g = np.nonzero(out["n_iter"] == k)[0]
        ref = _run(pcreg, models[mk], src, T0[g], nn, iters=int(k))
        for key in ("T", "rmse", "n_used", "status", "idx", "n_extrap"):
            assert _eq(out[key][g], ref[key]), (k, key)
        assert _eq(out["rmse_hist"][g, :k + 1], ref["rmse_hist"]), k


def test_decisions_match_the_reference_on_the_gpu_poses(pcreg, prob, models, monkeypatch):
    """Poses T_0..T_K from iters = 0..K calls; update u extrapolated on the GPU when n_extrap grew from the iters = u - 1 call.  The
    reference replayed on those poses takes the same decision wherever it is not within 1e-9 of a threshold, and its jump lands where
    the GPU's does."""
    model, src, T0 = prob
    mk, nn, env = PATHS["fused"]
    _setenv(monkeypatch, env)
    kw = dict(mode=pcreg.ICP_PLAIN, thDist2=9.0)
    runs = [_run(pcreg, models[mk], src, T0, nn, iters=k, **kw) for k in range(ITERS + 1)]
    tree = KDTreeNN(np.asarray(model, dtype=np.float64))
    seen, compared = set(), 0
    for h in range(T0.shape[0]):
        if runs[-1]["status"][h] != 0:
            continue
        poses = [r["T"][h] for r in runs]
        ref = icp_single_extrap(model, src, T0[h], replay=poses, nn=tree, **kw)
        for t in ref["trace"]:
            u = t["u"]
            gpu = runs[u]["n_extrap"][h] - runs[u - 1]["n_extrap"][h]
            if t["margin"] <= 1e-9:
                continue
            compared += 1
            assert gpu == (t["branch"] != BRANCH_NONE), (h, u, t)
            seen.add(t["branch"])
            if gpu:
                R, Rr = poses[u][:3, :3], t["T"][:3, :3]
                assert np.linalg.norm(R - Rr) <= 1e-6 and np.linalg.norm(poses[u][3, :3] - t["T"][3, :3]) <= 1e-6 * max(1.0, np.linalg.norm(t["T"][3, :3]))
    assert compared > 100 and {BRANCH_V1, BRANCH_V2, BRANCH_VMAX} <= seen, (compared, seen)


def _windows(src, T0):
    """Three windows: two crops of the source and the whole of it, uneven pose counts."""
    return [src[:250], src[200:], src], [T0[:3], T0[3:8], T0[8:]]


@pytest.mark.parametrize("fused", ["1", "0"])
def test_each_window_is_its_own_call(pcreg, prob, models, monkeypatch, fused):
    _, src, T0 = prob
    _setenv(monkeypatch, {"PCREG_FUSED": fused})
    srcs, T0s = _windows(src, T0)
    m = models["vox"]
    pcreg.set_profiling(2)
    try:
        outs = pcreg.icp_batch_windows(m, srcs, T0s, mode=pcreg.ICP_KNN, iters=ITERS, nn=pcreg.NN_GRID, return_idx=True, return_hist=True,
                                       extrapolate=True)
        assert pcreg.last_profile()["fused"] == (1.0 if fused == "1" else 0.0)
    finally:
        pcreg.set_profiling(False)
    assert sum(int(o["n_extrap"].sum()) for o in outs) > 0
    for s, t, o in zip(srcs, T0s, outs):
        one = _run(pcreg, m, s, t, "grid")
        for k in OUT_KEYS + ("n_extrap",):
            assert _eq(o[k], one[k]), k
        assert o["best"] == one["best"]


@pytest.fixture()
def multi(pcreg, monkeypatch):
    monkeypatch.setenv("PCREG_ALLOW_DUP_DEVICES", "1")
    yield pcreg
    pcreg.init(0)


def test_results_do_not_depend_on_device_count(multi, prob):
    P = multi
    model, src, T0 = prob
    srcs, T0s = _windows(src, T0)
    P.init(0)
    m = P.Model(model, grid=True)
    ref = P.icp_batch_windows(m, srcs, T0s, mode=P.ICP_KNN, iters=ITERS, nn=P.NN_GRID, return_idx=True, return_hist=True, tolerance=TOL,
                              extrapolate=True)
    m.destroy()
    for devs in ([0, 0], [0, 0, 0]):
        P.init(devs)
        m = P.Model(model, grid=True)
        outs = P.icp_batch_windows(m, srcs, T0s, mode=P.ICP_KNN, iters=ITERS, nn=P.NN_GRID, return_idx=True, return_hist=True,
                                   tolerance=TOL, extrapolate=True)
        for a, r in zip(outs, ref):
            for k in OUT_KEYS + ("n_iter", "converged", "n_extrap"):
                assert _eq(a[k], r[k]), (devs, k)
        m.destroy()


@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_device_entry_equals_host_entry(pcreg, prob, models, monkeypatch, path):
    import torch
    from pcreg_b200 import torch_ops
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    m = models[mk]
    host = _run(pcreg, m, src, T0, nn, tolerance=TOL)
    dev = torch.device("cuda", 0)
    src_cm = torch_ops.src_to_abi_t(torch.as_tensor(src, device=dev))
    T0_abi = torch_ops.T_to_abi_t(torch.as_tensor(np.asarray(T0), device=dev)).reshape(-1, 16).contiguous()
    H, ns = T0.shape[0], src.shape[0]
    out = torch_ops.IcpDeviceBuffers(H, ns, ITERS, dev, want_idx=True, want_hist=True, want_n_iter=True, want_n_extrap=True)
    o = pcreg.icp_opts(pcreg.ICP_KNN, ITERS, 0.85, nn=pcreg.NN_GRID)
    torch_ops.icp_batch_device(m, src_cm, None, T0_abi, o, out, stop=pcreg.icp_stop(*TOL, 3), extrap=pcreg.icp_extrap())
    torch.cuda.synchronize()
    assert np.array_equal(torch_ops.T_from_abi_t(out.T).cpu().numpy(), host["T"])
    for k, v in (("rmse", out.rmse), ("n_used", out.n_used), ("status", out.status), ("idx", out.idx), ("rmse_hist", out.hist),
                 ("n_iter", out.n_iter), ("converged", out.converged), ("n_extrap", out.n_extrap)):
        assert _eq(v.cpu().numpy(), host[k]), k
    assert int(out.best.item()) == host["best"]
    # the windows device entry: the same for a two-window split of the poses
    wout = torch_ops.IcpWindowsDeviceBuffers(H, H * ns, 2, ITERS, dev, want_idx=True, want_n_extrap=True)
    src2 = torch.cat([src_cm, src_cm], dim=1).contiguous()
    torch_ops.icp_windows_device(m, src2, [0, ns, 2 * ns], None, T0_abi, [0, 5, H], o, wout, extrap=pcreg.icp_extrap())
    torch.cuda.synchronize()
    plain = _run(pcreg, m, src, T0, nn)
    assert np.array_equal(torch_ops.T_from_abi_t(wout.T).cpu().numpy(), plain["T"])
    assert _eq(wout.n_extrap.cpu().numpy(), plain["n_extrap"])


def test_argument_errors(pcreg, prob, models):
    _, src, T0 = prob
    m = models["vox"]
    for bad in ((0.0, 25.0), (-1.0, 25.0), (180.5, 25.0), (math.nan, 25.0), (10.0, 0.0), (10.0, -1.0), (10.0, math.inf), (10.0, math.nan)):
        rc, _ = _raw(pcreg, m, src, T0[:1], "grid", pcreg.icp_extrap(*bad), iters=3)
        assert rc == -1, bad                                  # PCREG_ERR_ARG
        with pytest.raises(pcreg.PcregError):
            _run(pcreg, m, src, T0[:1], "grid", iters=3, extrapolate=bad)
    assert _raw(pcreg, m, src, T0[:1], "grid", pcreg.icp_extrap(180.0, 1e-3), iters=3)[0] == 0
    for bad in ((-1.0, 0.5, 3), (math.nan, 0.5, 3), (0.01, 0.5, 0), (0.01, 0.5, 17)):
        rc, _ = _raw(pcreg, m, src, T0[:1], "grid", pcreg.icp_extrap(), stop=pcreg.icp_stop(*bad), iters=3)
        assert rc == -1, bad
    from pcreg_b200 import _lib as L
    o = pcreg.icp_opts(pcreg.ICP_KNN, 3, nn=pcreg.NN_GRID)
    a = np.asfortranarray(src.astype(np.float64))
    T = np.empty((1, 16))
    T0a = np.eye(4).reshape(1, 16).copy()
    for soff, hoff in (([1, 600], [0, 1]), ([0, 600], [1, 1]), ([0, 300, 200], [0, 1, 1]), ([0, 0], [0, 1])):
        so, ho = np.array(soff, dtype=np.int64), np.array(hoff, dtype=np.int64)
        rc = L.lib().pcreg_icp_batch_extrap(m.handle, a.ctypes.data_as(C.c_void_p), 1, 600, so.ctypes.data_as(L.c_i64p), None,
                                            ho.ctypes.data_as(L.c_i64p), len(soff) - 1, T0a.ctypes.data_as(L.c_f64p), C.byref(o), None,
                                            C.byref(pcreg.icp_extrap()), T.ctypes.data_as(L.c_f64p), *([None] * 9))
        assert rc == -1, (soff, hoff)
    for metric in ("point_to_plane", "plane_to_plane"):
        with pytest.raises(ValueError):
            pcreg.icp_batch(m, src, T0[:1], iters=3, metric=metric, extrapolate=True)
        with pytest.raises(ValueError):
            pcreg.icp_batch_windows(m, [src], [T0[:1]], iters=3, metric=metric, extrapolate=True)
