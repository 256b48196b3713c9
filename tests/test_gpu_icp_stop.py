"""The ICP tolerance stop on the GPU (include/pcreg.h: pcreg_icp_stop, pcreg_icp_batch_stop{,_dev}).

The defining property: a hypothesis that stops after k updates returns exactly what pcreg_icp_batch with iters = k returns
for it (T, rmse, n_used, status, idx bit for bit; rmse_hist columns 0..k that call's, k..iters the final rmse), on the fused
kernel, the per-pass kernels and brute force; a stopped hypothesis does no further NN work; a disabled tolerance changes no
bit; decisions match the FP64 reference (tests/icp_stop_reference.py)."""
import ctypes as C
import math

import numpy as np
import pytest

from icp_stop_reference import icp_batch_stop
from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

ITERS = 20
TOL = (0.01, 0.5)
OUT_KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


@pytest.fixture(scope="module")
def prob():
    """12 poses up to 12 deg / 2 mm from the truth: some converge early (at several different updates), some never do."""
    model = synth.make_model(20_000, 100)
    src, T_gt, c = synth.make_source(model, 600, 0.3, 101)
    T0 = synth.pose_grid(T_gt, c, 3, (2, 2, 1), 12.0, 2.0, 102)
    return model, src, T0


@pytest.fixture()
def models(pcreg, prob):
    """Per test: the device-count test re-initialises the library, which invalidates model handles."""
    model = prob[0]
    ms = dict(vox=pcreg.Model(model, grid=True, voxel_map=1), novox=pcreg.Model(model, grid=True, voxel_map=-1))
    yield ms
    for m in ms.values():
        m.destroy()


# path -> (model, nn, environment)
PATHS = {
    "fused": ("vox", "grid", {"PCREG_FUSED": "1"}),
    "per-pass": ("vox", "grid", {"PCREG_FUSED": "0"}),
    "per-pass-lanes": ("vox", "grid", {"PCREG_FUSED": "0", "PCREG_LANES": "2", "PCREG_MAX_CHUNK_HYP": "2"}),
    "brute": ("vox", "brute", {}),
    "grid-novox": ("novox", "grid", {}),
}


def _setenv(monkeypatch, env):
    for k in ("PCREG_FUSED", "PCREG_LANES", "PCREG_MAX_CHUNK_HYP"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _run(P, m, src, T0, nn, iters=ITERS, tolerance=None, window=3, **kw):
    kw.setdefault("mode", P.ICP_KNN)
    return P.icp_batch(m, src, T0, iters=iters, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE, return_idx=True,
                       return_hist=True, tolerance=tolerance, window=window, **kw)


MODES = {
    "plain": lambda P, src: dict(mode=P.ICP_PLAIN, thDist2=9.0),
    "knn": lambda P, src: dict(mode=P.ICP_KNN, k_frac=0.85),
    "weighted": lambda P, src: dict(mode=P.ICP_WEIGHTED, R_w=3.5, w_src=synth.rng(77).uniform(0.5, 1.0, src.shape[0])),
}


@pytest.mark.parametrize("path", ["fused", "per-pass", "brute", "grid-novox"])
@pytest.mark.parametrize("mode", list(MODES))
def test_disabled_tolerance_is_bit_identical(pcreg, prob, models, monkeypatch, path, mode):
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    kw = MODES[mode](pcreg, src)
    ref = _run(pcreg, models[mk], src, T0, nn, iters=12, **kw)
    out = _run(pcreg, models[mk], src, T0, nn, iters=12, tolerance=(0.0, 0.0), **kw)
    for k in OUT_KEYS:
        assert _eq(out[k], ref[k]), (path, mode, k)
    assert out["best"] == ref["best"]
    assert not out["converged"].any()
    assert np.all(out["n_iter"][out["status"] == 0] == 12)


def _check_stop_at_k(P, m, src, T0, nn, out, iters=ITERS, **kw):
    """Group the hypotheses by n_iter and rerun each group with iters = n_iter: every output bit for bit."""
    for k in np.unique(out["n_iter"]):
        g = np.nonzero(out["n_iter"] == k)[0]
        ref = _run(P, m, src, T0[g], nn, iters=int(k), **kw)
        for key in ("T", "rmse", "n_used", "status", "idx"):
            assert _eq(out[key][g], ref[key]), (k, key)
        assert _eq(out["rmse_hist"][g, :k + 1], ref["rmse_hist"]), k
        assert _eq(out["rmse_hist"][g, k:], np.repeat(out["rmse"][g, None], iters + 1 - k, axis=1)), k


def _assert_not_vacuous(out, iters=ITERS):
    stopped = np.unique(out["n_iter"][out["converged"] == 1])
    assert len(stopped[stopped < iters]) >= 3, out["n_iter"]
    assert np.any((out["converged"] == 0) & (out["n_iter"] == iters)), out["n_iter"]


@pytest.mark.parametrize("path", list(PATHS))
def test_stop_at_k_equals_fixed_iteration_run(pcreg, prob, models, monkeypatch, path):
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    out = _run(pcreg, models[mk], src, T0, nn, tolerance=TOL)
    _assert_not_vacuous(out)
    _check_stop_at_k(pcreg, models[mk], src, T0, nn, out)


@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_stopped_hypotheses_do_no_further_work(pcreg, prob, models, monkeypatch, path):
    """Device-counted voxel-list entries read and queries walked of the stop run = the sum over the iters = k reruns."""
    _, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    pcreg.set_profiling(True)
    try:
        out = _run(pcreg, models[mk], src, T0, nn, tolerance=TOL)
        p = pcreg.last_profile()
        assert p["fused"] == (1.0 if path == "fused" else 0.0) and p["voxel_map"] == 1.0
        got = (p["list_entries_read"], p["walked_queries"])
        want = [0.0, 0.0]
        for k in np.unique(out["n_iter"]):
            g = np.nonzero(out["n_iter"] == k)[0]
            _run(pcreg, models[mk], src, T0[g], nn, iters=int(k))
            q = pcreg.last_profile()
            want[0] += q["list_entries_read"]
            want[1] += q["walked_queries"]
    finally:
        pcreg.set_profiling(False)
    _assert_not_vacuous(out)
    assert got == tuple(want) and got[0] > 0
    # the query / correspondence counts are those of the passes run: n_iter + 1, one more after a freeze
    run = src.shape[0] * float(np.sum(out["n_iter"] + 1 + out["status"]))
    assert p["nn_queries"] == run and p["correspondences"] == run, (p["nn_queries"], run)


@pytest.mark.parametrize("path", ["fused", "brute"])
def test_decisions_match_the_reference(pcreg, prob, models, monkeypatch, path):
    model, src, T0 = prob
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    ref = icp_batch_stop(model, src, T0, TOL, 3, mode=1, iters=ITERS, k_frac=0.85)
    # no decision of the reference is within rounding of its tolerance
    for r in ref["results"]:
        for mt, mr in r["stop_means"]:
            assert abs(mt - TOL[0]) >= 1e-6 * TOL[0] and abs(mr - TOL[1]) >= 1e-6 * TOL[1], (mt, mr)
    out = _run(pcreg, models[mk], src, T0, nn, tolerance=TOL)
    assert np.array_equal(out["n_iter"], ref["n_iter"]) and np.array_equal(out["converged"], ref["converged"])
    assert np.array_equal(out["status"], ref["status"]) and np.array_equal(out["n_used"], ref["n_used"])
    assert np.array_equal(out["idx"], ref["idx"])
    for h in range(T0.shape[0]):
        assert np.linalg.norm(out["T"][h][:3, :3] - ref["T"][h][:3, :3], "fro") <= 1e-6
        to = ref["T"][h][3, :3]
        assert np.linalg.norm(out["T"][h][3, :3] - to) <= 1e-6 * max(np.linalg.norm(to), 1e-12)
        assert abs(out["rmse"][h] - ref["rmse"][h]) <= 1e-7 * ref["rmse"][h]
    np.testing.assert_allclose(out["rmse_hist"], ref["rmse_hist"], rtol=1e-7)


@pytest.fixture()
def multi(pcreg, monkeypatch):
    monkeypatch.setenv("PCREG_ALLOW_DUP_DEVICES", "1")
    yield pcreg
    pcreg.init(0)


def test_results_do_not_depend_on_device_count(multi, prob):
    P = multi
    model, src, T0 = prob
    cases = [dict(nn="grid"), dict(nn="brute")]
    P.init(0)
    m = P.Model(model, grid=True)
    ref = [_run(P, m, src, T0, tolerance=TOL, **kw) for kw in cases]
    m.destroy()
    for devs in ([0, 0], [0, 0, 0]):
        P.init(devs)
        m = P.Model(model, grid=True)
        for kw, r in zip(cases, ref):
            a = _run(P, m, src, T0, tolerance=TOL, **kw)
            for k in OUT_KEYS + ("n_iter", "converged"):
                assert _eq(a[k], r[k]), (devs, kw, k)
            assert a["best"] == r["best"]
        m.destroy()


def test_degenerate_hypothesis_and_argument_errors(pcreg, prob, models):
    _, src, T0 = prob
    m = models["vox"]
    for nn in ("grid", "brute"):
        # fewer than 3 correspondences survive: frozen before the first update, exactly as without the tolerance
        ref = _run(pcreg, m, src, T0[:3], nn, iters=5, mode=pcreg.ICP_PLAIN, thDist2=1e-12)
        out = _run(pcreg, m, src, T0[:3], nn, iters=5, tolerance=TOL, mode=pcreg.ICP_PLAIN, thDist2=1e-12)
        assert np.all(out["status"] == 1) and not out["converged"].any() and np.all(out["n_iter"] == 0)
        for k in OUT_KEYS:
            assert _eq(out[k], ref[k]), (nn, k)
    from pcreg_b200 import _lib as L
    lib = L.lib()
    a = np.ascontiguousarray(src.T).ravel()
    T0a = np.ascontiguousarray(np.transpose(np.asarray(T0[:1]), (0, 2, 1))).reshape(1, 16)
    T = np.empty((1, 16))
    o = pcreg.icp_opts(pcreg.ICP_KNN, 5, nn=pcreg.NN_GRID)
    f64 = lambda x: x.ctypes.data_as(L.c_f64p)  # noqa: E731
    for bad in ((-1.0, 0.5, 3), (math.nan, 0.5, 3), (0.01, math.nan, 3), (0.01, -0.5, 3), (0.01, 0.5, 0), (0.01, 0.5, 17)):
        s = pcreg.icp_stop(*bad)
        rc = lib.pcreg_icp_batch_stop(m.handle, a.ctypes.data_as(C.c_void_p), 1, src.shape[0], src.shape[0], None, f64(T0a), 1,
                                      C.byref(o), C.byref(s), f64(T), None, None, None, None, None, None, None, None)
        assert rc == -1, bad                                  # PCREG_ERR_ARG
        with pytest.raises(pcreg.PcregError):
            pcreg.icp_batch(m, src, T0[:1], iters=5, tolerance=bad[:2], window=bad[2])
    s = pcreg.icp_stop(0.01, 0.5, 16)
    assert lib.pcreg_icp_batch_stop(m.handle, a.ctypes.data_as(C.c_void_p), 1, src.shape[0], src.shape[0], None, f64(T0a), 1,
                                    C.byref(o), C.byref(s), f64(T), None, None, None, None, None, None, None, None) == 0


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
    out = torch_ops.IcpDeviceBuffers(H, ns, ITERS, dev, want_idx=True, want_hist=True, want_n_iter=True)
    o = pcreg.icp_opts(pcreg.ICP_KNN, ITERS, 0.85, nn=pcreg.NN_GRID)
    torch_ops.icp_batch_device(m, src_cm, None, T0_abi, o, out, stop=pcreg.icp_stop(*TOL, 3))
    torch.cuda.synchronize()
    assert np.array_equal(torch_ops.T_from_abi_t(out.T).cpu().numpy(), host["T"])
    for k, v in (("rmse", out.rmse), ("n_used", out.n_used), ("status", out.status), ("idx", out.idx), ("rmse_hist", out.hist),
                 ("n_iter", out.n_iter), ("converged", out.converged)):
        assert _eq(v.cpu().numpy(), host[k]), k
    assert int(out.best.item()) == host["best"]


def _freeze_problem():
    """40 model points (plus a far cluster that is never the nearest neighbour) and 12 noisy copies of some of them, fitted
    on k_frac = 0.3 of the correspondences within sqrt(thDist2): after an update or more most poses keep fewer than 3 and
    freeze.  A pose 1000 units away (every query outside the voxel map's box, answered by the pyramid walk) freezes before
    its first update."""
    g = np.random.default_rng(1)
    for _ in range(23):                                      # the 23rd draw of this generator is the case
        m = g.normal(0, 5, (40, 3))
        src = m[:12] + g.normal(0, 0.8, (12, 3))
        thd = float(g.uniform(0.3, 2.0))
    model = np.vstack([m, synth.make_model(3000, 5) + 300.0])
    T0 = [np.eye(4)]
    for k in range(4):
        T0.append(synth.perturb_pose(np.eye(4), src.mean(axis=0), synth.rot_axis_angle([1.0, k, 2.0 - k], np.deg2rad(1.5)),
                                     np.array([0.1 * k, -0.2, 0.1])))
    far = np.eye(4)
    far[3, :3] = 1000.0
    T0.append(far)
    return model, src, np.stack(T0), thd


@pytest.mark.parametrize("path", ["fused", "per-pass"])
def test_early_stops_and_freezes_with_even_iters(pcreg, monkeypatch, path):
    """Hypotheses that stop or freeze after 0, 1 or a few updates, with an even pass count (the final pass reads the
    correspondence buffer of the odd passes as its warm start on the per-pass path): a freeze after p updates (n_iter = p,
    hist columns p+1.. the final rmse) and a stop at update 1 (window = 1) return the bits of the runs they stand for, and
    every correspondence is a valid model index."""
    model, src, T0, thd = _freeze_problem()
    _setenv(monkeypatch, PATHS[path][2])
    iters = 8
    m = pcreg.Model(model, grid=True, voxel_map=1)
    try:
        kw = dict(mode=pcreg.ICP_KNN, k_frac=0.3, thDist2=thd)
        plain = _run(pcreg, m, src, T0, "grid", iters=iters, **kw)
        # tolerance off: only the freezes end a hypothesis early; every output as without the tolerance
        out = _run(pcreg, m, src, T0, "grid", iters=iters, tolerance=(0.0, 0.0), **kw)
        assert not out["converged"].any() and np.array_equal(out["status"], plain["status"])
        for k in OUT_KEYS:
            assert _eq(out[k], plain[k]), k
        assert out["idx"].min() >= 0 and out["idx"].max() < model.shape[0]
        assert out["status"][-1] == 1 and out["n_iter"][-1] == 0
        assert np.any((out["status"] == 1) & (out["n_iter"] >= 1)), out["n_iter"]
        # n_iter = p of a freeze: an iters = p run applies the same p updates, an iters = p + 1 run freezes
        for h in np.nonzero(out["status"] == 1)[0]:
            p = int(out["n_iter"][h])
            a = _run(pcreg, m, src, T0[h:h + 1], "grid", iters=p, **kw)
            b = _run(pcreg, m, src, T0[h:h + 1], "grid", iters=p + 1, **kw)
            assert a["status"][0] == 0 and b["status"][0] == 1, (h, p)
            assert _eq(out["T"][h], a["T"][0]) and _eq(out["rmse_hist"][h, :p + 1], a["rmse_hist"][0]), (h, p)
            assert _eq(out["rmse_hist"][h, p + 1:], np.full(iters - p, out["rmse"][h])), (h, p)
        # window 1, both criteria off: every hypothesis that does not freeze first stops at update 1
        out = _run(pcreg, m, src, T0, "grid", iters=iters, tolerance=(math.inf, math.inf), window=1, **kw)
        live = out["status"] == 0
        assert live.sum() >= 3 and np.all(out["n_iter"][live] == 1) and np.all(out["converged"][live] == 1)
        assert out["idx"].min() >= 0 and out["idx"].max() < model.shape[0]
        g = np.nonzero(live)[0]
        one = _run(pcreg, m, src, T0[g], "grid", iters=1, **kw)
        for k in ("T", "rmse", "n_used", "status", "idx"):
            assert _eq(out[k][g], one[k]), k
        assert _eq(out["rmse_hist"][g, :2], one["rmse_hist"])
        assert _eq(out["rmse_hist"][g, 1:], np.repeat(out["rmse"][g, None], iters, axis=1))
        d = np.nonzero(~live)[0]
        for k in OUT_KEYS:                                   # those that freeze before update 1: as without the tolerance
            assert _eq(out[k][d], plain[k][d]), k
        assert np.all(out["n_iter"][d] == 0)
    finally:
        m.destroy()
