"""The batched ICP on rank-deficient correspondences on the GPU (the rank rule of pcreg_icp_opts.reflection_fix, include/pcreg.h).

Problems from tests/icp_degenerate.py: a slab with an exactly planar face (axis-aligned and tilted, at offsets 0 and 1e3) and a
source patch on it (H of rank 2 at every update), a curved patch mirrored in its tangent plane (the data prefer a reflection),
a collinear source on a straight ridge, coincident source points, and three collinear positive weights (rank <= 1).  Against the
FP64 oracle with the same rule:
  - planar: det = +1 on every path in both modes, T / rmse / idx / n_used / status / best at the bars of test_gpu_icp.py;
  - mirrored: det = -1 with reflection_fix = 0 (R = V*U' reproduced), +1 with 1, same bars;
  - rank <= 1: R is not unique, so the transformed (weighted) source matches the oracle's, so do its idx, and every pose is proper;
and every path (fused, per-pass, two lanes, brute force, map-less grid) gives the same bits; the windows entry (fused launch and
loop, with the tolerance stop and with extrapolation, host and device entries) gives each window's own bits; an extrapolating call
on the mirrored patch never steps off an improper Kabsch pose and equals tests/icp_extrap_reference.py."""
import numpy as np
import pytest

import icp_degenerate as D
import oracle
from icp_extrap_reference import icp_single_extrap
from oracle.nn import KDTreeNN
from oracle.primitives import quickTF

pytestmark = pytest.mark.gpu

ITERS = 12
TOL = (0.01, 0.5)
OUT_KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")

PROBLEMS = {
    "plane-axis-0": lambda: D.planar_problem(11, False, 0.0),
    "plane-axis-1e3": lambda: D.planar_problem(11, False, 1e3),
    "plane-tilted-0": lambda: D.planar_problem(12, True, 0.0),
    "plane-tilted-1e3": lambda: D.planar_problem(12, True, 1e3),
    "mirrored": lambda: D.mirrored_problem(5),
    "edge": lambda: D.edge_problem(13),
    "coincident": lambda: D.coincident_problem(14),
    "three-weighted": lambda: D.three_weighted_problem(20),
}
RANK_LE1 = ("edge", "coincident", "three-weighted")

PATHS = {
    "fused": ("vox", "grid", {"PCREG_FUSED": "1"}),
    "per-pass": ("vox", "grid", {"PCREG_FUSED": "0"}),
    "per-pass-lanes": ("vox", "grid", {"PCREG_FUSED": "0", "PCREG_LANES": "2", "PCREG_MAX_CHUNK_HYP": "2"}),
    "brute": ("vox", "brute", {}),
    "grid-novox": ("novox", "grid", {}),
}


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


def _setenv(monkeypatch, env):
    for k in ("PCREG_FUSED", "PCREG_LANES", "PCREG_MAX_CHUNK_HYP"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


_PROBS = {}


def _prob(name):
    """(model, src, T0, w_src or None), built once per session."""
    if name not in _PROBS:
        p = PROBLEMS[name]()
        _PROBS[name] = p if len(p) == 4 else p + (None,)
    return _PROBS[name]


@pytest.fixture(scope="module")
def model_cache(pcreg):
    made = {}
    yield made
    for ms in made.values():
        for m in ms.values():
            m.destroy()


def _models(pcreg, cache, name):
    if name not in cache:
        model = _prob(name)[0]
        cache[name] = dict(vox=pcreg.Model(model, grid=True, voxel_map=1), novox=pcreg.Model(model, grid=True, voxel_map=-1))
    return cache[name]


def _mode_kw(P, name, mode):
    w = _prob(name)[3]
    if mode == "plain":
        return dict(mode=P.ICP_PLAIN, thDist2=25.0)
    if mode == "knn":
        return dict(mode=P.ICP_KNN, k_frac=0.85)
    ns = _prob(name)[1].shape[0]
    return dict(mode=P.ICP_WEIGHTED, R_w=3.5, w_src=w if w is not None else D.rng(77).uniform(0.5, 1.0, ns))


CASES = [(p, m) for p in PROBLEMS for m in ("plain", "knn", "weighted") if p != "three-weighted" or m == "weighted"]


def _run(P, m, src, T0, nn, refl, iters=ITERS, **kw):
    return P.icp_batch(m, src, T0, iters=iters, nn=P.NN_GRID if nn == "grid" else P.NN_BRUTE, return_idx=True, return_hist=True,
                       reflection_fix=refl, **kw)


def _oracle(name, kw, refl):
    model, src, T0, _ = _prob(name)
    okw = {k: v for k, v in kw.items() if k != "mode"}
    return oracle.icp_batch(model, src, T0, mode=kw["mode"], iters=ITERS, reflection_fix=refl, **okw)


def _proper_orthogonal(T):
    R = T[:, :3, :3]
    assert np.all(np.linalg.det(R) > 0)
    assert np.max(np.abs(np.einsum("hji,hjk->hik", R, R) - np.eye(3))) < 1e-9


def _check_against_oracle(name, kw, refl, out, ref):
    """Planar / mirrored: poses at test_gpu_icp.py's tolerances with the stated handedness, idx, n_used, status and best equal, rmse
    to 1e-7 relative.  Rank <= 1: the transformed (weighted) source to 1e-9 x extent, idx of the weighted points exact (a point of
    weight zero moves with the rotation about the line, which is not unique), n_used and status equal, and the winner's rmse is the
    oracle's smallest (the hypotheses of the coincident problem all converge to the same rmse, so the index is a tie)."""
    _, src, _, _ = _prob(name)
    assert np.array_equal(out["n_used"], ref["n_used"]) and np.array_equal(out["status"], ref["status"])
    if name in RANK_LE1:
        k = kw["w_src"] > 0 if name == "three-weighted" else np.ones(src.shape[0], dtype=bool)
        assert np.array_equal(out["idx"][:, k], ref["idx"][:, k])
        ext = max(float(np.ptp(src[k], axis=0).max()), 1.0)
        assert abs(ref["rmse"][out["best"]] - ref["rmse"][ref["best"]]) <= 1e-7 * ref["rmse"][ref["best"]] + 1e-9 * ext
        for h in range(out["T"].shape[0]):
            err = np.max(np.linalg.norm(quickTF(src[k], out["T"][h]) - quickTF(src[k], ref["T"][h]), axis=1))
            assert err <= 1e-9 * ext, (h, err)
        _proper_orthogonal(out["T"])
        assert np.allclose(out["rmse"], ref["rmse"], rtol=1e-7, atol=1e-9 * ext)
        return
    assert np.array_equal(out["idx"], ref["idx"]) and out["best"] == ref["best"]
    sign = -1.0 if (name == "mirrored" and not refl) else 1.0
    assert np.all(np.sign(np.linalg.det(out["T"][:, :3, :3])) == sign)
    assert np.all(np.sign(np.linalg.det(ref["T"][:, :3, :3])) == sign)
    for h in range(out["T"].shape[0]):
        assert np.linalg.norm(out["T"][h, :3, :3] - ref["T"][h, :3, :3]) < 1e-6, h
        tn = max(1.0, np.linalg.norm(ref["T"][h, 3, :3]))
        assert np.linalg.norm(out["T"][h, 3, :3] - ref["T"][h, 3, :3]) < 1e-6 * tn, h
    assert np.allclose(out["rmse"], ref["rmse"], rtol=1e-7, atol=0)


@pytest.mark.parametrize("refl", [False, True], ids=["refl0", "refl1"])
@pytest.mark.parametrize("name,mode", CASES)
def test_every_path_matches_the_oracle(pcreg, model_cache, monkeypatch, name, mode, refl):
    model, src, T0, _ = _prob(name)
    ms = _models(pcreg, model_cache, name)
    kw = _mode_kw(pcreg, name, mode)
    outs = {}
    for path, (mk, nn, env) in PATHS.items():
        _setenv(monkeypatch, env)
        outs[path] = _run(pcreg, ms[mk], src, T0, nn, refl, **kw)
    ref = outs["fused"]
    for path, out in outs.items():
        for k in OUT_KEYS:
            assert _eq(out[k], ref[k]), (path, k)
        assert out["best"] == ref["best"], path
    _check_against_oracle(name, kw, refl, ref, _oracle(name, kw, refl))


@pytest.mark.parametrize("refl", [False, True], ids=["refl0", "refl1"])
@pytest.mark.parametrize("fused", ["1", "0"], ids=["fused-launch", "loop"])
@pytest.mark.parametrize("name", ["plane-tilted-1e3", "mirrored", "edge", "three-weighted"])
def test_windows_entry_with_stop_and_extrapolation(pcreg, model_cache, monkeypatch, name, fused, refl):
    """Two windows (a crop of the source and the whole of it) in one call, with the tolerance stop and with extrapolation (and
    both): each window equals its own icp_batch call bit for bit, and every pose has the problem's handedness."""
    _, src, T0, _ = _prob(name)
    m = _models(pcreg, model_cache, name)["vox"]
    _setenv(monkeypatch, {"PCREG_FUSED": fused})
    mode = "weighted" if name == "three-weighted" else "knn"
    kw = _mode_kw(pcreg, name, mode)
    w = kw.pop("w_src", None)
    half = src.shape[0] // 2
    srcs, T0s = [src[:half] if w is None else src, src], [T0[:2], T0]
    ws = None if w is None else [w, w]
    for extra in (dict(tolerance=TOL), dict(extrapolate=True), dict(tolerance=TOL, extrapolate=True)):
        pcreg.set_profiling(2)
        try:
            outs = pcreg.icp_batch_windows(m, srcs, T0s, iters=ITERS, nn=pcreg.NN_GRID, return_idx=True, return_hist=True,
                                           reflection_fix=refl, w_src_list=ws, **kw, **extra)
            assert pcreg.last_profile()["fused"] == (1.0 if fused == "1" else 0.0)
        finally:
            pcreg.set_profiling(False)
        for s, t, wk, o in zip(srcs, T0s, ws or [None, None], outs):
            one = _run(pcreg, m, s, t, "grid", refl, w_src=wk, **kw, **extra)
            for k in OUT_KEYS + tuple(k for k in ("n_iter", "converged", "n_extrap") if k in one):
                assert _eq(o[k], one[k]), (extra, k)
            assert o["best"] == one["best"]
            dets = np.linalg.det(o["T"][:, :3, :3])
            if name == "mirrored" and not refl:
                assert np.all(dets < 0), extra
            else:
                assert np.all(dets > 0), extra


@pytest.mark.parametrize("path", list(PATHS))
def test_extrapolation_keeps_the_handedness_of_the_kabsch_pose(pcreg, model_cache, monkeypatch, path):
    """Mirrored patch, reflection_fix = 0: every Kabsch pose is improper, so no update extrapolates, every returned pose is the
    Kabsch pose (the bits of the call without extrapolation) with det -1, and the extrapolation reference agrees."""
    model, src, T0, _ = _prob("mirrored")
    ms = _models(pcreg, model_cache, "mirrored")
    mk, nn, env = PATHS[path]
    _setenv(monkeypatch, env)
    kw = _mode_kw(pcreg, "mirrored", "knn")
    for tol in (None, TOL):
        out = _run(pcreg, ms[mk], src, T0, nn, False, tolerance=tol, extrapolate=True, **kw)
        plain = _run(pcreg, ms[mk], src, T0, nn, False, tolerance=tol, **kw)
        assert np.all(out["n_extrap"] == 0)
        for k in OUT_KEYS + (("n_iter", "converged") if tol else ()):
            assert _eq(out[k], plain[k]), (tol, k)
        assert np.all(np.linalg.det(out["T"][:, :3, :3]) < 0)
        tree = KDTreeNN(np.asarray(model, dtype=np.float64))
        for h in range(T0.shape[0]):
            ref = icp_single_extrap(model, src, T0[h], mode=kw["mode"], k_frac=kw["k_frac"], iters=ITERS, tolerance=tol, nn=tree)
            assert ref["n_extrap"] == 0 and all(t["skipped"] for t in ref["trace"])
            assert np.linalg.det(ref["T"][:3, :3]) < 0
            assert np.linalg.norm(out["T"][h, :3, :3] - ref["T"][:3, :3]) < 1e-6, h
            assert np.linalg.norm(out["T"][h, 3, :3] - ref["T"][3, :3]) < 1e-6 * max(1.0, np.linalg.norm(ref["T"][3, :3])), h
            assert np.array_equal(out["idx"][h], ref["idx"]) and out["n_used"][h] == ref["n_used"], h
            assert np.isclose(out["rmse"][h], ref["rmse"], rtol=1e-7, atol=0), h
            if tol:
                assert out["n_iter"][h] == ref["n_iter"] and out["converged"][h] == ref["converged"], h


@pytest.mark.parametrize("refl", [False, True], ids=["refl0", "refl1"])
@pytest.mark.parametrize("name", ["plane-axis-1e3", "mirrored", "coincident"])
def test_device_entries_equal_the_host_entries(pcreg, model_cache, name, refl):
    """pcreg_icp_batch_windows_dev (stop) and pcreg_icp_batch_extrap_dev (extrapolation) through torch_ops: the host entries' bits."""
    import torch
    from pcreg_b200 import torch_ops
    _, src, T0, _ = _prob(name)
    m = _models(pcreg, model_cache, name)["vox"]
    dev = torch.device("cuda", 0)
    H, ns = T0.shape[0], src.shape[0]
    src_cm = torch_ops.src_to_abi_t(torch.as_tensor(src, device=dev))
    T0_abi = torch_ops.T_to_abi_t(torch.as_tensor(T0, device=dev)).reshape(-1, 16).contiguous()
    o = pcreg.icp_opts(pcreg.ICP_KNN, ITERS, k_frac=0.85, nn=pcreg.NN_GRID, reflection_fix=refl)
    for extrap in (None, pcreg.icp_extrap()):
        host = _run(pcreg, m, src, T0, "grid", refl, mode=pcreg.ICP_KNN, k_frac=0.85, tolerance=TOL, extrapolate=extrap is not None)
        out = torch_ops.IcpWindowsDeviceBuffers(H, H * ns, 1, ITERS, dev, want_idx=True, want_hist=True, want_n_iter=True,
                                                want_n_extrap=extrap is not None)
        torch_ops.icp_windows_device(m, src_cm, [0, ns], None, T0_abi, [0, H], o, out, stop=pcreg.icp_stop(*TOL, 3), extrap=extrap)
        torch.cuda.synchronize()
        assert np.array_equal(torch_ops.T_from_abi_t(out.T).cpu().numpy(), host["T"])
        assert np.array_equal(out.idx.cpu().numpy().reshape(H, ns), host["idx"])
        for key, v in (("rmse", out.rmse), ("n_used", out.n_used), ("status", out.status), ("rmse_hist", out.hist),
                       ("n_iter", out.n_iter), ("converged", out.converged)) + ((("n_extrap", out.n_extrap),) if extrap else ()):
            assert _eq(v.cpu().numpy(), host[key]), key
        assert int(out.best.cpu().numpy()[0]) == host["best"]
