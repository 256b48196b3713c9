"""Every exact nearest-neighbour path on adversarial inputs (tests/nn_adversarial.py: near-ties inside the FP32 error bands,
exact FP64 ties between FP32-inexact points, far and huge queries, equidistant crowds) against the FP64 oracle.
Bar: index and squared distance bit for bit, ties -> smallest original index (as tests/test_gpu_nn.py)."""
import numpy as np
import pytest

import nn_adversarial as A
import oracle
from icp_plane_reference import knn_exact, normals_reference
from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

GEN = list(A.GENERATORS)
VIDS = [A.variant_id(v) for v in A.VARIANTS]


def _same(tag, gi, gd, oi, od):
    bad = np.nonzero(gi != oi)[0]
    assert bad.size == 0, "%s: %d of %d index mismatches, first at %s: got %s want %s (d2 %s vs %s)" % (
        tag, bad.size, oi.size, bad[:5], gi[bad[:5]], oi[bad[:5]], gd[bad[:5]], od[bad[:5]])
    assert np.array_equal(gd, od), "%s: d2 not bit-exact at %s" % (tag, np.nonzero(gd != od)[0][:5])


def _profiled(pcreg, m, q, kind):
    pcreg.set_profiling(True)
    try:
        out = m.nn_search(q, kind)
        return out, pcreg.last_profile()
    finally:
        pcreg.set_profiling(False)


# ---- 1. the NN entry point, every path -----------------------------------------------------------------------------------
@pytest.mark.parametrize("v", A.VARIANTS, ids=VIDS)
@pytest.mark.parametrize("name", GEN)
def test_nn_search_every_path(pcreg, monkeypatch, name, v):
    """Brute force (model split across blockIdx.y), the grid walk (voxel_map=-1), the voxel map as built, the voxel map with
    lists capped at 8 entries (dropped lists: walked), and a band-limited voxel map (voxels beyond the band: walked)."""
    model, q = A.generate(name, v)
    oi, od = oracle.nn_brute(model, q)
    m = pcreg.Model(model, grid=False)
    _same("brute", *m.nn_search(q, pcreg.NN_BRUTE), oi, od)
    m.destroy()
    m = pcreg.Model(model, grid=True, voxel_map=-1)
    _same("brute on a grid model", *m.nn_search(q, pcreg.NN_BRUTE), oi, od)
    _same("grid walk", *m.nn_search(q, pcreg.NN_GRID), oi, od)
    m.destroy()
    sp = A.spacing(np.asarray(model, dtype=np.float64))
    for tag, env in (("voxel map", {}), ("voxel map, lists capped", {"PCREG_VOX_CAP": "8"}),
                     ("voxel map, band-limited", {"PCREG_VOX_BAND": repr(2.0 * sp)})):
        for k, val in env.items():
            monkeypatch.setenv(k, val)
        m = pcreg.Model(model, grid=True, voxel_map=1)
        for k in env:
            monkeypatch.delenv(k)
        info = m.voxel_info()
        assert info["voxels"] > 0, tag
        (gi, gd), prof = _profiled(pcreg, m, q, pcreg.NN_GRID)
        _same(tag, gi, gd, oi, od)
        assert prof["voxel_map"] == 1.0, tag
        # the intended branch ran: queries outside the padded box (far, huge) are walked, and so are nearly all crowd queries --
        # the voxels around the sphere's centre and the cylinder's axis would list hundreds of equidistant points, so their
        # lists are dropped (at the finest level or above it: voxel_info counts only the former) or lie beyond the band
        if name in ("far", "huge"):
            assert prof["walked_queries"] > 0, (tag, prof)
        if name == "crowd":
            assert prof["walked_queries"] >= 0.5 * q.shape[0], (tag, prof)
        if "PCREG_VOX_BAND" in env and name != "ties":
            assert info["outside_band"] > 0, info
        m.destroy()


@pytest.mark.parametrize("name", ["bisector", "ties", "huge"])
def test_nn_brute_many_queries_wide_kernel(pcreg, name):
    """> 148 * 256 * 8 queries on a small model: the 8-queries-per-thread kernel without a model split"""
    v = (np.float64, 1e3, 1.0)
    model, q = A.generate(name, v, **({"nq": 320_000} if name == "ties" else {"n_model": 4096, "nq": 320_000}))
    oi, od = oracle.nn_brute(model, q)
    m = pcreg.Model(model, grid=False)
    _same("brute, wide", *m.nn_search(q, pcreg.NN_BRUTE), oi, od)
    m.destroy()


# ---- 2. the correspondences of every ICP pass ---------------------------------------------------------------------------
ICP_VARIANTS = [(np.float32, 0.0, 1.0), (np.float64, 1e3, 1.0)]
# path -> (voxel_map, nn, mode, environment)
ICP_PATHS = {
    "brute": (-1, "brute", "knn", {}),
    "lists-knn": (-1, "grid", "knn", {}),
    "lists-weighted": (-1, "grid", "weighted", {}),
    "lists-rows-lane": (-1, "grid", "knn", {"PCREG_ROWSCAN": "lane", "PCREG_WALK": "lane"}),
    "lists-rows-warp": (-1, "grid", "knn", {"PCREG_ROWSCAN": "warp", "PCREG_WALK": "warp"}),
    "vox-per-pass": (1, "grid", "knn", {"PCREG_FUSED": "0"}),
    "vox-fused": (1, "grid", "knn", {"PCREG_FUSED": "1"}),
    "vox-fused-windows": (1, "grid", "knn", {"PCREG_FUSED": "1"}),
}
ITERS = (0, 1, 2, 5, 12)


def _icp_problem(name, v, H=8):
    """anchors: model points mapped by the inverse of the true pose (weight 1); probes: the generated queries mapped the same
    way (weight 0, so they never move the pose).  T0 is the truth for most hypotheses, a few are turned by 1e-9 .. 1e-7 rad."""
    model, q = A.generate(name, v, nq=600, **({} if name == "ties" else {"n_model": 15_000}))
    m64 = np.asarray(model, dtype=np.float64)
    g = synth.rng(17)
    T_true = synth.make_T(synth.rot_xyz(g.uniform(0, 2 * np.pi, 3)), np.array([13.0, 25.0, -17.0]) * np.abs(m64).max() / 50.0)
    Ti = oracle.invertTF(T_true)
    anchors = m64[g.choice(m64.shape[0], 300, replace=False)]
    src = np.vstack([oracle.quickTF(anchors, Ti), oracle.quickTF(q, Ti)])
    w = np.concatenate([np.ones(anchors.shape[0]), np.zeros(q.shape[0])])
    c = m64.mean(0)
    T0 = [T_true] * (H - 3) + [synth.perturb_pose(T_true, c, synth.rot_axis_angle(g.normal(size=3), a), np.zeros(3))
                               for a in (1e-9, 1e-8, 1e-7)]
    return model, q, src, w, np.stack(T0)


def _gate(model, q, src, T, share0):
    """near-ties survive at the returned poses: the share of probes whose oracle gap is below 1e-6 stays at least half of
    that of the generated queries"""
    nprobe = q.shape[0]
    for h in range(T.shape[0] - 3):                       # the hypotheses started at the truth
        qq = oracle.quickTF(src[-nprobe:], T[h])
        share = np.mean(A.gaps(model, qq) < 1e-6)
        assert share >= 0.5 * share0, (h, share, share0)


@pytest.mark.parametrize("path", list(ICP_PATHS))
@pytest.mark.parametrize("v", ICP_VARIANTS, ids=[A.variant_id(v) for v in ICP_VARIANTS])
@pytest.mark.parametrize("name", GEN)
def test_icp_pass_correspondences(pcreg, monkeypatch, name, v, path):
    """idx of the final pass of every ICP call equals the oracle's NN at the returned poses, for 0 .. 12 iterations"""
    vm, nn, mode, env = ICP_PATHS[path]
    model, q, src, w, T0 = _icp_problem(name, v)
    share0 = np.mean(A.gaps(model, q) < 1e-6)
    m = pcreg.Model(model, grid=True, voxel_map=vm)
    for k, val in env.items():
        monkeypatch.setenv(k, val)
    gmode = pcreg.ICP_KNN if mode == "knn" else pcreg.ICP_WEIGHTED
    kind = pcreg.NN_BRUTE if nn == "brute" else pcreg.NN_GRID
    for iters in ITERS:
        pcreg.set_profiling(iters == ITERS[-1])
        if path == "vox-fused-windows":
            h = T0.shape[0] // 2
            na = src.shape[0] - q.shape[0]
            np_half = q.shape[0] // 2
            srcs = [src[: na + np_half], np.vstack([src[:na], src[na + np_half:]])]
            ws = [w[: na + np_half], np.concatenate([w[:na], w[na + np_half:]])]
            outs = pcreg.icp_batch_windows(m, srcs, [T0[:h], T0[h:]], mode=gmode, iters=iters, nn=kind, w_src_list=ws, return_idx=True)
            runs = list(zip(srcs, outs))
        else:
            res = pcreg.icp_batch(m, src, T0, mode=gmode, iters=iters, nn=kind, w_src=w, return_idx=True)
            runs = [(src, res)]
        if iters == ITERS[-1]:
            prof = pcreg.last_profile()
            pcreg.set_profiling(False)
            assert prof["fused"] == (1.0 if "fused" in path else 0.0), prof
            assert prof["voxel_map"] == (1.0 if path.startswith("vox") else 0.0), prof
        for s, res in runs:
            for hh in range(res["T"].shape[0]):
                oi, _ = oracle.nn_brute(model, oracle.quickTF(s, res["T"][hh]))
                bad = np.nonzero(res["idx"][hh] != oi)[0]
                assert bad.size == 0, "%s iters %d hyp %d: %d correspondence mismatches, first at %s" % (path, iters, hh, bad.size, bad[:5])
    m.destroy()
    if path == "brute":                                   # once per input: the near-ties are still there at the returned poses
        _gate(model, q, src, res["T"], share0)


# ---- 3. lazy trimming next to its bound -----------------------------------------------------------------------------------
def _pca_normals(m64, k=12):
    from scipy.spatial import cKDTree
    _, nb = cKDTree(m64).query(m64, k)
    X = m64[nb] - m64[nb].mean(1, keepdims=True)
    _, V = np.linalg.eigh(np.einsum("nki,nkj->nij", X, X))
    return V[:, :, 0]


@pytest.mark.parametrize("mode", ["knn", "weighted", "plain"])
def test_lazy_trim_shell_just_outside(pcreg, mode):
    """A shell of source points sits just above the trim radius tau (offset tau (1 + eps) along the model normal, eps spread
    over 1e-9 .. 1e-2), the rest below it, plus gross outliers; the start pose is several spacings off, so the early passes
    move a lot and the bound of the skipping test is tight.  Grid ICP without a voxel map (candidate lists, lazy trimming)
    must equal brute-force ICP bit for bit, and it must have skipped searches."""
    model = synth.make_model(60_000, 505)
    m64 = np.asarray(model, dtype=np.float64)
    g = synth.rng(506)
    sp = A.spacing(m64)
    tau = 2.0 * sp
    nrm = _pca_normals(m64)
    n_in, n_shell, n_out = 1100, 250, 150
    pick = g.choice(m64.shape[0], n_in + n_shell + n_out, replace=False)
    sign = g.choice([-1.0, 1.0], pick.size)[:, None]
    rho = np.concatenate([g.uniform(0, tau, n_in), tau * (1 + 10.0 ** g.uniform(-9, -2, n_shell)), g.uniform(4, 8, n_out) * tau])
    pts = m64[pick] + sign * nrm[pick] * rho[:, None]
    T_gt = synth.make_T(synth.rot_xyz(g.uniform(0, 2 * np.pi, 3)), np.array([13.0, 25.0, -17.0]))
    src = oracle.quickTF(pts, oracle.invertTF(T_gt))
    c = pts.mean(0)
    T0 = np.stack([synth.perturb_pose(T_gt, c, synth.rot_axis_angle(g.normal(size=3), np.deg2rad(a)), t)
                   for a, t in ((0.0, np.zeros(3)), (2.0, np.array([3 * sp, -2 * sp, sp])), (4.0, np.array([-4 * sp, 0, 2 * sp])),
                                (1.0, np.array([0, 5 * sp, 0])), (0.5, np.array([2 * sp, 2 * sp, -2 * sp])), (3.0, np.zeros(3)))])
    kw = dict(knn=dict(mode=pcreg.ICP_KNN, k_frac=n_in / pick.size), weighted=dict(mode=pcreg.ICP_WEIGHTED, R_w=tau),
              plain=dict(mode=pcreg.ICP_PLAIN, thDist2=tau * tau))[mode]
    m = pcreg.Model(model, grid=True, voxel_map=-1)
    pcreg.set_profiling(True)
    a = pcreg.icp_batch(m, src, T0, iters=25, nn=pcreg.NN_GRID, return_idx=True, return_hist=True, **kw)
    prof = pcreg.last_profile()
    pcreg.set_profiling(False)
    b = pcreg.icp_batch(m, src, T0, iters=25, nn=pcreg.NN_BRUTE, return_idx=True, return_hist=True, **kw)
    for k in ("T", "rmse_hist", "idx", "n_used", "status"):
        assert np.array_equal(a[k], b[k], equal_nan=True) if a[k].dtype.kind == "f" else np.array_equal(a[k], b[k]), k
    assert prof["lazy_skipped_queries"] > 0, prof
    m.destroy()


# ---- 4. k-NN ties in compute_normals ---------------------------------------------------------------------------------------
def _corrugated_lattice(jitter, seed=3):
    """a sheet on a lattice of spacing 0.1 at offset 1e3 (not FP32 values), every other row lifted by 0.05, 10 % of the
    points duplicated: exact and near ties at the k-th neighbour whose choice moves the normal"""
    ax = 1e3 + 0.1 * np.arange(40)
    X, Y = np.meshgrid(ax, ax, indexing="ij")
    Z = 1e3 + 0.05 * (np.arange(40)[:, None] % 2) + 0.0 * Y
    pts = np.column_stack([X.ravel(), Y.ravel(), Z.ravel()])
    g = synth.rng(seed)
    pts = np.vstack([pts, pts[g.choice(pts.shape[0], pts.shape[0] // 10, replace=False)]])
    pts = pts + g.uniform(-jitter, jitter, pts.shape)
    return np.ascontiguousarray(pts[g.permutation(pts.shape[0])])


@pytest.mark.parametrize("jitter", [0.0, 1e-9])
@pytest.mark.parametrize("k", [3, 6, 20])
def test_compute_normals_knn_ties(pcreg, k, jitter):
    model = _corrugated_lattice(jitter)
    m = pcreg.Model(model, grid=True, voxel_map=-1)
    try:
        m.compute_normals(k)
        n = m.normals()
    finally:
        m.destroy()
    nr, w = normals_reference(model, k)
    # the bar of test_gpu_icp_plane._check_normals on every point whose normal is defined (smallest eigenvalue separated)
    # (and whose neighbourhood is not a line: k = 3 with a duplicate, or three points of one lattice row)
    sep = ((w[:, 1] - w[:, 0]) > 1e-6 * w[:, 1]) & (w[:, 1] > 1e-9 * w[:, 2])
    assert sep.sum() >= 50, sep.sum()
    assert np.allclose(np.linalg.norm(n, axis=1), 1.0, rtol=0, atol=1e-15)
    bad = np.nonzero(np.abs((n * nr).sum(axis=1))[sep] < 1 - 1e-9)[0]
    assert bad.size == 0, "%d of %d normals differ from the (d2, index) neighbourhood's" % (bad.size, sep.sum())
    # teeth: the opposite tie rule (largest index first among equal d2) gives other normals on many points
    x = np.asarray(model, dtype=np.float64)
    nb = knn_exact(x, k)
    rev = knn_exact(x[::-1], k)
    rev = (x.shape[0] - 1 - rev)[::-1]
    differ = np.any(np.sort(nb, 1) != np.sort(rev, 1), axis=1)
    if jitter == 0.0 and k > 3:
        assert differ.mean() > 0.05, differ.mean()
