"""Fused ICP kernel over batches of many waves of blocks and over windows of very different sizes in one launch.

The fused kernel runs one hypothesis per block, so a batch larger than the blocks the device holds at once runs in waves; a
windowed launch sizes its shared memory for the largest window and indexes each window's rows from its own first row.  Whatever
wave or window a hypothesis lands in, its results must be the per-pass path's or its own call's, bit for bit."""
import numpy as np
import pytest

from pcreg_b200 import synth

pytestmark = pytest.mark.gpu

ITERS = 8
KEYS = ("T", "rmse", "n_used", "status", "idx", "rmse_hist")


def _eq(a, b):
    return np.array_equal(a, b, equal_nan=True) if np.asarray(a).dtype.kind == "f" else np.array_equal(a, b)


@pytest.fixture(scope="module")
def model_pts():
    return synth.make_model(20_000, 100)


@pytest.fixture()
def vox(pcreg, model_pts):
    m = pcreg.Model(model_pts, grid=True, voxel_map=1)
    yield m
    m.destroy()


def _setenv(monkeypatch, fused):
    for k in ("PCREG_LANES", "PCREG_MAX_CHUNK_HYP"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("PCREG_FUSED", fused)


def _run(P, fn, *args, **kw):
    P.set_profiling(True)
    try:
        r = fn(*args, **kw)
        fused = P.last_profile()["fused"]
    finally:
        P.set_profiling(False)
    return r, fused


MODES = {
    "knn": lambda P: dict(mode=P.ICP_KNN, k_frac=0.85),
    "plain": lambda P: dict(mode=P.ICP_PLAIN, thDist2=9.0),
}


@pytest.mark.parametrize("mode", list(MODES))
def test_many_waves_of_slots_equal_the_per_pass_path(pcreg, model_pts, vox, monkeypatch, mode):
    """1536 hypotheses: more than 5 waves of the 296 blocks a B200 holds at once."""
    src, T_gt, c = synth.make_source(model_pts, 1000, 0.3, 401)
    T0 = synth.pose_grid(T_gt, c, 96, (2, 2, 4), 8.0, 1.0, 402).reshape(-1, 4, 4)
    assert T0.shape[0] == 1536
    kw = dict(MODES[mode](pcreg), iters=ITERS, nn=pcreg.NN_GRID, return_idx=True, return_hist=True)
    out = {}
    for fused in ("1", "0"):
        _setenv(monkeypatch, fused)
        out[fused], ran = _run(pcreg, pcreg.icp_batch, vox, src, T0, **kw)
        assert ran == float(fused)
    for k in KEYS:
        assert _eq(out["1"][k], out["0"][k]), k
    assert out["1"]["best"] == out["0"]["best"]


def test_windows_of_very_different_sizes_in_one_launch(pcreg, model_pts, vox, monkeypatch):
    """6000-, 70- and 1500-point windows in one fused launch, 400 hypotheses each, against one call per window."""
    srcs, T0s = [], []
    for ns, seed in ((6000, 411), (70, 412), (1500, 413)):
        src, T_gt, c = synth.make_source(model_pts, ns, 0.3, seed)
        srcs.append(src)
        T0s.append(synth.pose_grid(T_gt, c, 100, (2, 2, 1), 8.0, 1.0, seed + 50).reshape(-1, 4, 4))
    _setenv(monkeypatch, "1")
    kw = dict(mode=pcreg.ICP_KNN, k_frac=0.85, iters=ITERS, nn=pcreg.NN_GRID, return_idx=True, return_hist=True)
    got, ran = _run(pcreg, pcreg.icp_batch_windows, vox, srcs, T0s, **kw)
    assert ran == 1.0
    for w, (s, T0, g) in enumerate(zip(srcs, T0s, got)):
        assert T0.shape[0] == 400
        ref = pcreg.icp_batch(vox, s, T0, **kw)
        for k in KEYS:
            assert _eq(g[k], ref[k]), (w, k)
        assert g["best"] == ref["best"], w
