"""The ICP tolerance stop without a GPU: the FP64 reference of the rule (tests/icp_stop_reference.py) against the fixed-iteration
oracle, the window mean and the strict compares at the boundary, and the C-ABI struct / defaults (include/pcreg.h:
pcreg_icp_stop)."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from icp_stop_reference import icp_single_stop, update_motion, window_means  # noqa: E402
from pcreg_b200 import synth  # noqa: E402


@pytest.fixture(scope="module")
def problem():
    model = synth.make_model(6000, 4242)
    src, T_gt, c = synth.make_source(model, 250, 0.3, 4243)
    T0 = synth.pose_grid(T_gt, c, 1, (2, 1, 1), 6.0, 1.0, 4244)
    return model, src, T0


def test_stop_at_k_equals_fixed_iteration_run(problem):
    """A hypothesis that stops after k updates returns what the plain loop with iters = k returns."""
    model, src, T0 = problem
    seen = set()
    for h in range(T0.shape[0]):
        for mode in (oracle.ICP_PLAIN, oracle.ICP_KNN):
            r = icp_single_stop(model, src, T0[h], (0.02, 0.2), 3, mode=mode, iters=25)
            k = r["n_iter"]
            assert r["converged"] == 1 and r["status"] == 0 and 3 <= k < 25
            seen.add(k)
            f = oracle.icp_single(model, src, T0[h], mode=mode, iters=k, return_hist=True)
            assert np.array_equal(r["T"], f["T"]) and r["rmse"] == f["rmse"] and r["n_used"] == f["n_used"]
            assert np.array_equal(r["idx"], f["idx"])
            assert np.array_equal(r["rmse_hist"][:k + 1], f["rmse_hist"])
            assert np.all(r["rmse_hist"][k:] == r["rmse"])
    assert seen


def test_disabled_tolerance_runs_every_iteration(problem):
    model, src, T0 = problem
    f = oracle.icp_single(model, src, T0[0], iters=12, return_hist=True)
    for tol in ((0.0, 0.0), (0.0, math.inf), (math.inf, 0.0)):
        r = icp_single_stop(model, src, T0[0], tol, 3, iters=12)
        assert r["n_iter"] == 12 and r["converged"] == 0
        assert np.array_equal(r["T"], f["T"]) and np.array_equal(r["rmse_hist"], f["rmse_hist"])
    # both criteria off: the first update the rule is evaluated at stops
    for window in (1, 3, 16):
        r = icp_single_stop(model, src, T0[0], (math.inf, math.inf), window, iters=20)
        assert r["n_iter"] == min(window, 20) and r["converged"] == (1 if window <= 20 else 0)


def test_window_mean_and_strict_boundary(problem):
    """The decision compares the mean of the last `window` motions, strictly: a tolerance equal to the mean does not stop,
    the next double above it does."""
    model, src, T0 = problem
    full = icp_single_stop(model, src, T0[0], (0.0, 0.0), 3, iters=10)
    assert len(full["stop_means"]) == 10 - 3 + 1
    # recompute the means from the motions of the fixed run
    Ts = [np.asarray(T0[0], dtype=np.float64)]
    for k in range(1, 11):
        Ts.append(oracle.icp_single(model, src, T0[0], iters=k)["T"])
    motion = [update_motion(Ts[u - 1], Ts[u]) for u in range(1, 11)]
    for u in range(3, 11):
        mt, mr = window_means(motion[:u], 3)
        assert (mt, mr) == full["stop_means"][u - 3]
        assert mt == (motion[u - 3][0] + motion[u - 2][0] + motion[u - 1][0]) / 3
    # an update whose mean is a strict running minimum: a tolerance equal to it must not stop there, the next double up must
    for c in (0, 1):
        means = [m[c] for m in full["stop_means"]]
        u = max(v for v in range(3, 11) if all(means[v - 3] < x for x in means[:v - 3]))
        assert u > 3, means
        tol = means[u - 3]
        off = [math.inf, math.inf]
        off[c] = tol
        r_eq = icp_single_stop(model, src, T0[0], tuple(off), 3, iters=10)
        off[c] = np.nextafter(tol, math.inf)
        r_up = icp_single_stop(model, src, T0[0], tuple(off), 3, iters=10)
        assert r_up["n_iter"] == u and r_up["converged"] == 1
        assert r_eq["converged"] == 0 or r_eq["n_iter"] > u


def test_rotation_angle_is_accurate_at_small_angles():
    """atan2 form: exact to rounding where acos((trace - 1) / 2) loses half the digits."""
    for deg in (1e-7, 1e-4, 0.3, 30.0, 179.0):
        a = np.radians(deg)
        R = synth.rot_axis_angle([0.3, -0.5, 0.8], a)
        Tc = np.eye(4)
        Tn = np.eye(4)
        Tn[:3, :3] = R
        Tn[3, :3] = [3.0, 4.0, 0.0]
        dt, dr = update_motion(Tc, Tn)
        assert dt == 5.0
        assert abs(dr - deg) <= 1e-9 * deg


def test_degenerate_hypothesis_counts_updates_before_freeze(problem):
    model, src, T0 = problem
    r = icp_single_stop(model, src, T0[0], (0.01, 0.5), 3, iters=5, thDist2=1e-12)
    assert r["status"] == 1 and r["converged"] == 0 and r["n_iter"] == 0
    assert np.array_equal(r["T"], np.asarray(T0[0]))


def test_stop_struct_layout_and_defaults():
    from pcreg_b200 import _lib
    from pcreg_b200.build import build_library
    assert C.sizeof(_lib.IcpStop) == 24
    build_library()
    s = _lib.IcpStop()
    _lib.load().pcreg_icp_stop_default(C.byref(s))
    assert (s.tol_t, s.tol_r_deg, s.window) == (0.01, 0.5, 3)
