"""The ICP rigid fit on rank-deficient correspondences, on the host build of pcreg_math.cuh (no GPU needed).

kabsch_from_sums with the ICP rank rule (ICP_RANK2_TAU) is checked against oracle.icp._weighted_kabsch, which states the same rule
in FP64 from a two-pass H and LAPACK's SVD:
  - a sweep of sigma_3 / sigma_1 from 1e-1 down to rounding, on data preferring the rotation and on a mirrored patch preferring the
    reflection, with the pivot near the patch and 1e3 away: the handedness is the oracle's except within a factor 8 of tau;
  - planar correspondences (axis-aligned and tilted plane): always proper, and the oracle's rotation;
  - rank <= 1 (collinear, coincident, three weighted collinear points): R is not unique, so only the invariants: the images of
    the source, orthogonality and det = +1;
  - extrap_step on an improper Kabsch pose: no step, the history restarts, the handedness is kept;
and the problem builders of tests/icp_degenerate.py are checked to be what they claim."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import icp_degenerate as D  # noqa: E402
import oracle.icp as oicp  # noqa: E402
from oracle.primitives import quickTF  # noqa: E402
from pcreg_b200.build import build_hostmath  # noqa: E402

dp = C.POINTER(C.c_double)
TAU = oicp.RANK2_TAU


@pytest.fixture(scope="module")
def hm():
    lib = C.CDLL(build_hostmath())
    lib.hm_kabsch_from_sums_icp.argtypes = [dp, dp, dp, C.c_int, dp]
    lib.hm_svd3.argtypes = [dp, dp, dp, dp]
    lib.hm_icp_rank2_tau.restype = C.c_double
    lib.hm_extrap_step.argtypes = [C.c_double, C.c_double, dp, dp, dp, dp, dp, C.c_int, dp, dp]
    lib.hm_extrap_step.restype = C.c_int
    return lib


def _p(a):
    return a.ctypes.data_as(dp)


def kernel_dT(hm, m, q, w, p, refl):
    s = D.sums17(q, m, w, p)
    dT = np.empty(16)
    hm.hm_kabsch_from_sums_icp(_p(s), _p(np.ascontiguousarray(p, dtype=np.float64)), _p(np.ascontiguousarray(p, dtype=np.float64)),
                               int(refl), _p(dT))
    return dT.reshape(4, 4)


def kernel_ratio(hm, m, q, w, p):
    """sigma_3 / sigma_1 of H as the kernel sees it (svd3 of the one-pass H)."""
    H = np.ascontiguousarray(D.kernel_H(D.sums17(q, m, w, p)))
    U, S, V = np.empty(9), np.empty(3), np.empty(9)
    hm.hm_svd3(_p(H), _p(U), _p(S), _p(V))
    return S[2] / S[0]


def oracle_ratio(m, q, w):
    S = np.linalg.svd(D.oracle_H(m, q, w), compute_uv=False)
    return S[2] / S[0], S[1] / S[0]


def test_tau_is_the_oracle_constant(hm):
    assert hm.hm_icp_rank2_tau() == TAU


SAGS = 10.0 ** np.arange(0.5, -9.01, -0.25)


@pytest.mark.parametrize("pivot_offset", [5.0, 1e3], ids=["pivot-near", "pivot-1e3"])
@pytest.mark.parametrize("mirrored", [False, True], ids=["rotation", "mirrored"])
def test_handedness_sweep_follows_the_oracle(hm, mirrored, pivot_offset):
    """sigma_3 / sigma_1 swept by the patch's sag; the kernel's det dT is the oracle's except within a factor 8 of tau, and R is the
    oracle's to 1e-10 wherever the decision agrees (sigma_2 stays well above sigma_3 here)."""
    seen = {0: set(), 1: set()}
    ratios = []
    for seed in range(4):
        for sag in SAGS:
            m, q, w, p = D.curved_pair(100 + seed, sag, mirrored, pivot_offset=pivot_offset)
            r3, r2 = oracle_ratio(m, q, w)
            ratios.append(r3)
            assert r2 > 0.1
            for refl in (0, 1):
                ref = oicp._weighted_kabsch(m, q, w, bool(refl))
                got = kernel_dT(hm, m, q, w, p, refl)
                dref, dgot = np.sign(np.linalg.det(ref[:3, :3])), np.sign(np.linalg.det(got[:3, :3]))
                seen[refl].add(dgot)
                if TAU / 8 <= r3 <= 8 * TAU:
                    continue
                assert dgot == dref, (seed, sag, r3, refl)
                # the reference's own rule: above tau reflection_fix = 0 keeps R = V*U' and its sign follows the data
                want = -1.0 if (mirrored and refl == 0 and r3 > TAU) else 1.0
                assert dref == want, (seed, sag, r3, refl)
                assert np.linalg.norm(got[:3, :3] - ref[:3, :3]) < 1e-10, (seed, sag, r3, refl)
                assert np.linalg.norm(got[3, :3] - ref[3, :3]) < 1e-9 * (1.0 + pivot_offset), (seed, sag, r3, refl)
    assert max(ratios) > 1e-1 and min(ratios) < 1e-15               # the sweep spans tau from far above to rounding
    assert seen[1] == {1.0}
    assert seen[0] == ({-1.0, 1.0} if mirrored else {1.0})          # the mirrored patch flips its handedness at tau


@pytest.mark.parametrize("offset", [0.0, 1e3])
def test_rounding_of_the_sums_stays_far_below_tau(hm, offset):
    """tau's margin: an exactly planar set (sag 0) 1e3 from the pivot and a tilted plane 1e3 from the origin keep the kernel's
    sigma_3 / sigma_1 below tau / 100."""
    worst = 0.0
    for seed in range(50):
        m, q, w, p = D.curved_pair(300 + seed, 0.0, False, pivot_offset=offset)
        worst = max(worst, kernel_ratio(hm, m, q, w, p))
        m, q, w, p = D.flat_pair(400 + seed, tilted=True, offset=offset)
        worst = max(worst, kernel_ratio(hm, m, q, w, p))
    assert worst < TAU / 100, worst


@pytest.mark.parametrize("offset", [0.0, 1e3])
@pytest.mark.parametrize("inplane", [False, True], ids=["noise-3d", "noise-in-plane"])
@pytest.mark.parametrize("tilted", [False, True], ids=["axis-plane", "tilted-plane"])
def test_planar_correspondences_give_the_oracle_rotation(hm, tilted, inplane, offset):
    """Rank 2: det dT = +1 in both modes and R within 1e-10 of the oracle's.  Without the rank rule about half of these updates
    come out improper (the sign of det(V U') is then set by how svd3 completes the null direction)."""
    improper = 0
    n = 0
    for seed in range(100):
        m, q, w, p = D.flat_pair(seed, tilted=tilted, inplane_noise=inplane, offset=offset)
        assert oracle_ratio(m, q, w)[0] < TAU / 100                  # the generator: H of rank 2
        for refl in (0, 1):
            ref = oicp._weighted_kabsch(m, q, w, bool(refl))
            got = kernel_dT(hm, m, q, w, p, refl)
            n += 1
            if np.linalg.det(got[:3, :3]) < 0:
                improper += 1
                continue
            assert np.linalg.det(ref[:3, :3]) > 0
            assert np.linalg.norm(got[:3, :3] - ref[:3, :3]) < 1e-10, (seed, refl)
            assert np.linalg.norm(got[3, :3] - ref[3, :3]) < 1e-9 * (1.0 + offset), (seed, refl)
    assert improper == 0, "%d of %d planar updates improper" % (improper, n)


def _extent(m, q, w):
    k = w > 0
    return max(np.max(np.linalg.norm(x[k] - x[k].mean(0), axis=1)) for x in (m, q))


@pytest.mark.parametrize("kind", ["collinear", "coincident", "three-weighted"])
def test_rank_le1_invariants(hm, kind):
    """Rank <= 1: R is not unique, the images of the weighted source points are.  They match the oracle's to 1e-12 x extent, R is
    orthogonal to 1e-12 and proper in both modes."""
    make = dict(collinear=D.collinear_pair, coincident=D.coincident_pair, **{"three-weighted": D.three_weighted_pair})[kind]
    improper = 0
    for seed in range(100):
        m, q, w, p = make(seed)
        k = w > 0
        ext = _extent(m, q, w)
        for refl in (0, 1):
            ref = oicp._weighted_kabsch(m, q, w, bool(refl))
            got = kernel_dT(hm, m, q, w, p, refl)
            R = got[:3, :3]
            assert np.max(np.abs(R.T @ R - np.eye(3))) < 1e-12, (seed, refl)
            improper += np.linalg.det(R) < 0
            assert np.linalg.det(ref[:3, :3]) > 0
            err = np.max(np.linalg.norm(quickTF(q[k], got) - quickTF(q[k], ref), axis=1))
            assert err < 1e-12 * ext, (seed, refl, err / ext)
    assert improper == 0, "%d of 200 rank <= 1 updates improper" % improper


# ---- extrap_step on improper Kabsch poses ----

def _extrap(hm, s, p, c, Tc, Tn, u, st):
    Tn = np.ascontiguousarray(Tn, dtype=np.float64).copy()
    tr = np.empty(5)
    br = hm.hm_extrap_step(10.0, 25.0, _p(s), _p(p), _p(c), _p(np.ascontiguousarray(Tc)), _p(Tn), u, _p(st), _p(tr))
    return br, Tn, tr


def _steady_run(hm, seed, n_upd, st=None, u0=0):
    """n_upd updates of a pose creeping along a slowly turning path, so the extrapolation fires; update u is passed as u0 + u and
    starts from the state st (zero: a fresh run).  Returns (src, m, p, c, poses, state, branches)."""
    g = D.rng(seed)
    src = g.normal(0.0, 5.0, (120, 3)) + np.array([10.0, -4.0, 2.0])
    m = src + np.array([1.0, 0.2, 0.0]) + g.normal(0.0, 0.05, src.shape)       # the target lies ahead of the path
    c = src.mean(0)
    p = np.array([12.0, -3.0, 1.0])
    st = np.zeros(20) if st is None else st
    axis = g.standard_normal(3)
    Ts = [np.eye(4)]
    brs = []
    for u in range(1, n_upd + 1):
        Tc = Ts[-1]
        K = Tc @ D.pose_about(D.synth.rot_axis_angle(axis, 0.002 / u), c, (0.05, 0.01, 0.0))
        q = quickTF(src, Tc)
        s = D.sums17(q, m, np.ones(len(q)), p)
        br, Tn, _ = _extrap(hm, s, p, c, Tc, K, u0 + u, st)
        brs.append(br)
        Ts.append(Tn)
    return src, m, p, c, Ts, st, brs


def test_extrap_step_skips_an_improper_update_and_restarts(hm):
    src, m, p, c, Ts, st, brs = _steady_run(hm, 5, 6)
    assert any(b != 0 for b in brs)                                   # the run does extrapolate
    n_ex = st[18]
    Tc = Ts[-1]
    q = quickTF(src, Tc)
    s = D.sums17(q, m, np.ones(len(q)), p)
    mirror = np.diag([1.0, 1.0, -1.0, 1.0])
    K = Tc @ D.pose_about(np.eye(3), c, (0.02, 0.0, 0.0)) @ mirror
    assert np.linalg.det(K[:3, :3]) < 0
    br, Tn, tr = _extrap(hm, s, p, c, Tc, K, 7, st)
    assert br == 0 and np.array_equal(Tn, K)                          # no step: T_u = K_u, improper as its Kabsch pose
    assert st[19] == 1.0 and st[18] == n_ex and math.isnan(tr[0]) and tr[3] == 0.0
    # an improper T_{u-1} is not extrapolated either, whatever K_u is
    K2 = Tn @ mirror
    br, Tn2, _ = _extrap(hm, s, p, c, Tn, K2, 8, st)
    assert br == 0 and np.array_equal(Tn2, K2) and np.linalg.det(Tn2[:3, :3]) > 0 and st[19] == 1.0
    # the next update with both poses proper starts the history afresh: the same bits as update 1 from a zero state
    K3 = Tn2 @ D.pose_about(D.synth.rot_axis_angle([0.0, 0.0, 1.0], 0.01), c, (0.01, 0.0, 0.0))
    fresh = np.zeros(20)
    b_f, T_f, tr_f = _extrap(hm, s, p, c, Tn2, K3, 1, fresh)
    b_r, T_r, tr_r = _extrap(hm, s, p, c, Tn2, K3, 9, st)
    assert b_r == b_f == 0 and np.array_equal(T_r, T_f)
    assert np.array_equal(st[:18], fresh[:18], equal_nan=True) and st[19] == 0.0 and st[18] == n_ex
    assert np.array_equal(tr_r, tr_f, equal_nan=True)


def test_extrap_restart_waits_two_updates_as_a_fresh_start(hm):
    """After a restart the updates behave as updates 1, 2, 3, .. of a fresh run: the same branches and poses, bit for bit (the
    first two cannot extrapolate), and the count of extrapolated updates carries on."""
    _, _, _, _, Ts_ref, _, brs_ref = _steady_run(hm, 6, 6)
    st = np.zeros(20)
    st[19], st[18] = 1.0, 4.0                                         # a restart pending, as after an improper update
    _, _, _, _, Ts, st, brs = _steady_run(hm, 6, 6, st=st, u0=20)
    assert brs == brs_ref and brs[0] == brs[1] == 0 and any(b != 0 for b in brs)
    assert all(np.array_equal(a, b) for a, b in zip(Ts, Ts_ref))
    assert st[18] == 4.0 + sum(b != 0 for b in brs_ref)


# ---- the problem builders ----

@pytest.mark.parametrize("offset", [0.0, 1e3])
@pytest.mark.parametrize("tilted", [False, True], ids=["axis-face", "tilted-face"])
def test_planar_problem_has_rank_2_at_every_oracle_pass(monkeypatch, tilted, offset):
    model, src, T0 = D.planar_problem(11 + int(tilted), tilted, offset)
    seen = []
    orig = oicp._weighted_kabsch

    def spy(m, q, w, refl):
        seen.append(oracle_ratio(m, q, w)[0])
        return orig(m, q, w, refl)

    monkeypatch.setattr(oicp, "_weighted_kabsch", spy)
    for mode in (oicp.ICP_PLAIN, oicp.ICP_KNN):
        r = oicp.icp_batch(model, src, T0, mode=mode, iters=12, thDist2=25.0)
        assert np.all(r["status"] == 0)
    assert len(seen) == 2 * 12 * T0.shape[0]
    assert max(seen) < TAU / 100, max(seen)


def test_mirrored_problem_makes_the_default_oracle_improper():
    model, src, T0 = D.mirrored_problem(5)
    for refl, sign in ((False, -1.0), (True, 1.0)):
        r = oicp.icp_batch(model, src, T0, mode=oicp.ICP_KNN, iters=12, reflection_fix=refl)
        assert np.all(np.sign(np.linalg.det(r["T"][:, :3, :3])) == sign)
        assert np.all(r["status"] == 0)


def test_degenerate_sources_have_the_stated_rank():
    _, src, _ = D.edge_problem(13)
    assert np.linalg.matrix_rank(src - src.mean(0)) == 1
    _, src, _ = D.coincident_problem(14)
    assert np.all(src == src[0])                                      # rank 0
    _, src, _, w = D.three_weighted_problem(20)
    k = w > 0
    assert k.sum() == 3 and np.linalg.matrix_rank(src[k] - src[k].mean(0), tol=1e-9) == 1
    for maker in (D.collinear_pair, D.three_weighted_pair):
        m, q, w, _ = maker(3)
        k = w > 0
        assert np.linalg.matrix_rank(q[k] - q[k].mean(0), tol=1e-9) == 1
