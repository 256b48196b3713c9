"""The ICP update's rotation by polar3 (pcreg_math.cuh), on the host build of pcreg_math.cuh (no GPU needed).

  - polar3 against the svd3-based R = V U' on random H with sigma_1 / sigma_3 from 1 to 1e6, det of both signs, scales 1e-6 to 1e6:
    |Q - R_svd3|_F <= C eps sigma_1 / sigma_3 + 64 eps with C = 16, |Q'Q - I|_F <= 16 eps, sign det Q = sign det H, <= 7 steps;
  - the certificate of kabsch_rotation: matrices just either side of each clause take the intended path, and estimateTransform's
    update (no ICP rule) never takes polar3;
  - updates that must keep svd3 (rank 2, rank <= 1, noise-level H, S[2] / S[0] near tau, reflection_fix = 1 with det H < 0) give
    the bits of the svd3-only update (tests/golden/kabsch_svd_bits.json);
  - the H of every update of oracle ICP runs on a small C3-like problem take polar3 and give LAPACK's V U'."""
import ctypes as C
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import icp_degenerate as D  # noqa: E402
import oracle.icp as oicp  # noqa: E402
from pcreg_b200.build import build_hostmath  # noqa: E402

dp = C.POINTER(C.c_double)
EPS = np.finfo(np.float64).eps
TAU = oicp.RANK2_TAU


@pytest.fixture(scope="module")
def hm():
    lib = C.CDLL(build_hostmath())
    lib.hm_svd3.argtypes = [dp, dp, dp, dp]
    lib.hm_polar3.argtypes = [dp, dp]
    lib.hm_polar3.restype = C.c_int
    lib.hm_kabsch_rotation.argtypes = [dp, C.c_double, C.c_int, C.c_int, dp]
    lib.hm_kabsch_rotation.restype = C.c_int
    lib.hm_kabsch_from_sums_icp.argtypes = [dp, dp, dp, C.c_int, dp]
    for name in ("hm_icp_rank2_tau", "hm_icp_polar_det_c", "hm_icp_polar_noise_f"):
        getattr(lib, name).restype = C.c_double
    return lib


def _p(a):
    return a.ctypes.data_as(dp)


def polar(hm, H):
    Q = np.empty(9)
    it = hm.hm_polar3(_p(np.ascontiguousarray(H, dtype=np.float64)), _p(Q))
    return Q.reshape(3, 3), it


def svd3_R(hm, H):
    U, S, V = np.empty(9), np.empty(3), np.empty(9)
    hm.hm_svd3(_p(np.ascontiguousarray(H, dtype=np.float64)), _p(U), _p(S), _p(V))
    U, V = U.reshape(3, 3), V.reshape(3, 3)
    R = np.array([[V[r, 0] * U[c, 0] + V[r, 1] * U[c, 1] + V[r, 2] * U[c, 2] for c in range(3)] for r in range(3)])   # kabsch_rotation's order
    return R, S


def rotation(hm, H, f2, refl, icp=True):
    R = np.empty(9)
    path = hm.hm_kabsch_rotation(_p(np.ascontiguousarray(H, dtype=np.float64)), f2, int(refl), int(icp), _p(R))
    return R.reshape(3, 3), path


def random_orth(g):
    Q, _ = np.linalg.qr(g.standard_normal((3, 3)))
    return Q


def with_singular_values(g, s, sign):
    """U diag(s) V' with random U, V, scaled so that sign det = sign."""
    U, V = random_orth(g), random_orth(g)
    H = (U * s) @ V.T
    return H if np.sign(np.linalg.det(H)) == sign else -H


def test_certificate_constants(hm):
    c, nf = hm.hm_icp_polar_det_c(), hm.hm_icp_polar_noise_f()
    assert hm.hm_icp_rank2_tau() == TAU
    assert c >= 100 * TAU          # S[2] / S[0] >= c on the polar path: far from the rank rule's S[2] <= tau S[0]
    assert nf > 3.0 * (1 + 1e-3)   # |H|_F^2 <= 3 S[0]^2: S[0] strictly above the noise clause's tau sqrt(f2)


@pytest.mark.parametrize("kappa", [1.0, 10.0, 1e2, 1e3, 1e4, 1e5, 1e6])
def test_polar3_is_the_svd3_rotation(hm, kappa):
    g = np.random.default_rng(int(np.log10(kappa)) + 11)
    C_KAPPA = 16.0
    for t in range(400):
        mid = np.exp(g.uniform(0.0, np.log(kappa))) if kappa > 1 else 1.0
        s = np.array([1.0, 1.0 / mid, 1.0 / kappa]) * 10.0 ** g.uniform(-6.0, 6.0)
        sign = 1.0 if t % 2 == 0 else -1.0
        H = with_singular_values(g, s, sign)
        Q, it = polar(hm, H)
        assert 1 <= it <= 7, (kappa, t, it)
        R, S = svd3_R(hm, H)
        err = np.linalg.norm(Q - R)
        assert err <= C_KAPPA * EPS * S[0] / S[2] + 64 * EPS, (kappa, t, err)
        assert np.linalg.norm(Q.T @ Q - np.eye(3)) <= 16 * EPS
        assert np.sign(np.linalg.det(Q)) == sign


def test_polar3_reports_failure_on_singular_and_non_finite_input(hm):
    assert polar(hm, np.zeros((3, 3)))[1] == 0
    assert polar(hm, np.diag([1.0, 1.0, 0.0]))[1] == 0
    assert polar(hm, np.full((3, 3), np.nan))[1] == 0


def test_certificate_det_clause_either_side(hm):
    """|det H| > c |H|_F^3: with S = (1, s2, r) that is (s2 r)^2 > c^2 (1 + s2^2 + r^2)^3.  Just above the root r* the update takes
    polar3, just below it svd3, with both reflection_fix settings and both signs of det H (reflection_fix = 1 only for det H > 0)."""
    c = hm.hm_icp_polar_det_c()
    g = np.random.default_rng(5)
    for s2 in (1.0, 0.1, 1e-2):
        lo, hi = 0.0, 1.0                        # bisection for r*: f(r) = s2 r - c (1 + s2^2 + r^2)^1.5 changes sign once
        for _ in range(200):
            mid = 0.5 * (lo + hi)
            lo, hi = (lo, mid) if s2 * mid - c * (1 + s2 * s2 + mid * mid) ** 1.5 > 0 else (mid, hi)
        for sign in (1.0, -1.0):
            for refl in (0, 1):
                for r, want in ((hi * (1 + 1e-6), True), (hi * (1 - 1e-6), False)):
                    H = with_singular_values(g, np.array([1.0, s2, r]), sign)
                    R, path = rotation(hm, H, 0.0, refl)
                    fast = want and (refl == 0 or sign > 0)
                    assert (path > 0) == fast, (s2, sign, refl, r / hi)
                    Rs, _ = svd3_R(hm, H)
                    if fast:
                        assert np.linalg.norm(R - Rs) <= 16 * EPS / r + 64 * EPS
                    else:
                        # the svd3 path, rank rule not firing (S[2] / S[0] >= r ~ c s2^-1 >> tau): flipped only by reflection_fix
                        if refl and sign < 0:
                            assert np.linalg.det(R) > 0
                        else:
                            assert np.array_equal(R, Rs)


def test_certificate_noise_clause_either_side(hm):
    """|H|_F^2 >= ICP_POLAR_NOISE_F tau^2 f2, with f2 the squared norm of the uncentred sum: f2 just below the bound takes polar3,
    just above it svd3."""
    nf = hm.hm_icp_polar_noise_f()
    g = np.random.default_rng(6)
    H = with_singular_values(g, np.array([3.0, 2.0, 1.0]), 1.0)
    f2_star = np.sum(H * H) / (nf * TAU * TAU)
    assert rotation(hm, H, f2_star * (1 - 1e-9), 0)[1] > 0
    assert rotation(hm, H, f2_star * (1 + 1e-9), 0)[1] == 0


def test_estimate_transform_update_keeps_svd3(hm):
    g = np.random.default_rng(7)
    for refl in (0, 1):
        H = with_singular_values(g, np.array([3.0, 2.0, 1.0]), 1.0)
        R, path = rotation(hm, H, 0.0, refl, icp=False)
        assert path == 0 and np.array_equal(R, svd3_R(hm, H)[0])


def test_improper_fit_keeps_its_handedness(hm):
    """A mirrored patch (det H < 0, well conditioned) with reflection_fix = 0: polar3 returns the improper V U', as svd3 did."""
    m, q, w, p = D.curved_pair(3, 1.0, True)
    s = D.sums17(q, m, w, p)
    H = D.kernel_H(s)
    assert np.linalg.det(H) < 0
    R, path = rotation(hm, H, float(np.sum(s[7:16] ** 2)), 0)
    assert path > 0 and np.linalg.det(R) < 0
    assert np.linalg.norm(R - svd3_R(hm, H)[0]) <= 1e-13


def test_svd3_updates_keep_their_bits(hm):
    rows = json.load(open(os.path.join(ROOT, "tests", "golden", "kabsch_svd_bits.json")))
    kinds = {r["kind"] for r in rows}
    assert {"planar", "collinear", "coincident", "three-weighted", "between-tau-and-certificate", "mirrored"} <= kinds
    for r in rows:
        s = np.array([float.fromhex(v) for v in r["sums"]])
        p = np.array([float.fromhex(v) for v in r["pivot"]])
        dT = np.empty(16)
        hm.hm_kabsch_from_sums_icp(_p(s), _p(p), _p(p), r["refl"], _p(dT))
        want = np.array([float.fromhex(v) for v in r["dT"]])
        assert np.array_equal(dT, want), (r["kind"], r["refl"])
        f2 = 0.0
        for k in range(9):                       # kabsch_from_sums's f2, in its order
            f2 += s[7 + k] * s[7 + k]
        assert rotation(hm, D.kernel_H(s), f2, r["refl"])[1] == 0, (r["kind"], r["refl"])


def test_oracle_icp_updates_take_polar3(hm, monkeypatch):
    """Every H of oracle ICP runs on a small C3-like problem (bench.py's C3 pose grid and source, 50 000 model points, 1000
    source points, 24 of the poses, 30 KNN iterations): polar3 with at most 7 steps, and LAPACK's V U' to 1e-13."""
    from bench import WORKLOADS, make_inputs
    w = dict(WORKLOADS["c3"], nm=50_000, ns=1000)
    model, src, T0, _, _ = make_inputs(w, 0)
    rec = []
    kabsch = oicp._weighted_kabsch

    def spy(m_pts, q_pts, ww, refl):
        sw = ww.sum()
        cd = (ww[:, None] * m_pts).sum(axis=0) / sw
        cq = (ww[:, None] * q_pts).sum(axis=0) / sw
        rec.append((((q_pts - cq) * ww[:, None]).T @ (m_pts - cd), float(np.sum(((ww[:, None] * q_pts).T @ m_pts) ** 2))))
        return kabsch(m_pts, q_pts, ww, refl)

    monkeypatch.setattr(oicp, "_weighted_kabsch", spy)
    sel = np.linspace(0, T0.shape[0] - 1, 24).astype(int)
    oicp.icp_batch(model, src, T0[sel], mode=oicp.ICP_KNN, iters=w["iters"], k_frac=0.85)
    assert len(rec) == 24 * w["iters"]
    steps = []
    for H, f2 in rec:
        R, path = rotation(hm, H, f2, 0)
        U, _, Vt = np.linalg.svd(H)
        assert 1 <= path <= 7
        assert np.abs(R - Vt.T @ U.T).max() <= 1e-13
        steps.append(path)
    assert np.median(steps) <= 6
