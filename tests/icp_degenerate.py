"""Rank-deficient inputs of the ICP rigid fit, each built from a seed.  TEST INFRASTRUCTURE ONLY.

The Kabsch update of an ICP pass fits a rotation to H = sum w q~ m~', and that fit is ill-posed when H loses rank:
  rank 2   the model side of every correspondence lies on one plane (a flat region of the model): the rotation and the
           reflection fit equally well;
  rank 1   a collinear source (a ridge), or three weighted points on a line;
  rank 0   coincident source points.
A mirrored curved patch has full rank but really prefers a reflection, which reflection_fix = 0 reproduces (R = V*U').

Two kinds of builders:
  *_pair    one update's correspondences (m, q, w) and a pivot, for the host build of pcreg_math.cuh;
  *_problem a whole ICP problem (model, source, initial poses[, w_src]) for the GPU paths and the FP64 oracle.
Poses are row-vector 4 x 4 ([p 1] T), as everywhere in the project.
"""
from __future__ import annotations

import numpy as np

from pcreg_b200 import synth


def rng(seed):
    return synth.rng(seed)


def pose_about(R, c, t=(0.0, 0.0, 0.0)):
    """[p 1] T = (p - c) R' + c + t: rotation R (column convention) about the point c, then a shift t."""
    T = np.eye(4)
    T[:3, :3] = R.T
    T[3, :3] = c - c @ R.T + np.asarray(t, dtype=np.float64)
    return T


def frame(tilted, seed):
    """Orthonormal rows (e1, e2, n) of a face frame: the axes, or a random tilt of them."""
    if not tilted:
        return np.eye(3)
    R = synth.rot_axis_angle(rng(seed).standard_normal(3), 0.7)
    return R.T


def sums17(q, m, w, p):
    """The 17 one-pass sums of pcreg_math.cuh (KabschSums) relative to the pivot p."""
    qq, mm = q - p, m - p
    s = np.zeros(17)
    s[0] = w.sum()
    s[1:4] = (w[:, None] * qq).sum(0)
    s[4:7] = (w[:, None] * mm).sum(0)
    s[7:16] = ((w[:, None] * qq).T @ mm).reshape(9)
    s[16] = (w * ((m - q) ** 2).sum(1)).sum()
    return s


def kernel_H(s):
    """H as kabsch_from_sums forms it from the sums (same operations, same bits)."""
    inv = 1.0 / s[0]
    cm = s[4:7] * inv
    return s[7:16].reshape(3, 3) - s[1:4][:, None] * cm[None, :]


def oracle_H(m, q, w):
    """H as oracle.icp._weighted_kabsch forms it (two-pass, FP64)."""
    sw = w.sum()
    cd = (w[:, None] * m).sum(0) / sw
    cq = (w[:, None] * q).sum(0) / sw
    return ((q - cq) * w[:, None]).T @ (m - cd)


# ---- one update's correspondences ----

def flat_pair(seed, n=200, tilted=False, inplane_noise=False, offset=0.0):
    """Model side on a plane (z = 5, or a tilted plane through (0, 0, 5)), source = the model moved by a ~0.1 rad rotation plus
    N(0, 0.3) noise (or noise in the plane only).  The plane's points are at `offset` along (1, -1, 1) / sqrt(3) from the origin;
    the pivot is 30 along x from the patch."""
    g = rng(seed)
    F = frame(tilted, seed + 1)
    o = np.array([0.0, 0.0, 5.0]) + offset * np.array([1.0, -1.0, 1.0]) / np.sqrt(3.0)
    uv = g.uniform(-10.0, 10.0, (n, 2))
    m = o + uv[:, :1] * F[0] + uv[:, 1:] * F[1]
    if not tilted:
        m[:, 2] = o[2]                                          # exactly planar
    R = synth.rot_axis_angle(g.standard_normal(3), g.uniform(0.05, 0.15))
    noise = g.normal(0.0, 0.3, (n, 3))
    if inplane_noise:
        noise -= np.outer(noise @ F[2], F[2])
    q = (m - o) @ R + o + g.uniform(-1.0, 1.0, 3) + noise
    return m, q, np.ones(n), o + np.array([30.0, 0.0, 0.0])


def curved_pair(seed, sag, mirrored, n=200, pivot_offset=0.0):
    """A curved patch m = (x, y, sag * f(x, y)) on [-10, 10]^2 (f of order 10, not symmetric under any rotation), and q = the patch
    moved by a small rotation: with mirrored, q is first mirrored in the tangent plane (z -> -z), so the correspondences prefer
    a reflection.  sigma_3 / sigma_1 of H scales as sag^2.  The pivot sits at pivot_offset along (1, 1, 1) / sqrt(3) from the
    patch centre."""
    g = rng(seed)
    xy = g.uniform(-10.0, 10.0, (n, 2))
    x, y = xy[:, 0], xy[:, 1]
    f = 0.08 * x * x + 0.03 * y * y + 0.004 * x ** 3 + 0.05 * x * y + 0.2 * y
    c = np.array([3.0, -2.0, 7.0])
    m = c + np.stack([x, y, sag * f], axis=1)
    q = m - c
    if mirrored:
        q = q * np.array([1.0, 1.0, -1.0])
    R = synth.rot_axis_angle(g.standard_normal(3), g.uniform(0.05, 0.15))
    q = q @ R + c + g.uniform(-1.0, 1.0, 3)
    return m, q, np.ones(n), c + pivot_offset * np.ones(3) / np.sqrt(3.0)


def collinear_pair(seed, n=200):
    """Source on a line (rank 1), model a noisy neighbourhood of the moved line."""
    g = rng(seed)
    d = g.standard_normal(3)
    d /= np.linalg.norm(d)
    a = np.array([4.0, 1.0, -3.0])
    q = a + np.outer(g.uniform(-12.0, 12.0, n), d)
    R = synth.rot_axis_angle(g.standard_normal(3), 0.1)
    m = q @ R + g.uniform(-1.0, 1.0, 3) + g.normal(0.0, 0.3, (n, 3))
    return m, q, np.ones(n), a + np.array([30.0, 0.0, 0.0])


def coincident_pair(seed, n=50):
    """Every source point the same point (rank 0), the model side scattered."""
    g = rng(seed)
    q = np.tile(np.array([2.5, -1.25, 6.0]), (n, 1))
    m = q + g.normal(0.0, 0.5, (n, 3))
    return m, q, np.ones(n), np.array([32.5, -1.25, 6.0])


def three_weighted_pair(seed, n=60):
    """Weighted correspondences with only three positive weights, on three collinear source points (rank 1)."""
    g = rng(seed)
    q = g.normal(0.0, 5.0, (n, 3)) + np.array([1.0, 2.0, 3.0])
    d = np.array([1.0, 2.0, -0.5]) / np.linalg.norm([1.0, 2.0, -0.5])
    pick = g.choice(n, 3, replace=False)
    q[pick] = np.array([1.0, 2.0, 3.0]) + np.outer([-4.0, 1.0, 6.5], d)
    m = q + g.normal(0.0, 0.5, (n, 3))
    w = np.zeros(n)
    w[pick] = g.uniform(0.5, 2.0, 3)
    return m, q, w, np.array([31.0, 2.0, 3.0])


# ---- whole ICP problems ----

def face_model(seed, tilted, offset):
    """A slab whose top face is a plane (exactly, on the axis-aligned frame) and whose bottom is curved; returns (model, o, F):
    the face is o + u F[0] + v F[1], u, v in [-30, 30], with F[2] its outward normal.  12 000 face + 4 000 bottom points."""
    g = rng(seed)
    F = frame(tilted, seed + 1)
    o = offset * np.array([1.0, -1.0, 1.0]) / np.sqrt(3.0) + np.array([0.0, 0.0, 5.0])
    uv = g.uniform(-30.0, 30.0, (12_000, 2))
    face = o + uv[:, :1] * F[0] + uv[:, 1:] * F[1]
    if not tilted:
        face[:, 2] = o[2]
    uvb = g.uniform(-30.0, 30.0, (4_000, 2))
    wb = -20.0 + 3.0 * np.sin(uvb[:, 0] / 7.0) * np.cos(uvb[:, 1] / 9.0)
    back = o + uvb[:, :1] * F[0] + uvb[:, 1:] * F[1] + wb[:, None] * F[2]
    return np.concatenate([face, back]), o, F


def face_hypotheses(c, F, seed, n_spin=3, n_tilt=2):
    """Poses of the source about its centre c: spins about the face normal (up to 10 deg), spins combined with a tilt (up to
    4 deg about an in-plane axis) and a 1.5-unit in-plane shift."""
    g = rng(seed)
    out = []
    for k in range(n_spin):
        out.append(pose_about(synth.rot_axis_angle(F[2], np.deg2rad(g.uniform(-10.0, 10.0))), c,
                              g.uniform(-1.5, 1.5) * F[0] + g.uniform(-1.5, 1.5) * F[1]))
    for k in range(n_tilt):
        Rs = synth.rot_axis_angle(F[2], np.deg2rad(g.uniform(-10.0, 10.0)))
        Rt = synth.rot_axis_angle(g.uniform(-1.0, 1.0) * F[0] + g.uniform(-1.0, 1.0) * F[1], np.deg2rad(g.uniform(2.0, 4.0)))
        out.append(pose_about(Rt @ Rs, c, g.uniform(-1.5, 1.5) * F[0]))
    return np.stack(out)


def planar_problem(seed, tilted, offset, ns=400):
    """Source: ns points on the face (a disc of radius 12 about the face centre), so every correspondence's model point lies on
    the face and H has rank 2 at every update."""
    model, o, F = face_model(seed, tilted, offset)
    g = rng(seed + 7)
    r = 12.0 * np.sqrt(g.uniform(0.0, 1.0, ns))
    a = g.uniform(0.0, 2.0 * np.pi, ns)
    src = o + (r * np.cos(a))[:, None] * F[0] + (r * np.sin(a))[:, None] * F[1]
    if not tilted:
        src[:, 2] = o[2]
    return model, src, face_hypotheses(o, F, seed + 8)


def edge_problem(seed, ns=200):
    """A straight ridge of model points (x in [-30, 30], spacing 0.1) on top of the axis-aligned slab, and a collinear source on
    it (rank 1): the source is a stretch of the ridge line.  Hypotheses spin about the face normal and tilt."""
    model, o, F = face_model(seed, False, 0.0)
    ridge = o + np.outer(np.arange(-300, 301) * 0.1, F[0]) + 2.0 * F[2]
    g = rng(seed + 7)
    src = o + np.outer(g.uniform(-10.0, 10.0, ns), F[0]) + 2.0 * F[2]
    c = o + 2.0 * F[2]
    return np.concatenate([model, ridge]), src, face_hypotheses(c, F, seed + 8, n_spin=2, n_tilt=2)


def coincident_problem(seed, ns=64):
    """Every source point the same point above the face (rank 0)."""
    model, o, F = face_model(seed, False, 0.0)
    src = np.tile(o + np.array([1.3, -2.7, 0.4]), (ns, 1))
    return model, src, face_hypotheses(src[0], F, seed + 8, n_spin=2, n_tilt=1)


def three_weighted_problem(seed, ns=300):
    """A curved source patch with w_src zero except at three collinear points (weighted mode, rank 1)."""
    model = synth.make_model(20_000, seed)
    src, T_gt, c = synth.make_source(model, ns, 0.3, seed + 1)
    g = rng(seed + 2)
    a = int(g.integers(ns))
    d2 = ((src - src[a]) ** 2).sum(1)
    d2[a] = np.inf
    b = int(np.argmin(d2))                                           # a's nearest source point
    c3 = next(k for k in range(ns) if k not in (a, b))
    src[c3] = 0.5 * (src[a] + src[b])                                # on the chord a-b: near the surface, collinear with a, b
    pick = np.array([a, b, c3])
    w = np.zeros(ns)
    w[pick] = g.uniform(0.5, 1.0, 3)
    T0 = synth.pose_grid(T_gt, c, 2, (2, 1, 1), 4.0, 1.0, seed + 3)
    return model, src, T0, w


def mirrored_problem(seed, ns=400):
    """A curved model sheet z = f(x, y) over [-40, 40]^2 (24 000 points, no rotational symmetry) and a source that is a patch of
    it mirrored in the tangent plane at the patch centre, so the correspondences prefer a reflection at every update.
    Hypotheses: small spins about the normal and tilts about the centre."""
    g = rng(seed)
    xy = g.uniform(-40.0, 40.0, (24_000, 2))

    def f(x, y):
        return 0.03 * x * x + 0.012 * y * y + 0.0006 * x ** 3 + 0.01 * x * y

    model = np.stack([xy[:, 0], xy[:, 1], f(xy[:, 0], xy[:, 1])], axis=1)
    r = 10.0 * np.sqrt(g.uniform(0.0, 1.0, ns))
    a = g.uniform(0.0, 2.0 * np.pi, ns)
    x, y = r * np.cos(a), r * np.sin(a)
    src = np.stack([x, y, -f(x, y)], axis=1)                         # tangent plane at the origin: z = 0
    F = np.eye(3)
    return model, src, face_hypotheses(np.zeros(3), F, seed + 8, n_spin=2, n_tilt=2)
