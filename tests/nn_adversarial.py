"""Adversarial inputs for the exact nearest-neighbour paths -- TEST INFRASTRUCTURE ONLY (no GPU).

Every fast NN path of the library (brute force, grid walk, candidate lists, voxel map, fused ICP) scans in FP32, keeps
everything inside an error band and decides that in FP64.  Random data almost never puts two model points inside that
band, so these generators build queries whose two nearest model points are (nearly or exactly) equidistant:

  bisector    the midpoint of a model point and its nearest neighbour, moved along their difference by a relative
              gap spread from exact over a few FP64 ulps to 1e-3
  ties        exact FP64 ties whose coordinates are not FP32 values: mirror pairs q +- d and x/y-swapped offsets
  far         near-ties 3 to 1000 point spacings off the surface, many outside the model's (and voxel map's) box
  crowd       a sphere and a cylinder of points around empty cores, queries near the centre / axis
  huge        queries 1e4 to 1e30 model extents away (FP32 band terms overflow, FP64 distances collapse into ties)

Each generator returns (model, queries) from a seed and runs on any model VARIANT: dtype (float32 or float64), an
offset of the whole model and a scale.  The expected answer is always oracle.nn_brute.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

import oracle
from pcreg_b200 import synth

OFFSET_DIR = np.array([0.512, -0.302, 0.997])
# (dtype, offset, scale): both dtypes at three offsets, and both dtypes at two more scales
VARIANTS = [(dt, off, 1.0) for dt in (np.float32, np.float64) for off in (0.0, 1e3, 1e5)] + \
           [(dt, 0.0, sc) for dt in (np.float32, np.float64) for sc in (1e-3, 1e3)]
GAP_EDGES = (0.0, 1e-12, 1e-9, 1e-7, 1e-6, 1e-5)       # buckets: exact, (0,1e-12), [1e-12,1e-9), ... [1e-5, inf)


def variant_id(v):
    dt, off, sc = v
    return "%s-off%g-scale%g" % ("f32" if dt == np.float32 else "f64", off, sc)


def _place(p, dtype, offset, scale):
    """model coordinates of a synth-frame cloud: scaled, offset, rounded to the model's dtype"""
    return np.ascontiguousarray((np.asarray(p, dtype=np.float64) * scale + offset * OFFSET_DIR).astype(dtype))


def surface_model(n, seed, dtype=np.float32, offset=0.0, scale=1.0):
    return _place(synth.make_model(n, seed, np.float64), dtype, offset, scale)


def spacing(m64):
    d, _ = cKDTree(m64).query(m64[:: max(1, m64.shape[0] // 4000)], k=2)
    return float(np.median(d[:, 1]))


def rels(g, n):
    """signed relative gaps (second - first) / first: exact, a few FP64 ulps, log-uniform 1e-14 .. 1e-3"""
    u = g.uniform(size=n)
    r = np.where(u < 0.1, 0.0, np.where(u < 0.2, g.uniform(1, 8, n) * 2.0 ** -52, 10.0 ** g.uniform(-14, -3, n)))
    return r * g.choice([-1.0, 1.0], n)


def onto_bisector(m64, q, rel, rounds=3):
    """Move each query along the difference of its two nearest model points (a, b) until
    |q-b|^2 - |q-a|^2 = rel |q-a|^2 (a few rounds: the move may change which two are nearest)."""
    t = cKDTree(m64)
    q = np.array(q, dtype=np.float64)
    for _ in range(rounds):
        _, j = t.query(q, k=2)
        a, b = m64[j[:, 0]], m64[j[:, 1]]
        ab = b - a
        L2 = (ab * ab).sum(1)
        ok = L2 > 0
        qa = q - a
        D2 = (qa * qa).sum(1)
        f = L2 - 2.0 * (qa * ab).sum(1)                 # |q-b|^2 - |q-a|^2
        s = np.where(ok, (f - rel * D2) / (2.0 * np.where(ok, L2, 1.0)), 0.0)
        q = q + s[:, None] * ab
    return q


def bisector(seed, dtype=np.float32, offset=0.0, scale=1.0, n_model=30_000, nq=3000):
    model = surface_model(n_model, 1000 + seed, dtype, offset, scale)
    m = model.astype(np.float64)
    g = synth.rng(seed)
    d, j = cKDTree(m).query(m, k=2)
    cand = np.nonzero(d[:, 1] > 0)[0]
    p1 = g.choice(cand, nq, replace=nq > cand.size)
    A, B = m[p1], m[j[p1, 1]]
    u = B - A
    L = np.sqrt((u * u).sum(1))
    q = 0.5 * (A + B) + (rels(g, nq) * 0.125)[:, None] * u      # |q-B|^2 - |q-A|^2 = rel (L/2)^2
    return model, q


def ties(seed, dtype=np.float32, offset=0.0, scale=1.0, nq=3000):
    """Exact FP64 ties: pairs p = q +- d (mirror) and p = q + (dx,dy,dz), q + (dy,dx,dz) (swap).  q and d live on a binary
    grid (step 2^-40 of the largest magnitude for float64 models, the float32 ulp for float32 models) so that every
    difference is exact; q itself sits on the half step, so it is not an FP32 value.  Pairs are 6 scale units apart, the
    offsets at most 0.9: the pair is always the nearest.  The two points of a pair get random original indices."""
    g = synth.rng(seed)
    side = int(np.ceil(nq ** (1 / 3)))
    ijk = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)[:nq]
    c = (ijk * 6.0 + g.uniform(-1, 1, (nq, 3))) * scale + offset * OFFSET_DIR
    mag = np.abs(c).max() + 10.0 * scale
    bits = 40 if dtype == np.float64 else 23
    step = 2.0 ** (np.ceil(np.log2(mag)) - bits)
    qi = 2 * np.round(c / step).astype(np.int64)
    d = g.uniform(-0.9, 0.9, (nq, 3)) * scale
    di = 2 * np.round(d / step).astype(np.int64)
    mirror = g.uniform(size=nq) < 0.5
    # mirror pairs: q on the half grid (odd), d with the same parity, so q +- d are on the grid
    par = g.integers(0, 2, (nq, 3))
    qi = qi + np.where(mirror[:, None], par, 0)
    di = di + np.where(mirror[:, None], par, 0)
    p1 = np.where(mirror[:, None], (qi + di) // 2, qi // 2 + di // 2)
    p2 = np.where(mirror[:, None], (qi - di) // 2, qi // 2 + di[:, [1, 0, 2]] // 2)
    pts = np.vstack([p1, p2]).astype(np.float64) * step
    model = np.ascontiguousarray(pts[g.permutation(pts.shape[0])].astype(dtype))
    q = qi.astype(np.float64) * (0.5 * step)
    return model, q


def far(seed, dtype=np.float32, offset=0.0, scale=1.0, n_model=30_000, nq=3000):
    """near-ties 3 to 1000 point spacings from the surface (outward, or any direction), on the bisector of the two nearest"""
    model = surface_model(n_model, 2000 + seed, dtype, offset, scale)
    m = model.astype(np.float64)
    g = synth.rng(seed)
    sp = spacing(m)
    p = m[g.integers(0, m.shape[0], nq)]
    out = p - m.mean(0)
    out /= np.linalg.norm(out, axis=1, keepdims=True)
    rnd = g.normal(size=(nq, 3))
    rnd /= np.linalg.norm(rnd, axis=1, keepdims=True)
    dirn = np.where((g.uniform(size=nq) < 0.7)[:, None], out, rnd)
    k = 10.0 ** g.uniform(np.log10(3.0), 3.0, nq)
    q0 = p + dirn * (k * sp)[:, None]
    return model, onto_bisector(m, q0, rels(g, nq))


def crowd(seed, dtype=np.float32, offset=0.0, scale=1.0, n_model=30_000, n_crowd=3000, nq=3000):
    """A sphere (radius 6) and an x-aligned cylinder (radius 6, length 12) of points inside the surface model's empty core,
    each point's radius only as exact as its rounded coordinates; queries within 1e-9 .. 1e-1 radii of the sphere's centre
    and of the cylinder's axis."""
    g = synth.rng(seed)
    base = synth.make_model(n_model, 3000 + seed, np.float64)
    ctr = 0.5 * (base.min(0) + base.max(0))
    c1, c2, R = ctr + [0.0, 0.0, -12.0], ctr + [0.0, 0.0, 12.0], 6.0
    ns = n_crowd // 2
    v = g.normal(size=(ns, 3))
    sph = c1 + R * v / np.linalg.norm(v, axis=1, keepdims=True)
    ang = g.uniform(0, 2 * np.pi, n_crowd - ns)
    cyl = c2 + np.column_stack([g.uniform(-R, R, ang.size), R * np.cos(ang), R * np.sin(ang)])
    pts = np.vstack([base, sph, cyl])
    model = _place(pts[g.permutation(pts.shape[0])], dtype, offset, scale)
    nh = nq // 2
    e = g.normal(size=(nq, 3)) * (10.0 ** g.uniform(-9, -1, nq) * R)[:, None]
    q = np.vstack([c1 + e[:nh], c2 + np.column_stack([g.uniform(-0.6 * R, 0.6 * R, nq - nh), e[nh:, 1:]])])
    return model, q * scale + offset * OFFSET_DIR


def huge(seed, dtype=np.float32, offset=0.0, scale=1.0, n_model=30_000, nq=2000):
    """finite queries 1e4 .. 1e30 model extents away (random and axis directions); half of them moved onto the bisector of
    their two nearest model points (as far as FP64 can tell at that distance)"""
    model = surface_model(n_model, 4000 + seed, dtype, offset, scale)
    m = model.astype(np.float64)
    g = synth.rng(seed)
    ext = float((m.max(0) - m.min(0)).max())
    dirn = g.normal(size=(nq, 3))
    ax = g.uniform(size=nq) < 0.25
    dirn[ax] = np.eye(3)[g.integers(0, 3, ax.sum())] * g.choice([-1.0, 1.0], (ax.sum(), 1))
    dirn /= np.linalg.norm(dirn, axis=1, keepdims=True)
    K = 10.0 ** g.uniform(4, 30, nq)
    q = m.mean(0) + dirn * (K * ext)[:, None]
    h = nq // 2
    q[:h] = onto_bisector(m, q[:h], np.zeros(h), rounds=1)      # (a relative gap times |q|^2 would throw q much farther out)
    return model, q


GENERATORS = dict(bisector=bisector, ties=ties, far=far, crowd=crowd, huge=huge)


def generate(name, v, seed=1, **kw):
    dt, off, sc = v
    return GENERATORS[name](seed, dt, off, sc, **kw)


# ---- what makes an input adversarial -----------------------------------------------------------------------------------
def gaps(model, q, idx=None, d2=None):
    """relative gap (second - first) / first of the FP64 oracle; 0 for exact ties, inf for exact hits"""
    if idx is None:
        idx, d2 = oracle.nn_brute(model, q)
    sec = oracle.nn.nn_second(model, q, idx)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(d2 > 0, (sec - d2) / np.where(d2 > 0, d2, 1.0), np.where(sec > 0, np.inf, 0.0))


def gap_buckets(gap):
    """counts: [exact, (0,1e-12), [1e-12,1e-9), [1e-9,1e-7), [1e-7,1e-6), [1e-6,1e-5), >= 1e-5]"""
    out = [int(np.sum(gap == 0))]
    e = GAP_EDGES[1:] + (np.inf,)
    out.append(int(np.sum((gap > 0) & (gap < e[0]))))
    for lo, hi in zip(e[:-1], e[1:]):
        out.append(int(np.sum((gap >= lo) & (gap < hi))))
    return out


def naive_fp32(model, q, k=4):
    """a naive FP32 decision among the k nearest candidates (coordinates relative to the model centroid, rounded to
    float32, ties to the smaller index): what a kernel without an FP64 decision would return"""
    m = np.asarray(model, dtype=np.float64)
    _, j = cKDTree(m).query(q, k=min(k, m.shape[0]))
    j = j.reshape(q.shape[0], -1)
    c = m.mean(0)
    with np.errstate(over="ignore", invalid="ignore"):
        mq = (m[j] - c).astype(np.float32)
        qq = (np.asarray(q) - c).astype(np.float32)[:, None, :]
        d = (((mq[..., 0] - qq[..., 0]) ** 2 + (mq[..., 1] - qq[..., 1]) ** 2) + (mq[..., 2] - qq[..., 2]) ** 2).astype(np.float32)
    d = np.where(np.isnan(d), np.float32(np.inf), d)
    order = np.argsort(j, axis=1, kind="stable")
    js, ds = np.take_along_axis(j, order, 1), np.take_along_axis(d, order, 1)
    return js[np.arange(js.shape[0]), np.argmin(ds, axis=1)].astype(np.int32)


def quick_tf(src, T):
    return oracle.primitives.quickTF(src, T)
