"""Host-side mirror of the reference's MATLAB interface for the alignment hot path.

Same names, argument meaning, return values and error behaviour as the reference .m functions
(AlignPoints.m, AlignPoints_KNN.m, AlignPoints_knn.m, AlignPoints_weighted.m, AlignPoints_c.m,
AlignPoints_KNN_c.m, estimateTransform.m, ransac.m) plus the batched / ICP forms; everything
computes in libpcreg_b200.so on the GPU through the C ABI of include/pcreg.h.  "Returns []" in the
reference is ``None`` here.  Indices are 0-based (Python), transforms are 4x4 row-vector form
T = [R 0; t 1] with [p 1] @ T (quickTF.m:5-7).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from ._lib import AlignOpts, DescOpts, IcpExtrap, IcpOpts, IcpStop, MatchOpts, ModelOpts, PcregError, RansacOpts  # noqa: F401

NN_BRUTE, NN_GRID = 0, 1
ICP_PLAIN, ICP_KNN, ICP_WEIGHTED = 0, 1, 2
ICP_POINT_TO_POINT, ICP_POINT_TO_PLANE, ICP_PLANE_TO_PLANE = 0, 1, 2
METRICS = {"point_to_point": ICP_POINT_TO_POINT, "point_to_plane": ICP_POINT_TO_PLANE}
# the plane-to-plane metric has entries of its own (pcreg_icp_batch_gicp{,_dev}); it is no value of pcreg_icp_batch_metric's `metric`
# (pcreg_icp_batch_windows{,_dev} take all three: ICP_PLANE_TO_PLANE)
PLANE_TO_PLANE = "plane_to_plane"
GICP_EPS = 1e-3
METRIC_SAD, METRIC_SSD = 0, 1
ALIGN_PLAIN, ALIGN_KNN_FRAC, ALIGN_KNN_ABS, ALIGN_WEIGHTED, ALIGN_C, ALIGN_KNN_C = range(6)


def _ptr(a, typ):
    return a.ctypes.data_as(typ) if a is not None else None


def _cm_points(pts):
    """N x 3 array -> (column-major array, is_double, n).  float32 stays float32 (class single)."""
    pts = np.asarray(pts)
    if pts.ndim != 2 or pts.shape[1] != 3:
        raise ValueError("points must be N x 3")
    if pts.dtype != np.float32:
        pts = pts.astype(np.float64, copy=False)
    a = np.asfortranarray(pts)
    return a, int(a.dtype == np.float64), a.shape[0]


def _T_to_abi(T):
    """(..., 4, 4) math layout -> contiguous MATLAB column-major records."""
    T = np.asarray(T, dtype=np.float64)
    return np.ascontiguousarray(np.swapaxes(T, -1, -2))


def _T_from_abi(buf, n=None):
    a = np.asarray(buf, dtype=np.float64)
    a = a.reshape(4, 4) if n is None else a.reshape(n, 4, 4)
    return np.ascontiguousarray(np.swapaxes(a, -1, -2))


# ------------------------------------------------------------------------------------------------
# model handle
# ------------------------------------------------------------------------------------------------
class Model:
    """GPU-resident model cloud (pcreg_model_create).  ``grid=True`` also builds the uniform grid and, unless
    ``voxel_map=-1`` (or the model is too dense for the memory budget), the Voronoi voxel map on top of it."""

    def __init__(self, pts, grid: bool = False, cell_size: float = 0.0, cells_per_point: float = 0.0,
                 max_cells: int = 0, shuffle_seed: int = 0, voxel_map: int = 0, voxel_scale: float = 0.0,
                 voxel_margin: float = 0.0, max_voxels: int = 0):
        lib = L.lib()
        a, is_double, n = _cm_points(pts)
        opts = ModelOpts(int(bool(grid)), float(cell_size), float(cells_per_point), int(max_cells), int(shuffle_seed),
                         int(voxel_map), float(voxel_scale), float(voxel_margin), int(max_voxels))
        h = C.c_void_p()
        L.check(lib.pcreg_model_create(a.ctypes.data_as(C.c_void_p), is_double, n, n, C.byref(opts), C.byref(h)),
                "pcreg_model_create")
        self._h = h
        self.n = n
        self.has_grid = bool(grid)

    @property
    def handle(self):
        if self._h is None:
            raise PcregError("model handle already destroyed")
        return self._h

    def grid_info(self):
        dims = (C.c_int32 * 3)()
        cell = C.c_double()
        occ = C.c_int64()
        L.check(L.lib().pcreg_model_grid_info(self.handle, dims, C.byref(cell), C.byref(occ)), "pcreg_model_grid_info")
        return dict(dims=tuple(dims), cell_size=cell.value, occupied=occ.value)

    def voxel_info(self):
        """Voronoi voxel map facts (dims all zero when the model has none)."""
        dims = (C.c_int32 * 3)()
        vs = C.c_double()
        st = (C.c_int64 * 10)()
        L.check(L.lib().pcreg_model_voxel_info(self.handle, dims, C.byref(vs), st), "pcreg_model_voxel_info")
        return dict(dims=tuple(dims), voxel_size=vs.value, voxels=st[0], listed=st[1], entries=st[2], too_long=st[3],
                    no_room=st[4], max_len=st[5], build_ms=st[6] / 1000.0, bytes=st[7], outside_band=st[8], band=st[9] * 1e-6)

    def nn_search(self, q, nn: int = NN_BRUTE):
        """knnsearch(model, q, 'K', 1): returns (idx int32 [nq] 0-based, d2 float64 [nq] squared distance)."""
        a, is_double, nq = _cm_points(q)
        idx = np.empty(nq, dtype=np.int32)
        d2 = np.empty(nq, dtype=np.float64)
        L.check(L.lib().pcreg_nn_search(self.handle, a.ctypes.data_as(C.c_void_p), is_double, nq, nq, int(nn),
                                        _ptr(idx, L.c_i32p), _ptr(d2, L.c_f64p)), "pcreg_nn_search")
        return idx, d2

    def set_normals(self, nrm):
        """Upload one normal per model point (N x 3, original order); each row is normalised in FP64.  A zero or non-finite
        row raises (PCREG_ERR_ARG)."""
        a, is_double, n = _cm_points(nrm)
        if n != self.n:
            raise ValueError("set_normals: need one normal per model point")
        L.check(L.lib().pcreg_model_set_normals(self.handle, a.ctypes.data_as(C.c_void_p), is_double, n), "pcreg_model_set_normals")

    def compute_normals(self, k: int = 6, viewpoint=None):
        """pcnormals(ptCloud, k) on the device (include/pcreg.h: pcreg_model_compute_normals): the smallest-eigenvalue direction
        of the k nearest model points of every point, oriented toward `viewpoint` or, without one, away from the centre of
        the bounding box.  Needs a model built with grid=True."""
        vp = None if viewpoint is None else np.ascontiguousarray(np.asarray(viewpoint, dtype=np.float64).reshape(3))
        L.check(L.lib().pcreg_model_compute_normals(self.handle, int(k), _ptr(vp, L.c_f64p)), "pcreg_model_compute_normals")

    def normals(self):
        """The model's unit normals, N x 3 float64 (raises when it has none)."""
        out = np.empty((3, self.n), dtype=np.float64)
        L.check(L.lib().pcreg_model_get_normals(self.handle, _ptr(out, L.c_f64p)), "pcreg_model_get_normals")
        return np.ascontiguousarray(out.T)

    def destroy(self):
        if self._h is not None:
            L.lib().pcreg_model_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def cloud_normals(pts, k: int = 6, viewpoint=None):
    """Unit normals of any N x 3 cloud (N x 3 float64), by Model.compute_normals' rule (pcnormals(ptCloud, k) semantics, computed
    on the device): a temporary grid-only model of the points is built, its normals read back, and the model destroyed.  Meant for
    the source normals of icp_batch(..., metric="plane_to_plane", src_normals=cloud_normals(src))."""
    m = Model(pts, grid=True, voxel_map=-1)
    try:
        m.compute_normals(k, viewpoint)
        return m.normals()
    finally:
        m.destroy()


# ------------------------------------------------------------------------------------------------
# pose application (quickTF.m, invertTF.m, AutoAlignPointclouds.m:8)
# ------------------------------------------------------------------------------------------------
TF_FORWARD, TF_INVERT, TF_MRDIVIDE = 0, 1, 2


def quickTF(pts, TF, mode: int = TF_FORWARD):
    """quickTF.m:1-8 on the GPU: [pts 1] * TF (class of pts kept).  mode=TF_INVERT applies invertTF(TF) (invertTF.m:5-7, as
    AutoAlignPointclouds2.m:25 does), mode=TF_MRDIVIDE computes [pts 1] / TF (AutoAlignPointclouds.m:8)."""
    a, is_double, n = _cm_points(pts)
    out = np.empty_like(a, order="F")
    T = _T_to_abi(np.asarray(TF, dtype=np.float64).reshape(4, 4))
    L.check(L.lib().pcreg_quick_tf(a.ctypes.data_as(C.c_void_p), is_double, n, n, _ptr(T, L.c_f64p), int(mode),
                                   out.ctypes.data_as(C.c_void_p), n), "pcreg_quick_tf")
    return np.ascontiguousarray(out)


# ------------------------------------------------------------------------------------------------
# getLocalPoints
# ------------------------------------------------------------------------------------------------
def getLocalPoints_batch(model: Model, centres, R, min_points, max_points, return_idx=False):
    """getLocalPoints.m:5-36 for many centres against the resident model: list of (pts_sphere, dists[, idx]) per
    centre (points relative to the centre, original model order), (None, None) where the reference returns []."""
    c = np.asfortranarray(np.asarray(centres, dtype=np.float64).reshape(-1, 3))
    nc = c.shape[0]
    counts = np.empty(nc, dtype=np.int64)
    status = np.empty(nc, dtype=np.int32)
    mx = -1 if max_points is None or np.isinf(max_points) else int(max_points)
    lib = L.lib()
    L.check(lib.pcreg_local_points_count(model.handle, _ptr(c, L.c_f64p), nc, nc, float(R), int(min_points), mx,
                                         _ptr(counts, L.c_i64p), _ptr(status, L.c_i32p)), "pcreg_local_points_count")
    offsets = np.zeros(nc + 1, dtype=np.int64)
    np.cumsum(np.where(status == 0, counts, 0), out=offsets[1:])
    nt = int(offsets[-1])
    out = np.zeros((max(nt, 1), 3), dtype=np.float64, order="F")
    dists = np.zeros(max(nt, 1), dtype=np.float64)
    idx = np.zeros(max(nt, 1), dtype=np.int32) if return_idx else None
    L.check(lib.pcreg_local_points_fill(model.handle, _ptr(c, L.c_f64p), nc, nc, float(R), _ptr(offsets, L.c_i64p),
                                        _ptr(status, L.c_i32p), _ptr(out, L.c_f64p), max(nt, 1), _ptr(dists, L.c_f64p),
                                        _ptr(idx, L.c_i32p)), "pcreg_local_points_fill")
    res = []
    for k in range(nc):
        if status[k] != 0:
            res.append((None, None, None) if return_idx else (None, None))
        else:
            a, b = offsets[k], offsets[k + 1]
            item = (np.ascontiguousarray(out[a:b]), dists[a:b].copy())
            res.append(item + (idx[a:b].copy(),) if return_idx else item)
    return res


def getLocalPoints(pts, R, c, min_points, max_points):
    """getLocalPoints.m:5-36 -> (pts_sphere, dists), or (None, None) for [].  `pts` may be an N x 3 array (uploaded
    for the call, as the reference signature has it) or a resident Model."""
    own = not isinstance(pts, Model)
    m = Model(pts) if own else pts
    try:
        return getLocalPoints_batch(m, np.asarray(c, dtype=np.float64).reshape(1, 3), R, min_points, max_points)[0]
    finally:
        if own:
            m.destroy()


# ------------------------------------------------------------------------------------------------
# getSpacialHistogramDescriptors
# ------------------------------------------------------------------------------------------------
def spatial_histogram_edges(R, num_r=10, num_theta=7, num_phi=14):
    """The bin edges exactly as getSpacialHistogramDescriptors.m:155-158 writes them (host arithmetic)."""
    r_bins = np.cbrt(np.arange(num_r + 1) * (float(R) ** 3 / num_r))            # nthroot(0:R^3/NUM_R:R^3, 3)
    phi_bins = -np.pi + np.arange(num_phi + 1) * (2 * np.pi / num_phi)          # -pi:2*pi/NUM_PHI:pi
    theta_bins = np.arange(num_theta + 1) * (np.pi / num_theta)                 # 0:pi/NUM_THETA:pi
    return r_bins, theta_bins, phi_bins


def getSpacialHistogramDescriptors(pts, sample_pts, options, return_status=False):
    """getSpacialHistogramDescriptors.m:2-183 -> (feat, desc): the keypoints that survive the getLocalPoints count
    limits and the eigenvalue-ratio rejection, and their 980-bin spherical histograms (one row each).  `pts` is the
    N x 3 cloud (uploaded for the call, as the reference signature has it) or a resident Model; `options` is the
    reference's struct as a dict: min_pts, max_pts, R, thVar, k ('all' or a fraction), ALIGN_POINTS."""
    own = not isinstance(pts, Model)
    # an uploaded cloud gets the uniform grid (no voxel map) when it is large: getLocalPoints then walks the ball's cell rows
    m = Model(pts, grid=np.shape(pts)[0] >= 200_000, voxel_map=-1) if own else pts
    try:
        kp = np.asfortranarray(np.asarray(sample_pts, dtype=np.float64).reshape(-1, 3))
        nk = kp.shape[0]
        o = DescOpts()
        L.lib().pcreg_desc_opts_default(C.byref(o))
        o.min_pts = int(options["min_pts"])
        mp = options.get("max_pts", np.inf)
        o.max_pts = -1 if mp is None or np.isinf(mp) else int(mp)
        o.R = float(options["R"])
        th = options.get("thVar", (1.0, 1.0))
        o.thVar[0], o.thVar[1] = float(th[0]), float(th[1])
        k = options.get("k", "all")
        o.k_frac = 0.0 if isinstance(k, str) else float(k)
        o.align_points = int(bool(options.get("ALIGN_POINTS", True)))
        er, et, ep = (np.ascontiguousarray(e, dtype=np.float64) for e in spatial_histogram_edges(o.R))
        nb = (len(er) - 1) * (len(et) - 1) * (len(ep) - 1)
        desc = np.empty((nk, nb), dtype=np.float64)
        status = np.empty(nk, dtype=np.int32)
        counts = np.empty(nk, dtype=np.int64)
        L.check(L.lib().pcreg_spatial_histogram(m.handle, _ptr(kp, L.c_f64p), nk, nk, C.byref(o), _ptr(er, L.c_f64p), len(er) - 1,
                                                _ptr(et, L.c_f64p), len(et) - 1, _ptr(ep, L.c_f64p), len(ep) - 1,
                                                _ptr(desc, L.c_f64p), _ptr(status, L.c_i32p), _ptr(counts, L.c_i64p)),
                "pcreg_spatial_histogram")
        ok = status == 0
        out = (np.ascontiguousarray(kp[ok]), desc[ok])                           # :176-179: valid rows, keypoint order
        return out + (status, counts) if return_status else out
    finally:
        if own:
            m.destroy()


# ------------------------------------------------------------------------------------------------
# getMatches
# ------------------------------------------------------------------------------------------------
def getMatches(descSurface, descModel, par: dict, return_metric=False):
    """getMatches.m:1-56 -> matches [P, 2] (0-based rows of descSurface / descModel, ascending surface row).

    `par` is the reference's struct as a dict: UNNORMALIZE, norm_factor, CHANGE_METRIC, metric_factor, Method,
    MatchThreshold, MaxRatio, Metric ('SAD' | 'SSD'), Unique.  par['Method'] is accepted and ignored: the search is
    exhaustive (what matchFeatures' 'Approximate' kd-forest approximates).  With return_metric also the score of
    every pair (matchFeatures' second output)."""
    d1 = np.asfortranarray(np.asarray(descSurface, dtype=np.float64))
    d2 = np.asfortranarray(np.asarray(descModel, dtype=np.float64))
    if d1.ndim != 2 or d2.ndim != 2 or d1.shape[1] != d2.shape[1]:
        raise ValueError("descriptors must be N1 x D and N2 x D")
    n1, n2, dim = d1.shape[0], d2.shape[0], d1.shape[1]
    o = MatchOpts()
    L.lib().pcreg_match_opts_default(C.byref(o))
    o.unnormalize = int(bool(par.get("UNNORMALIZE", False)))
    o.norm_factor = float(par.get("norm_factor", 2.0))
    o.change_metric = int(bool(par.get("CHANGE_METRIC", False)))
    o.metric_factor = float(par.get("metric_factor", 0.6))
    o.match_threshold = float(par.get("MatchThreshold", 1.0))          # matchFeatures defaults for non-binary features
    o.max_ratio = float(par.get("MaxRatio", 0.6))
    metric = str(par.get("Metric", "SSD")).upper()
    if metric not in ("SAD", "SSD"):
        raise ValueError("Metric must be 'SAD' or 'SSD'")
    o.metric = METRIC_SAD if metric == "SAD" else METRIC_SSD
    o.unique = int(bool(par.get("Unique", False)))
    pairs = np.empty((max(n1, 1), 2), dtype=np.int32)
    mm = np.empty(max(n1, 1), dtype=np.float64)
    n = C.c_int64()
    L.check(L.lib().pcreg_get_matches(_ptr(d1, L.c_f64p), n1, max(n1, 1), _ptr(d2, L.c_f64p), n2, max(n2, 1), dim, C.byref(o),
                                      _ptr(pairs, L.c_i32p), _ptr(mm, L.c_f64p), C.byref(n)), "pcreg_get_matches")
    pairs = pairs[:n.value].astype(np.int64)
    return (pairs, mm[:n.value].copy()) if return_metric else pairs


def transfer_colors(colored: Model, pts, colors, nn: int = NN_BRUTE):
    """ColorCodeModel.m:12-18: every point of `pts` takes the colour of its nearest point of the coloured cloud
    (findNearestNeighbors(pc_col, point, 1) in a loop there; one batched exact 1-NN search here)."""
    idx, _ = colored.nn_search(pts, nn)
    return np.asarray(colors)[idx]


# ------------------------------------------------------------------------------------------------
# AlignPoints family
# ------------------------------------------------------------------------------------------------
def align_points_batch(kind: int, pts_list, k_frac=0.85, k_abs=500, R_w=3.5, r_local=2.0, min_local=25,
                       C1=False, C2=False):
    """Batched AlignPoints*: list of N_b x 3 arrays (one class) -> list of
    (pts_aligned | None, coeff_unambig | None, c) per neighbourhood."""
    arrs = [np.asarray(p) for p in pts_list]
    single = all(a.dtype == np.float32 for a in arrs)
    dt = np.float32 if single else np.float64
    sizes = np.array([a.shape[0] for a in arrs], dtype=np.int64)
    offsets = np.zeros(len(arrs) + 1, dtype=np.int64)
    np.cumsum(sizes, out=offsets[1:])
    ntotal = int(offsets[-1])
    cat = np.asfortranarray(np.concatenate([a.astype(dt, copy=False).reshape(-1, 3) for a in arrs], axis=0)) \
        if ntotal else np.zeros((0, 3), dtype=dt, order="F")
    out = np.zeros_like(cat, order="F")
    nb = len(arrs)
    coeff = np.empty((nb, 9), dtype=np.float64)
    c3 = np.empty((nb, 3), dtype=np.float64)
    status = np.empty(nb, dtype=np.int32)
    o = AlignOpts(float(k_frac), int(k_abs), float(R_w), float(r_local), int(min_local), int(bool(C1)), int(bool(C2)))
    ld = max(ntotal, 1)
    L.check(L.lib().pcreg_align_points(int(kind), cat.ctypes.data_as(C.c_void_p), int(not single), ld if ntotal else ld,
                                       _ptr(offsets, L.c_i64p), nb, C.byref(o), out.ctypes.data_as(C.c_void_p),
                                       _ptr(coeff, L.c_f64p), _ptr(c3, L.c_f64p), _ptr(status, L.c_i32p)),
            "pcreg_align_points")
    res = []
    for b in range(nb):
        if status[b] != 0:
            res.append((None, None, c3[b].copy()))
        else:
            res.append((np.ascontiguousarray(out[offsets[b]:offsets[b + 1]]), coeff[b].reshape(3, 3).T.copy(), c3[b].copy()))
    return res


def AlignPoints(pts):
    """AlignPoints.m:1-29 -> (pts_aligned, coeff_unambig)."""
    a, cu, _ = align_points_batch(ALIGN_PLAIN, [pts])[0]
    return a, cu


def AlignPoints_KNN(pts, *varargin):
    """AlignPoints_KNN.m:1-60 -> (pts_aligned, coeff_unambig, c); optional (C1, C2) as in the reference."""
    C1, C2 = (bool(varargin[0]), bool(varargin[1])) if len(varargin) == 2 else (False, False)
    return align_points_batch(ALIGN_KNN_FRAC, [pts], C1=C1, C2=C2)[0]


def AlignPoints_knn(pts, K):
    """AlignPoints_knn.m:1-43 -> (pts_aligned, coeff_unambig, c)."""
    return align_points_batch(ALIGN_KNN_ABS, [pts], k_abs=int(K))[0]


def AlignPoints_weighted(pts):
    """AlignPoints_weighted.m:1-49 -> (pts_aligned, coeff_unambig, c)."""
    return align_points_batch(ALIGN_WEIGHTED, [pts])[0]


def AlignPoints_c(pts):
    """AlignPoints_c.m:1-44 -> (pts_aligned | None, coeff_unambig | None) ([] in the reference -> None)."""
    a, cu, _ = align_points_batch(ALIGN_C, [pts])[0]
    return a, cu


def AlignPoints_KNN_c(pts):
    """AlignPoints_KNN_c.m:1-57 -> (pts_aligned | None, coeff_unambig | None, c)."""
    return align_points_batch(ALIGN_KNN_C, [pts])[0]


# ------------------------------------------------------------------------------------------------
# estimateTransform / ransac
# ------------------------------------------------------------------------------------------------
def estimate_transform_batch(pts1_list, pts2_list, weights_list=None, reflection_fix=False):
    """Batched estimateTransform.m: returns (T [B,4,4] with NaN where degenerate, status [B])."""
    nb = len(pts1_list)
    sizes = np.array([np.asarray(p).shape[0] for p in pts1_list], dtype=np.int64)
    offsets = np.zeros(nb + 1, dtype=np.int64)
    np.cumsum(sizes, out=offsets[1:])
    nt = int(offsets[-1])
    p1 = np.asfortranarray(np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 3) for p in pts1_list], axis=0))
    p2 = np.asfortranarray(np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 3) for p in pts2_list], axis=0))
    if p1.shape != p2.shape:
        raise ValueError("pts1 and pts2 must have the same shapes")
    w = None
    if weights_list is not None:
        w = np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.float64).reshape(-1) for x in weights_list]))
    T = np.empty((nb, 16), dtype=np.float64)
    st = np.empty(nb, dtype=np.int32)
    L.check(L.lib().pcreg_kabsch_batch(_ptr(p1, L.c_f64p), _ptr(p2, L.c_f64p), _ptr(w, L.c_f64p), max(nt, 1),
                                       _ptr(offsets, L.c_i64p), nb, int(bool(reflection_fix)), _ptr(T, L.c_f64p),
                                       _ptr(st, L.c_i32p)), "pcreg_kabsch_batch")
    return _T_from_abi(T, nb), st


def estimateTransform(pts1, pts2, reflection_fix=False):
    """estimateTransform.m:2-74 -> T (4x4, [pts2,1] @ T = [pts1,1]) or None where the reference returns []."""
    T, st = estimate_transform_batch([pts1], [pts2], None, reflection_fix)
    return None if st[0] != 0 else T[0]


def ransac(pts1, pts2, coef: dict, triplets, reflection_fix=False, return_all=False):
    """ransac.m:21-116 with the sample triplets supplied (0-based [iterNum, 3]).

    coef: dict with thDist (SQUARED distance threshold), thInlrRatio, REFINE.  Returns a dict with the
    reference's five outputs (T, inlierIdx, numSuccess, maxInliers, pct) plus per-hypothesis counts;
    T is None where the reference returns []."""
    p1 = np.asfortranarray(np.asarray(pts1, dtype=np.float64))
    p2 = np.asfortranarray(np.asarray(pts2, dtype=np.float64))
    P = p1.shape[0]
    tri = np.ascontiguousarray(np.asarray(triplets, dtype=np.int32).reshape(-1, 3))
    nh = tri.shape[0]
    o = RansacOpts(float(coef["thDist"]), float(coef["thInlrRatio"]), int(bool(coef.get("REFINE", True))), int(bool(reflection_fix)))
    Tb = np.empty(16, dtype=np.float64)
    inl = np.empty(P, dtype=np.int32)
    n_inl, n_succ, max_inl, best = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
    cnt = np.empty(nh, dtype=np.int32)
    cntr = np.empty(nh, dtype=np.int32)
    Tall = np.empty((nh, 16), dtype=np.float64) if return_all else None
    rc = L.check(L.lib().pcreg_ransac_score(_ptr(p1, L.c_f64p), _ptr(p2, L.c_f64p), P, P, _ptr(tri, L.c_i32p), nh,
                                            C.byref(o), _ptr(Tb, L.c_f64p), _ptr(inl, L.c_i32p), C.byref(n_inl),
                                            C.byref(n_succ), C.byref(max_inl), C.byref(best), _ptr(cnt, L.c_i32p),
                                            _ptr(cntr, L.c_i32p), _ptr(Tall, L.c_f64p)), "pcreg_ransac_score")
    out = dict(inlrNum=cnt, inlrNum_refined=cntr)
    if return_all:
        out["T_all"] = _T_from_abi(Tall, nh)
    if rc != 0:
        out.update(T=None, inlierIdx=np.zeros(0, dtype=np.int64), numSuccess=0, maxInliers=0, pct=0.0, best=-1)
    else:
        out.update(T=_T_from_abi(Tb), inlierIdx=inl[:n_inl.value].astype(np.int64), numSuccess=int(n_succ.value),
                   maxInliers=int(max_inl.value), pct=100.0 * max_inl.value / P, best=int(best.value))
    return out


def ransac_seeded(pts1, pts2, coef: dict, seed: int = 0, reflection_fix=False, return_triplets=False):
    """The whole ransac.m call (coef.iterNum samples) with the sampling done on the device by the documented
    counter-based generator of include/pcreg.h (MATLAB's randperm stream cannot be matched).  Same dict as
    ransac(); with return_triplets the drawn samples are returned too (0-based [iterNum, 3])."""
    p1 = np.asfortranarray(np.asarray(pts1, dtype=np.float64))
    p2 = np.asfortranarray(np.asarray(pts2, dtype=np.float64))
    P = p1.shape[0]
    nh = int(coef["iterNum"])
    o = RansacOpts(float(coef["thDist"]), float(coef["thInlrRatio"]), int(bool(coef.get("REFINE", True))), int(bool(reflection_fix)))
    Tb = np.empty(16, dtype=np.float64)
    inl = np.empty(P, dtype=np.int32)
    n_inl, n_succ, max_inl, best = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
    tri = np.empty((nh, 3), dtype=np.int32) if return_triplets else None
    rc = L.check(L.lib().pcreg_ransac_run(_ptr(p1, L.c_f64p), _ptr(p2, L.c_f64p), P, P, nh, int(seed) & (2 ** 64 - 1), C.byref(o),
                                          _ptr(Tb, L.c_f64p), _ptr(inl, L.c_i32p), C.byref(n_inl), C.byref(n_succ),
                                          C.byref(max_inl), C.byref(best), _ptr(tri, L.c_i32p)), "pcreg_ransac_run")
    out = {}
    if return_triplets:
        out["triplets"] = tri
    if rc != 0:
        out.update(T=None, inlierIdx=np.zeros(0, dtype=np.int64), numSuccess=0, maxInliers=0, pct=0.0, best=-1)
    else:
        out.update(T=_T_from_abi(Tb), inlierIdx=inl[:n_inl.value].astype(np.int64), numSuccess=int(n_succ.value),
                   maxInliers=int(max_inl.value), pct=100.0 * max_inl.value / P, best=int(best.value))
    return out


def ransac_batch(pts1_list, pts2_list, coef: dict, seeds=None, triplets_list=None, reflection_fix=False):
    """ransac.m for a batch of matching windows in ONE call (the reference runs one `ransac` per window under parfor:
    slideMatchingWindow_v2.m:178-198).  Window w is (pts1_list[w], pts2_list[w]).  Samples: `triplets_list[w]`
    (0-based [iterNum, 3], the same iterNum for every window) or, when None, drawn on the device from `seeds[w]`
    (default seeds = 0..nwin-1) by the sampler of ransac_seeded().  Returns one dict per window with the reference's
    five outputs; T is None where the reference returns [] (also for windows with fewer than 3 pairs)."""
    nw = len(pts1_list)
    sizes = np.array([np.asarray(p).reshape(-1, 3).shape[0] for p in pts1_list], dtype=np.int64)
    offsets = np.zeros(nw + 1, dtype=np.int64)
    np.cumsum(sizes, out=offsets[1:])
    nt = int(offsets[-1])
    p1 = np.asfortranarray(np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 3) for p in pts1_list], axis=0))
    p2 = np.asfortranarray(np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 3) for p in pts2_list], axis=0))
    if p1.shape != p2.shape:
        raise ValueError("pts1 and pts2 must have the same shapes")
    tri = sd = None
    if triplets_list is not None:
        tri = np.ascontiguousarray(np.stack([np.asarray(t, dtype=np.int32).reshape(-1, 3) for t in triplets_list], axis=0))
        nh = tri.shape[1]
    else:
        nh = int(coef["iterNum"])
        sd = np.array([int(x) & (2 ** 64 - 1) for x in (range(nw) if seeds is None else seeds)], dtype=np.uint64)
        if sd.shape != (nw,):
            raise ValueError("one seed per window")
    o = RansacOpts(float(coef["thDist"]), float(coef["thInlrRatio"]), int(bool(coef.get("REFINE", True))), int(bool(reflection_fix)))
    T = np.empty((nw, 16), dtype=np.float64)
    inl = np.empty(max(nt, 1), dtype=np.int32)
    n_inl, n_succ, max_inl, best = (np.empty(nw, dtype=np.int64) for _ in range(4))
    st = np.empty(nw, dtype=np.int32)
    L.check(L.lib().pcreg_ransac_batch(_ptr(p1, L.c_f64p), _ptr(p2, L.c_f64p), max(nt, 1), _ptr(offsets, L.c_i64p), nw, nh,
                                       _ptr(tri, L.c_i32p), _ptr(sd, C.POINTER(C.c_uint64)), C.byref(o), _ptr(T, L.c_f64p),
                                       _ptr(inl, L.c_i32p), _ptr(n_inl, L.c_i64p), _ptr(n_succ, L.c_i64p), _ptr(max_inl, L.c_i64p),
                                       _ptr(best, L.c_i64p), _ptr(st, L.c_i32p)), "pcreg_ransac_batch")
    Ts = _T_from_abi(T, nw)
    out = []
    for w in range(nw):
        if st[w] != 0:
            out.append(dict(T=None, inlierIdx=np.zeros(0, dtype=np.int64), numSuccess=0, maxInliers=0, pct=0.0, best=-1))
        else:
            a = int(offsets[w])
            out.append(dict(T=Ts[w], inlierIdx=inl[a:a + int(n_inl[w])].astype(np.int64), numSuccess=int(n_succ[w]),
                            maxInliers=int(max_inl[w]), pct=100.0 * int(max_inl[w]) / int(sizes[w]), best=int(best[w])))
    return out


# ------------------------------------------------------------------------------------------------
# batched ICP
# ------------------------------------------------------------------------------------------------
def icp_opts(mode=ICP_PLAIN, iters=50, k_frac=0.85, R_w=3.5, thDist2=0.0, nn=NN_BRUTE, reflection_fix=False) -> IcpOpts:
    return IcpOpts(int(mode), int(iters), float(k_frac), float(R_w), float(thDist2), int(nn), int(bool(reflection_fix)))


def icp_stop(tol_t, tol_r_deg, window=3) -> IcpStop:
    return IcpStop(float(tol_t), float(tol_r_deg), int(window))


def icp_extrap(angle_deg=10.0, vmax_scale=25.0) -> IcpExtrap:
    return IcpExtrap(float(angle_deg), float(vmax_scale))


def _extrap_of(extrapolate, metric):
    """The `extrapolate` keyword -> an IcpExtrap or None: False / None off, True the defaults (10 deg, 25), or (angle_deg, vmax_scale)."""
    if extrapolate is None or extrapolate is False:
        return None
    if metric != "point_to_point":
        raise ValueError("extrapolate is defined for metric='point_to_point' only")
    return icp_extrap() if extrapolate is True else icp_extrap(*extrapolate)


def icp_batch(model: Model, src, T0s, mode=ICP_PLAIN, iters=50, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src=None,
              nn=NN_BRUTE, reflection_fix=False, return_idx=False, return_hist=False, tolerance=None, window=3,
              metric="point_to_point", src_normals=None, gicp_eps=GICP_EPS, extrapolate=False):
    """Multi-start ICP of `src` against the resident `model` from the initial poses T0s [H,4,4].
    Returns dict(T [H,4,4], rmse [H], n_used [H], status [H], best, idx [H,ns]?, rmse_hist [H,iters+1]?).

    tolerance=(tol_t, tol_r_deg): each hypothesis stops once the mean translation change (model units) and the mean
    rotation change (degrees) of its last `window` updates are both below these (include/pcreg.h: pcreg_icp_stop); the
    result then also holds n_iter [H] (pose updates applied) and converged [H] (1 = stopped by the tolerance).

    metric="point_to_plane" minimises the point-to-plane distance with the model's normals (Model.set_normals /
    Model.compute_normals; include/pcreg.h: pcreg_icp_batch_metric); correspondences, weights and rmse are unchanged.
    metric="plane_to_plane" is generalized ICP (include/pcreg.h: pcreg_icp_batch_gicp): it needs the model's normals and
    `src_normals` (N x 3, one per source point, e.g. cloud_normals(src)); gicp_eps in (0, 1] is the covariance epsilon.  The C entry
    takes the normals in the source's type, so with a float32 source they are rounded to float32 before the library normalises
    them in FP64; pass the source as float64 to keep float64 normals.

    extrapolate=True or (angle_deg, vmax_scale) (point-to-point only; default (10, 25)): each hypothesis's pose jumps ahead along its
    recent path when the last updates keep pointing the same way (Besl & McKay's accelerated ICP; include/pcreg.h: pcreg_icp_extrap).
    The result then also holds n_extrap [H], the updates that extrapolated."""
    if _extrap_of(extrapolate, metric) is not None:
        return icp_batch_windows(model, [src], [T0s], mode, iters, k_frac, R_w, thDist2, None if w_src is None else [w_src], nn,
                                 reflection_fix, return_idx, return_hist, tolerance, window, extrapolate=extrapolate)[0]
    if metric not in METRICS and metric != PLANE_TO_PLANE:
        raise ValueError("metric must be one of %s" % sorted(list(METRICS) + [PLANE_TO_PLANE]))
    if metric == PLANE_TO_PLANE and src_normals is None:
        raise ValueError("metric='plane_to_plane' needs src_normals (one normal per source point, e.g. cloud_normals(src))")
    if metric != PLANE_TO_PLANE and src_normals is not None:
        raise ValueError("src_normals is used only by metric='plane_to_plane'")
    a, is_double, ns = _cm_points(src)
    if src_normals is not None:
        sn = np.asfortranarray(np.asarray(src_normals).astype(a.dtype, copy=False))
        if sn.shape != (ns, 3):
            raise ValueError("src_normals must be N x 3, one normal per source point")
    T0 = _T_to_abi(np.asarray(T0s, dtype=np.float64).reshape(-1, 4, 4))
    H = T0.shape[0]
    o = icp_opts(mode, iters, k_frac, R_w, thDist2, nn, reflection_fix)
    w = None if w_src is None else np.ascontiguousarray(np.asarray(w_src, dtype=np.float64).reshape(ns))
    T = np.empty((H, 16), dtype=np.float64)
    rmse = np.empty(H, dtype=np.float64)
    n_used = np.empty(H, dtype=np.int32)
    status = np.empty(H, dtype=np.int32)
    idx = np.empty((H, ns), dtype=np.int32) if return_idx else None
    hist = np.empty((H, iters + 1), dtype=np.float64) if return_hist else None
    best = C.c_int64()
    args = (model.handle, a.ctypes.data_as(C.c_void_p), is_double, ns, ns, _ptr(w, L.c_f64p), _ptr(T0, L.c_f64p), H, C.byref(o))
    outs = (_ptr(T, L.c_f64p), _ptr(rmse, L.c_f64p), _ptr(n_used, L.c_i32p), _ptr(status, L.c_i32p), _ptr(idx, L.c_i32p),
            _ptr(hist, L.c_f64p), C.byref(best))
    n_iter = np.empty(H, dtype=np.int32) if tolerance is not None else None
    converged = np.empty(H, dtype=np.int32) if tolerance is not None else None
    stop = icp_stop(tolerance[0], tolerance[1], window) if tolerance is not None else None
    if metric == PLANE_TO_PLANE:
        L.check(L.lib().pcreg_icp_batch_gicp(*args[:6], sn.ctypes.data_as(C.c_void_p), float(gicp_eps), *args[6:],
                                             C.byref(stop) if stop is not None else None, *outs, _ptr(n_iter, L.c_i32p),
                                             _ptr(converged, L.c_i32p)), "pcreg_icp_batch_gicp")
    elif metric != "point_to_point":
        L.check(L.lib().pcreg_icp_batch_metric(*args, METRICS[metric], C.byref(stop) if stop is not None else None, *outs,
                                               _ptr(n_iter, L.c_i32p), _ptr(converged, L.c_i32p)), "pcreg_icp_batch_metric")
    elif tolerance is None:
        L.check(L.lib().pcreg_icp_batch(*args, *outs), "pcreg_icp_batch")
    else:
        L.check(L.lib().pcreg_icp_batch_stop(*args, C.byref(stop), *outs, _ptr(n_iter, L.c_i32p), _ptr(converged, L.c_i32p)),
                "pcreg_icp_batch_stop")
    out = dict(T=_T_from_abi(T, H), rmse=rmse, n_used=n_used, status=status, best=int(best.value))
    if tolerance is not None:
        out["n_iter"] = n_iter
        out["converged"] = converged
    if return_idx:
        out["idx"] = idx
    if return_hist:
        out["rmse_hist"] = hist
    return out


def icp_batch_windows(model: Model, src_list, T0_list, mode=ICP_PLAIN, iters=50, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src_list=None,
                      nn=NN_BRUTE, reflection_fix=False, return_idx=False, return_hist=False, tolerance=None, window=3,
                      metric="point_to_point", src_normals_list=None, gicp_eps=GICP_EPS, extrapolate=False):
    """icp_batch for many matching windows in ONE call (include/pcreg.h: pcreg_icp_batch_windows): window w polishes the poses
    T0_list[w] [H_w,4,4] (H_w may be 0) against its own source cloud src_list[w] [ns_w,3], with w_src_list[w] / src_normals_list[w]
    when given; the model and every other keyword (as icp_batch) are shared.  Returns one dict per window, each what
    icp_batch(model, src_list[w], T0_list[w], ...) returns (best relative to the window, -1 without hypotheses), bit for bit.
    The windows' sources are passed as float32 only when all of them are float32.  extrapolate: as icp_batch
    (include/pcreg.h: pcreg_icp_batch_extrap; each window's results are then those of its own icp_batch call)."""
    ex = _extrap_of(extrapolate, metric)
    if metric not in METRICS and metric != PLANE_TO_PLANE:
        raise ValueError("metric must be one of %s" % sorted(list(METRICS) + [PLANE_TO_PLANE]))
    if metric == PLANE_TO_PLANE and src_normals_list is None:
        raise ValueError("metric='plane_to_plane' needs src_normals_list (one N x 3 array of normals per window)")
    if metric != PLANE_TO_PLANE and src_normals_list is not None:
        raise ValueError("src_normals_list is used only by metric='plane_to_plane'")
    nw = len(src_list)
    if len(T0_list) != nw or (w_src_list is not None and len(w_src_list) != nw) or (src_normals_list is not None and len(src_normals_list) != nw):
        raise ValueError("one source, one pose array (and one w_src / normals array, when given) per window")
    srcs = [np.asarray(p).reshape(-1, 3) for p in src_list]
    dt = np.float32 if all(p.dtype == np.float32 for p in srcs) else np.float64
    ns = np.array([p.shape[0] for p in srcs], dtype=np.int64)
    soff = np.zeros(nw + 1, dtype=np.int64)
    np.cumsum(ns, out=soff[1:])
    nt = int(soff[-1])
    cat = np.asfortranarray(np.concatenate([p.astype(dt, copy=False) for p in srcs], axis=0)) if nt else np.zeros((1, 3), dtype=dt, order="F")
    sn = None
    if src_normals_list is not None:
        nrm = [np.asarray(x).reshape(-1, 3) for x in src_normals_list]
        if any(x.shape[0] != n for x, n in zip(nrm, ns)):
            raise ValueError("src_normals_list[w] must be N_w x 3, one normal per source point of window w")
        sn = np.asfortranarray(np.concatenate([x.astype(dt, copy=False) for x in nrm], axis=0)) if nt else np.zeros((1, 3), dtype=dt, order="F")
    T0s = [np.asarray(t, dtype=np.float64).reshape(-1, 4, 4) for t in T0_list]
    H = np.array([t.shape[0] for t in T0s], dtype=np.int64)
    hoff = np.zeros(nw + 1, dtype=np.int64)
    np.cumsum(H, out=hoff[1:])
    nh = int(hoff[-1])
    T0 = _T_to_abi(np.concatenate(T0s, axis=0)) if nh else np.zeros((1, 4, 4))
    w = None
    if w_src_list is not None:
        ws = [np.asarray(x, dtype=np.float64).reshape(-1) for x in w_src_list]
        if any(x.shape[0] != n for x, n in zip(ws, ns)):
            raise ValueError("w_src_list[w] must hold one weight per source point of window w")
        w = np.ascontiguousarray(np.concatenate(ws)) if nt else np.zeros(1)
    o = icp_opts(mode, iters, k_frac, R_w, thDist2, nn, reflection_fix)
    ioff = np.zeros(nw + 1, dtype=np.int64)
    np.cumsum(H * ns, out=ioff[1:])
    T = np.empty((max(nh, 1), 16), dtype=np.float64)
    rmse = np.empty(max(nh, 1), dtype=np.float64)
    n_used = np.empty(max(nh, 1), dtype=np.int32)
    status = np.empty(max(nh, 1), dtype=np.int32)
    idx = np.empty(max(int(ioff[-1]), 1), dtype=np.int32) if return_idx else None
    hist = np.empty((max(nh, 1), iters + 1), dtype=np.float64) if return_hist else None
    best = np.empty(nw, dtype=np.int64)
    stop = icp_stop(tolerance[0], tolerance[1], window) if tolerance is not None else None
    n_iter = np.empty(max(nh, 1), dtype=np.int32) if tolerance is not None else None
    converged = np.empty(max(nh, 1), dtype=np.int32) if tolerance is not None else None
    mcode = ICP_PLANE_TO_PLANE if metric == PLANE_TO_PLANE else METRICS[metric]
    n_extrap = np.empty(max(nh, 1), dtype=np.int32) if ex is not None else None
    outs = (_ptr(T, L.c_f64p), _ptr(rmse, L.c_f64p), _ptr(n_used, L.c_i32p), _ptr(status, L.c_i32p), _ptr(idx, L.c_i32p),
            _ptr(hist, L.c_f64p), _ptr(best, L.c_i64p), _ptr(n_iter, L.c_i32p), _ptr(converged, L.c_i32p))
    if ex is not None:
        L.check(L.lib().pcreg_icp_batch_extrap(model.handle, cat.ctypes.data_as(C.c_void_p), int(dt == np.float64), cat.shape[0],
                                               _ptr(soff, L.c_i64p), _ptr(w, L.c_f64p), _ptr(hoff, L.c_i64p), nw, _ptr(T0, L.c_f64p),
                                               C.byref(o), C.byref(stop) if stop is not None else None, C.byref(ex), *outs,
                                               _ptr(n_extrap, L.c_i32p)), "pcreg_icp_batch_extrap")
    else:
        L.check(L.lib().pcreg_icp_batch_windows(model.handle, cat.ctypes.data_as(C.c_void_p), int(dt == np.float64), cat.shape[0],
                                                _ptr(soff, L.c_i64p), _ptr(w, L.c_f64p),
                                                sn.ctypes.data_as(C.c_void_p) if sn is not None else None, float(gicp_eps),
                                                _ptr(hoff, L.c_i64p), nw, _ptr(T0, L.c_f64p), C.byref(o), mcode,
                                                C.byref(stop) if stop is not None else None, *outs), "pcreg_icp_batch_windows")
    Ts = _T_from_abi(T, T.shape[0])
    out = []
    for k in range(nw):
        a, b = int(hoff[k]), int(hoff[k + 1])
        r = dict(T=Ts[a:b].copy(), rmse=rmse[a:b].copy(), n_used=n_used[a:b].copy(), status=status[a:b].copy(), best=int(best[k]))
        if tolerance is not None:
            r["n_iter"] = n_iter[a:b].copy()
            r["converged"] = converged[a:b].copy()
        if ex is not None:
            r["n_extrap"] = n_extrap[a:b].copy()
        if return_idx:
            r["idx"] = idx[int(ioff[k]):int(ioff[k + 1])].reshape(b - a, int(ns[k])).copy()
        if return_hist:
            r["rmse_hist"] = hist[a:b].copy()
        out.append(r)
    return out


def icp_covariance(model: Model, src, T, mode=ICP_PLAIN, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src=None, nn=NN_BRUTE, ref=None,
                   targets=None, return_info=False):
    """Pose covariance of the point-to-plane objective at the poses T [H,4,4] (include/pcreg.h: pcreg_icp_covariance): one scoring pass
    with icp_batch's correspondences, rejection, mode and weights, no update.  Needs the model's normals.
    Returns dict(cov [H,6,6] (unknowns (omega, tau), rad and model units, about `ref` -- a model-frame point, default the origin),
    sigma2 [H], rmse [H], n_used [H], status [H] (1: degenerate, cov and tre NaN), tre [H,K] (the predicted RMS displacement of each
    model-frame target, targets [K,3]; [H,0] without targets), info [H,6,6]? (the unscaled Hessian, return_info=True)).
    For an icp_batch result passed with the same options, rmse and n_used equal that call's bit for bit."""
    return icp_covariance_windows(model, [src], [T], mode, k_frac, R_w, thDist2, None if w_src is None else [w_src], nn, ref, targets,
                                  return_info)[0]


def icp_covariance_windows(model: Model, src_list, T_list, mode=ICP_PLAIN, k_frac=0.85, R_w=3.5, thDist2=0.0, w_src_list=None,
                           nn=NN_BRUTE, ref=None, targets=None, return_info=False):
    """icp_covariance for many matching windows in ONE call: window w evaluates the poses T_list[w] [H_w,4,4] against its own source
    src_list[w] (with w_src_list[w] when given); ref, targets and every other keyword are shared.  One dict per window, each what
    icp_covariance(model, src_list[w], T_list[w], ...) returns."""
    nw = len(src_list)
    if len(T_list) != nw or (w_src_list is not None and len(w_src_list) != nw):
        raise ValueError("one source, one pose array (and one w_src array, when given) per window")
    srcs = [np.asarray(p).reshape(-1, 3) for p in src_list]
    dt = np.float32 if all(p.dtype == np.float32 for p in srcs) else np.float64
    ns = np.array([p.shape[0] for p in srcs], dtype=np.int64)
    soff = np.zeros(nw + 1, dtype=np.int64)
    np.cumsum(ns, out=soff[1:])
    nt = int(soff[-1])
    cat = np.asfortranarray(np.concatenate([p.astype(dt, copy=False) for p in srcs], axis=0)) if nt else np.zeros((1, 3), dtype=dt, order="F")
    Ts = [np.asarray(t, dtype=np.float64).reshape(-1, 4, 4) for t in T_list]
    hoff = np.zeros(nw + 1, dtype=np.int64)
    np.cumsum([t.shape[0] for t in Ts], out=hoff[1:])
    nh = int(hoff[-1])
    T = _T_to_abi(np.concatenate(Ts, axis=0)) if nh else np.zeros((1, 4, 4))
    w = None
    if w_src_list is not None:
        ws = [np.asarray(x, dtype=np.float64).reshape(-1) for x in w_src_list]
        if any(x.shape[0] != n for x, n in zip(ws, ns)):
            raise ValueError("w_src_list[w] must hold one weight per source point of window w")
        w = np.ascontiguousarray(np.concatenate(ws)) if nt else np.zeros(1)
    rf = None if ref is None else np.ascontiguousarray(np.asarray(ref, dtype=np.float64).reshape(3))
    tg = np.zeros((0, 3)) if targets is None else np.asarray(targets, dtype=np.float64).reshape(-1, 3)
    K = tg.shape[0]
    tg_cm = np.asfortranarray(tg) if K else None
    o = icp_opts(mode, 0, k_frac, R_w, thDist2, nn)
    H1 = max(nh, 1)
    cov = np.empty((H1, 36))
    info = np.empty((H1, 36)) if return_info else None
    sigma2, rmse = np.empty(H1), np.empty(H1)
    n_used, status = np.empty(H1, dtype=np.int32), np.empty(H1, dtype=np.int32)
    tre = np.empty((H1, max(K, 1)))
    L.check(L.lib().pcreg_icp_covariance(model.handle, cat.ctypes.data_as(C.c_void_p), int(dt == np.float64), cat.shape[0],
                                         _ptr(soff, L.c_i64p), _ptr(w, L.c_f64p), _ptr(hoff, L.c_i64p), nw, _ptr(T, L.c_f64p), C.byref(o),
                                         _ptr(rf, L.c_f64p), _ptr(tg_cm, L.c_f64p), K, _ptr(cov, L.c_f64p), _ptr(info, L.c_f64p),
                                         _ptr(sigma2, L.c_f64p), _ptr(rmse, L.c_f64p), _ptr(n_used, L.c_i32p), _ptr(status, L.c_i32p),
                                         _ptr(tre, L.c_f64p) if K else None), "pcreg_icp_covariance")
    out = []
    for k in range(nw):
        a, b = int(hoff[k]), int(hoff[k + 1])
        r = dict(cov=cov[a:b].reshape(-1, 6, 6).copy(), sigma2=sigma2[a:b].copy(), rmse=rmse[a:b].copy(), n_used=n_used[a:b].copy(),
                 status=status[a:b].copy(), tre=tre[a:b, :K].copy())
        if return_info:
            r["info"] = info[a:b].reshape(-1, 6, 6).copy()
        out.append(r)
    return out


def set_profiling(enabled):
    """True / 1: event times + work counters; 2: event times only (no counter atomics in the kernels); False: off."""
    L.check(L.lib().pcreg_set_profiling(int(enabled)), "pcreg_set_profiling")


def last_profile() -> dict:
    """Timing / device-side counts of the last ICP or NN call (include/pcreg.h: pcreg_last_profile)."""
    buf = (C.c_double * 32)()
    L.check(L.lib().pcreg_last_profile(buf), "pcreg_last_profile")
    v = list(buf)
    return dict(nn_launches=v[0], nn_ms=v[1], nn_queries=v[2], brute_pairs=v[3], update_launches=v[4],
                update_ms=v[5], correspondences=v[6], grid_points_visited=v[7] + v[15], grid_cells_visited=v[8] + v[16],
                grid_nodes_popped=v[9], certified_queries=v[10] - v[23], lazy_skipped_queries=v[23], walked_queries=v[11], rowscan_queries=v[12],
                list_entries_read=v[13], list_points_gathered=v[14],
                rowscan_points=v[7], rowscan_rows=v[8], walk_points=v[15], walk_leaves=v[16],
                list_ms=v[17], rowscan_ms=v[18], walk_ms=v[19], list_launches=v[20], rowscan_launches=v[21], walk_launches=v[22],
                match_score_ms=v[24], match_terms=v[25], voxel_map=v[26], fused=v[27], fused_phase_share=dict(nn=v[28], select=v[29], sums=v[30], svd=v[31]))


def launch_count() -> int:
    return int(L.load().pcreg_launch_count())
