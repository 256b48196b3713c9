/* pcreg.h -- C ABI of the B200-native PCReg alignment hot path (libpcreg_b200.so).
 *
 * This is the drop-in boundary: a MEX gateway (pcreg_b200/csrc/pcreg_mex.cpp), the Python
 * ctypes mirror (pcreg_b200/api.py) and any other host bind exactly these symbols.  No MATLAB,
 * torch or C++ types cross it.  The reference (LCJebe/PCReg) is MATLAB-only and has no FFI; each
 * entry point cites the reference .m interface it replaces (file:line into the reference tree).
 *
 * Conventions (reference: quickTF.m:5-7, estimateTransform.m:66-71)
 *   - Point sets are N x 3 COLUMN-MAJOR (MATLAB memory order): x[0..N), y at +ld, z at +2*ld
 *     elements; `is_double` selects float64 (1) or float32 (0) element type.
 *   - Rigid transforms are 4 x 4 ROW-VECTOR form T = [R 0; t 1],  p' = [p 1] * T, stored
 *     COLUMN-MAJOR (MATLAB order): element (r,c) at T16[c*4 + r].  Batches are contiguous 16-double
 *     records.
 *   - Indices are 0-based at this boundary (the MATLAB shims add 1).
 *   - Every call returns int status: 0 = OK; > 0 = degenerate input ("the reference returns []");
 *     < 0 = CUDA / allocation / argument error, text via pcreg_last_error().
 *   - There is NO CPU fallback: without a usable CUDA device every compute call returns
 *     PCREG_ERR_CUDA.
 */
#ifndef PCREG_H
#define PCREG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCREG_OK              0
#define PCREG_DEGENERATE      1     /* reference would return [] */
#define PCREG_ERR_ARG        -1
#define PCREG_ERR_CUDA       -2
#define PCREG_ERR_ALLOC      -3
#define PCREG_ERR_STATE      -4     /* not initialised / bad handle */

typedef struct pcreg_model pcreg_model;   /* opaque, GPU-resident model cloud */

/* ---- library lifetime ------------------------------------------------------------------- */
/* devices[0..ndev) are CUDA ordinals (devices == NULL or ndev == 0: ordinal 0).  With ndev > 1 the library drives all of
 * them from this one process -- the replacement of the reference's parfor over windows / trials
 * (slideMatchingWindow_v2.m:178, completeExperiment.m:265): pcreg_model_create replicates the model on every device,
 * pcreg_icp_batch shards its hypotheses and pcreg_ransac_batch its windows contiguously over the devices (one host thread
 * and stream set per device, no communication during the iterations), every device copies its result records straight
 * into its slice of the caller's arrays, and the winner is the first-index arg-min over all of them.  Results are
 * bit-identical for any ndev.  The other entry points run on devices[0].  Calling pcreg_init again re-initialises
 * (model handles of the previous device set become invalid).  One process per GPU over torch.distributed
 * (pcreg_b200/sharded.py) remains possible: each rank then calls pcreg_init with its own ordinal. */
int  pcreg_init(const int* devices, int ndev);
int  pcreg_device_count(void);              /* number of devices selected by the last pcreg_init (0 before) */
int  pcreg_shutdown(void);
const char* pcreg_last_error(void);
/* Number of kernels this library launched since pcreg_init (bench.py's gpu_launches claim). */
int64_t pcreg_launch_count(void);
/* ABI version of this header (bumped on any signature change). */
int  pcreg_abi_version(void);

/* ---- model cloud handle ----------------------------------------------------------------- */
typedef struct {
    int     build_grid;        /* 1: also build the uniform grid + occupancy pyramid (device counting sort) */
    double  cell_size;         /* grid cell edge; <= 0: automatic (about cells_per_point cells per point)   */
    double  cells_per_point;   /* automatic sizing target, <= 0 -> 32                                       */
    int64_t max_cells;         /* cap on level-0 cells, <= 0 -> 2^27                                        */
    uint64_t shuffle_seed;     /* seed of the brute-force scan order permutation (any value; 0 is fine)     */
    /* Voronoi voxel map on top of the grid (build_grid = 1): every voxel of a uniform grid over the padded bounding
     * box lists the model points that can be the nearest neighbour of a location inside it, so a grid-NN query is one
     * short contiguous list scan (nn_vox.cu).  Costs HBM (header 8 B per voxel + 16 B per entry).                   */
    int     voxel_map;         /* 0: automatic (built unless the model is too dense for the budget), 1: always, -1: never */
    double  voxel_scale;       /* voxel edge in units of the estimated point spacing, <= 0 -> 1.25                   */
    double  voxel_margin;      /* padding around the bounding box (model units); 0 -> 4 % of the largest extent, < 0 -> none.
                                  Queries outside the padded box are answered by the pyramid walk.                    */
    int64_t max_voxels;        /* cap on the number of voxels, <= 0 -> min(2^28, device memory / 512 B); denser models get a band-limited map */
} pcreg_model_opts;

/* Upload a model cloud (the dense CT/MRI cloud every driver loads once: completeExperiment.m:15,
 * slideMatchingWindow_v2.m:15; class single as written by upsampleMesh.m:21).  Builds the FP32
 * float4 scan array, the FP64 array used for exact re-checks and, if asked, the grid. */
int  pcreg_model_create(const void* xyz, int is_double, int64_t n, int64_t ld,
                        const pcreg_model_opts* opts, pcreg_model** out);
int  pcreg_model_destroy(pcreg_model* m);
int64_t pcreg_model_size(const pcreg_model* m);
/* Grid facts for roofline accounting: dims[3], cell size, number of non-empty level-0 cells. */
int  pcreg_model_grid_info(const pcreg_model* m, int32_t dims[3], double* cell_size, int64_t* occupied);
/* Voxel-map facts (all zero when the model has none): dims[3], voxel edge, stats = {voxels, voxels with a list, entries,
 * voxels without a list because it was too long, ... because the pool was full, longest list, build time in us, bytes,
 * voxels without a list because they lie outside the band, band width in 1e-6 model units (0: no band -- every voxel of
 * the padded box has a list; dense models get a band-limited map: only voxels near the model are listed)}. */
int  pcreg_model_voxel_info(const pcreg_model* m, int32_t dims[3], double* voxel_size, int64_t stats[10]);

/* ---- nearest neighbour (knnsearch(model, q, 'K', 1) semantics: Euclidean, FP64, ties -> smallest
 *      index; the reference's only literal cloud->cloud 1-NN loop is ColorCodeModel.m:15-18) ---- */
#define PCREG_NN_BRUTE 0
#define PCREG_NN_GRID  1
int  pcreg_nn_search(const pcreg_model* m, const void* q, int is_double, int64_t nq, int64_t ld,
                     int nn_kind, int32_t* idx /*[nq]*/, double* d2 /*[nq] squared distance, may be NULL*/);

/* ---- pose application to a whole cloud: quickTF.m:1-8, invertTF.m:1-8, AutoAlignPointclouds.m:8 ------------ */
#define PCREG_TF_FORWARD   0   /* [p 1] * T                          (quickTF.m:5-7)                                      */
#define PCREG_TF_INVERT    1   /* [p 1] * invertTF(T) = [R' 0; -t R' 1]  (quickTF(pts, invertTF(T)), AutoAlignPointclouds2.m:25) */
#define PCREG_TF_MRDIVIDE  2   /* [p 1] / T, the general 4x4 inverse  (AutoAlignPointclouds.m:8)                           */
/* pts: n x 3 column-major (ld), class single or double; out: the same class and shape (ld_out).  The last step of the
 * reference path on the full model cloud (16 M points in C5). */
int  pcreg_quick_tf(const void* pts, int is_double, int64_t n, int64_t ld, const double* T16, int mode, void* out, int64_t ld_out);

/* ---- getLocalPoints.m:5-36, batched over centres ------------------------------------------------ */
/* For each centre c_k (nc x 3 column-major doubles, ld): the model points with vecnorm(p - c_k) < R
 * (strict), RELATIVE to c_k, in ORIGINAL model order, class double.  Two calls:
 *   count: counts[k] and status[k] (1 where the reference returns []: count < min_points or > max_points;
 *          max_points < 0 means inf as in AlignPoints_c.m:14);
 *   fill : the caller builds offsets[nc+1] (rows of centre k = offsets[k]..offsets[k+1]-1, normally the
 *          prefix sum of the counts of the centres with status 0, zero-length for the others) and gets
 *          pts_rel (ntotal x 3 column-major, ld_out), optional dists (vecnorm) and optional original indices.
 * Models created with build_grid = 1 answer from the grid (cost ~ the points near the ball; 10^5 centres on a 16 M-point
 * model: ~14 ms); models without a grid scan the whole cloud per 32 centres.  Same results, bit for bit. */
int  pcreg_local_points_count(const pcreg_model* m, const double* centres, int64_t nc, int64_t ld, double R,
                              int64_t min_points, int64_t max_points, int64_t* counts, int32_t* status);
int  pcreg_local_points_fill(const pcreg_model* m, const double* centres, int64_t nc, int64_t ld, double R,
                             const int64_t* offsets, const int32_t* status, double* pts_rel, int64_t ld_out,
                             double* dists, int32_t* orig_idx);

/* ---- getSpacialHistogramDescriptors.m:2-183 (+ histcn.m:97-131), batched over keypoints --------- */
typedef struct {
    int64_t min_pts, max_pts;   /* options.min_pts / max_pts (getLocalPoints.m:31-34); max_pts < 0 = inf        */
    double  R;                  /* options.R: neighbourhood radius (3.5 in GetSphericalDescriptors.m:133-139)    */
    double  thVar[2];           /* options.thVar: eigenvalue-ratio rejection (:117-120); [1,1] = off             */
    double  k_frac;             /* options.k: fraction of the points nearest to the centroid used for the PCA
                                   (:76-84); <= 0 or 1 = 'all'                                                  */
    int     align_points;       /* options.ALIGN_POINTS: rotate into the disambiguated PCA frame (:128-144)      */
} pcreg_desc_opts;
void pcreg_desc_opts_default(pcreg_desc_opts* o);
/* keypoints: nkey x 3 column-major doubles (ld).  Bin edges as the reference builds them (:155-158): r_edges
 * [nr+1] = nthroot(0:R^3/nr:R^3, 3), theta_edges [nt+1] = 0:pi/nt:pi, phi_edges [np+1] = -pi:2*pi/np:pi.
 * desc: [nkey][nr*nt*np] doubles, descriptor k contiguous, element order reshape(counts, [], 1) of the
 * nr x nt x np histogram (:164); rows of rejected keypoints are NaN.  status[k]: 0 = valid, 1 = getLocalPoints
 * returned [] (:50-53), 2 = variance rejection (:117-120).  The reference returns only the valid rows, in keypoint
 * order (:176-179) -- the host mirror compacts.  counts (optional): points inside each keypoint's sphere. */
int  pcreg_spatial_histogram(const pcreg_model* m, const double* keypoints, int64_t nkey, int64_t ld,
                             const pcreg_desc_opts* opts, const double* r_edges, int nr, const double* theta_edges, int nt,
                             const double* phi_edges, int np, double* desc, int32_t* status, int64_t* counts);

/* ---- getMatches.m:1-56: descriptor weighting + matchFeatures, EXHAUSTIVE search ------------------------- */
#define PCREG_METRIC_SAD 0
#define PCREG_METRIC_SSD 1
typedef struct {
    int    unnormalize;      /* par.UNNORMALIZE: append norm_factor * mean 1-norm as an extra element (getMatches.m:22-27) */
    double norm_factor;      /* par.norm_factor (2, completeExperiment.m:113)                                            */
    int    change_metric;    /* par.CHANGE_METRIC: element-wise power before matching (getMatches.m:35-37)               */
    double metric_factor;    /* par.metric_factor (0.6, completeExperiment.m:116)                                        */
    double match_threshold;  /* par.MatchThreshold, percent of the largest possible score (10)                           */
    double max_ratio;        /* par.MaxRatio: nearest / second nearest score (0.99)                                      */
    int    metric;           /* par.Metric: PCREG_METRIC_SAD ('SAD') or PCREG_METRIC_SSD ('SSD')                          */
    int    unique;           /* par.Unique: forward-backward 1-to-1 matches only                                         */
} pcreg_match_opts;
void pcreg_match_opts_default(pcreg_match_opts* o);      /* the values of completeExperiment.m:112-122 */
/* desc_surface: n1 x dim, desc_model: n2 x dim, COLUMN-MAJOR doubles (element (i,k) at [k*ld + i]) -- the matrices
 * getSpacialHistogramDescriptors returns.  matchFeatures semantics (documentation, 'Method','Exhaustive'): rows are
 * normalised to unit vectors, every surface descriptor is paired with its nearest model descriptor (first index on
 * ties), pairs above MatchThreshold, above MaxRatio or (Unique) not mutually nearest are dropped.  par.Method =
 * 'Approximate' (the reference's setting) is a randomised kd-forest of the closed toolbox: this is the search it
 * approximates.  Outputs: index_pairs [n1][2] (pair p = {surface row, model row}, 0-based, ascending surface row;
 * first *n_matches valid), match_metric [n1] (optional: the score of each pair). */
int  pcreg_get_matches(const double* desc_surface, int64_t n1, int64_t ld1, const double* desc_model, int64_t n2, int64_t ld2,
                       int64_t dim, const pcreg_match_opts* opts, int32_t* index_pairs, double* match_metric, int64_t* n_matches);

/* ---- AlignPoints family (AlignPoints.m:1-29, AlignPoints_KNN.m:1-60, AlignPoints_knn.m:1-43,
 *      AlignPoints_weighted.m:1-49, AlignPoints_c.m:1-44, AlignPoints_KNN_c.m:1-57), batched over
 *      neighbourhoods ---------------------------------------------------------------------------- */
#define PCREG_ALIGN_PLAIN     0   /* AlignPoints          */
#define PCREG_ALIGN_KNN_FRAC  1   /* AlignPoints_KNN      */
#define PCREG_ALIGN_KNN_ABS   2   /* AlignPoints_knn      */
#define PCREG_ALIGN_WEIGHTED  3   /* AlignPoints_weighted */
#define PCREG_ALIGN_C         4   /* AlignPoints_c        */
#define PCREG_ALIGN_KNN_C     5   /* AlignPoints_KNN_c    */
typedef struct {
    double  k_frac;     /* 0.85  (AlignPoints_KNN.m:20)          */
    int64_t k_abs;      /* AlignPoints_knn's K                   */
    double  R_w;        /* 3.5   (AlignPoints_weighted.m:16)     */
    double  r_local;    /* 2.0   (AlignPoints_c.m:13)            */
    int64_t min_local;  /* 25    (AlignPoints_c.m:14)            */
    int     C1;         /* AlignPoints_KNN varargin{1}           */
    int     C2;         /* AlignPoints_KNN varargin{2}           */
} pcreg_align_opts;
void pcreg_align_opts_default(pcreg_align_opts* o);
/* pts: ntotal x 3 column-major (ld = leading dimension), neighbourhood b = rows
 * offsets[b] .. offsets[b+1]-1.  Outputs: pts_aligned (same shape/class/ld as pts), coeff9
 * [nbatch][9] column-major 3x3 coeff_unambig, c3 [nbatch][3] centroid, status [nbatch]
 * (0 ok, 1 = reference returns []; rows of that neighbourhood are then left untouched). */
int  pcreg_align_points(int kind, const void* pts, int is_double, int64_t ld,
                        const int64_t* offsets, int64_t nbatch, const pcreg_align_opts* opts,
                        void* pts_aligned, double* coeff9, double* c3, int32_t* status);

/* ---- estimateTransform.m:2-74, batched ------------------------------------------------------ */
/* p1, p2: ntotal x 3 column-major doubles (ld), problem b = rows offsets[b]..offsets[b+1]-1,
 * optional weights w[ntotal] (NULL = 1).  T16[b] satisfies [p2,1]*T = [p1,1].  status[b] = 1
 * where the reference's rank guard (estimateTransform.m:11-14) returns [].
 * reflection_fix = 0 reproduces the reference (R = V*U', no determinant check). */
int  pcreg_kabsch_batch(const double* p1, const double* p2, const double* w, int64_t ld,
                        const int64_t* offsets, int64_t nbatch, int reflection_fix,
                        double* T16, int32_t* status);

/* ---- ransac.m:21-116 hypothesis scoring, sample triplets supplied by the host ---------------- */
typedef struct {
    double thDist;          /* compared against SQUARED distances (ransac.m:49)   */
    double thInlrRatio;     /* thInlr = round(thInlrRatio * P) (ransac.m:28)       */
    int    refine;          /* coef.REFINE (ransac.m:53-61)                        */
    int    reflection_fix;  /* 0 = reference                                       */
} pcreg_ransac_opts;
/* p1, p2: P x 3 column-major doubles (ld).  triplets: nhyp x 3, 0-based, hypothesis-major
 * (triplets[3*h+k]).  Outputs: T16_best (16), inl_idx [P] (first *n_inl entries valid, 0-based,
 * ascending), n_succ, max_inl, best_hyp (-1 on failure), optional per-hypothesis counts
 * inl_counts[nhyp] (3-point fit) and inl_counts_refined[nhyp], optional T16_all [nhyp][16]
 * (the TForms kept by ransac.m:60/63; NaN-filled where none).  Returns PCREG_DEGENERATE where
 * ransac.m:75-89 returns T = []. */
int  pcreg_ransac_score(const double* p1, const double* p2, int64_t P, int64_t ld,
                        const int32_t* triplets, int64_t nhyp, const pcreg_ransac_opts* opts,
                        double* T16_best, int32_t* inl_idx, int64_t* n_inl, int64_t* n_succ,
                        int64_t* max_inl, int64_t* best_hyp,
                        int32_t* inl_counts, int32_t* inl_counts_refined, double* T16_all);

/* The whole ransac.m:21-116 call with the sampling on the device.  MATLAB's global RNG stream
 * (randperm, ransac.m:42) cannot be matched, so the drop-in defines a documented counter-based sampler:
 * u_k = splitmix64(seed + 0x9E3779B97F4A7C15 * (3h+k+1)); i0 = u0 mod P, i1 = u1 mod (P-1) skipping i0,
 * i2 = u2 mod (P-2) skipping both -- a uniformly random ordered 3-subset, like randperm(P)(1:3).
 * triplets_out (optional, [iter_num][3]) returns the samples that were drawn.  Same outputs / return
 * value as pcreg_ransac_score. */
int  pcreg_ransac_run(const double* p1, const double* p2, int64_t P, int64_t ld, int64_t iter_num, uint64_t seed,
                      const pcreg_ransac_opts* opts, double* T16_best, int32_t* inl_idx, int64_t* n_inl,
                      int64_t* n_succ, int64_t* max_inl, int64_t* best_hyp, int32_t* triplets_out);

/* ransac.m:21-116 for a BATCH of windows in one call -- the reference runs one ransac per matching window under
 * parfor (slideMatchingWindow_v2.m:178-198: 21 windows per experiment, completeExperiment.m:265-278); here all
 * windows x iter_num hypotheses are one launch.  p1, p2: ntotal x 3 column-major doubles (ld); window w = rows
 * offsets[w] .. offsets[w+1]-1 (P_w pairs, thInlr = round(thInlrRatio * P_w) per window).
 * Samples: triplets != NULL -> [nwin][iter_num][3], 0-based RELATIVE to the window; else window w draws
 * iter_num samples with pcreg_ransac_run's sampler from seeds[w].
 * Outputs per window: T16 [nwin][16] (NaN where the reference returns []), inl_idx [ntotal] (window w's inliers,
 * 0-based relative to the window, ascending, in inl_idx[offsets[w] .. offsets[w]+n_inl[w]-1]), n_inl, n_succ,
 * max_inl, best_hyp (-1 = none), status [nwin]: 0 ok, 1 = T = [] (ransac.m:75-89; also a window with fewer than
 * 3 pairs, where the reference's randperm(ptNum)(1:3) would throw).  Each window's result equals a
 * pcreg_ransac_run / pcreg_ransac_score call on that window alone. */
int  pcreg_ransac_batch(const double* p1, const double* p2, int64_t ld, const int64_t* offsets, int64_t nwin,
                        int64_t iter_num, const int32_t* triplets, const uint64_t* seeds,
                        const pcreg_ransac_opts* opts, double* T16, int32_t* inl_idx, int64_t* n_inl,
                        int64_t* n_succ, int64_t* max_inl, int64_t* best_hyp, int32_t* status);

/* ---- batched ICP (composition of quickTF.m, the 85 % trim rule AlignPoints_KNN.m:20-26, the
 *      weights of AlignPoints_weighted.m:16-18, estimateTransform.m:41-71 and ransac.m's
 *      score / first-arg-best structure around an exact NN step; SURVEY.md section 8c) --------- */
#define PCREG_ICP_PLAIN    0
#define PCREG_ICP_KNN      1
#define PCREG_ICP_WEIGHTED 2
typedef struct {
    int    mode;            /* PCREG_ICP_*                                             */
    int    iters;           /* pose updates; one extra NN pass scores the final pose   */
    double k_frac;          /* KNN: keep round(k_frac * n_kept) smallest residuals     */
    double R_w;             /* WEIGHTED: w = max(R_w - r, 0)                           */
    double thDist2;         /* > 0: reject correspondences with d^2 >= thDist2         */
    int    nn;              /* PCREG_NN_BRUTE / PCREG_NN_GRID                          */
    int    reflection_fix;  /* 0 = reference; see the rank rule below                  */
} pcreg_icp_opts;
/* Rank rule of the ICP update (the project's own: the reference has no ICP).  The update fits a rotation to the cross-covariance H
 * of its correspondences (singular values S[0] >= S[1] >= S[2]).  When H is numerically of rank <= 2 -- S[2] <= tau S[0], or
 * S[0] <= tau |sum w q~ m~'|_F (H is rounding noise: coincident correspondences) -- the rotation and the reflection fit them
 * equally well (a flat region of the model, a ridge, a collinear source), and the update takes the PROPER solution whatever
 * reflection_fix says.  Above that, reflection_fix = 0 reproduces R = V*U', reflections included (a patch mirrored in its tangent
 * plane), and 1 always returns a rotation.  tau = 1e-8: the one-pass pivot-relative sums leave S[2] / S[0] of an exactly planar set
 * at up to ~4e-15 (D / L)^2 for a patch of size L at distance D >= L from the model's pivot (4e-11 at D = 100 L), and a curved patch
 * has S[2] / S[0] ~ (sag / L)^2, so only a patch flatter than a relative sag of 1e-4 counts as planar.  estimateTransform and
 * RANSAC do not apply the rule. */
void pcreg_icp_opts_default(pcreg_icp_opts* o);
/* src: ns x 3 column-major; w_src[ns] optional; T0_16 [nhyp][16] initial poses.  Outputs (any
 * may be NULL except T16): T16 [nhyp][16], rmse [nhyp], n_used [nhyp], status [nhyp] (0 ok,
 * 1 = fewer than 3 usable correspondences at some iteration: pose frozen there), idx
 * [nhyp][ns] final correspondences, rmse_hist [nhyp][iters+1], best = first-index arg-min of
 * rmse (-1 if all NaN). */
int  pcreg_icp_batch(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld,
                     const double* w_src, const double* T0_16, int64_t nhyp,
                     const pcreg_icp_opts* opts,
                     double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx,
                     double* rmse_hist, int64_t* best);

/* Same, with every array already resident on the device the library was initialised on
 * (src as float64 column-major, ld = ns) and launched on `stream` (a cudaStream_t passed as
 * void*; NULL = default stream).  Nothing crosses PCIe, but the call is SYNCHRONOUS with respect to
 * `stream`: it returns after its last kernel has finished (its scratch buffers go back to the pool on
 * return).  `best` is a device int64.  This is the entry bench.py's device-resident `value` is timed
 * through. */
int  pcreg_icp_batch_dev(const pcreg_model* m, const double* d_src, int64_t ns,
                         const double* d_w_src, const double* d_T0_16, int64_t nhyp,
                         const pcreg_icp_opts* opts,
                         double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status,
                         int32_t* d_idx, double* d_rmse_hist, int64_t* d_best, void* stream);

/* Convergence tolerance: each hypothesis stops once its pose stops changing.
 * Poses are row-vector T = [R 0; t 1]; update u (1..iters) takes T_{u-1} to T_u = T_{u-1} dT_u.  Its motion is
 *   dt_u = |t_u - t_{u-1}|_2                                   (model units)
 *   dr_u = atan2(|v|, (trace(dR) - 1) / 2) * 180 / pi           (degrees; dR = R_{u-1}' R_u is dT_u's rotation block,
 *          v = (dR32 - dR23, dR13 - dR31, dR21 - dR12) / 2;  not acos, which is inaccurate at small angles)
 * After update u >= window the hypothesis STOPS when mean(dt) < tol_t and mean(dr) < tol_r_deg over updates
 * u-window+1 .. u (each mean a left-to-right FP64 sum divided by window; strict compares: a tolerance of 0 never stops,
 * +inf switches that criterion off).  The stopping update is applied: T_u is the final pose, n_iter = u, converged = 1.
 * A stopped hypothesis returns exactly what pcreg_icp_batch with iters = n_iter returns for it (T, rmse, n_used, status,
 * idx, bit for bit); its rmse_hist columns 0..n_iter are that call's and columns n_iter..iters all hold the final rmse.
 * A degenerate update (status 1) stops the hypothesis too: n_iter = the updates applied before it, converged = 0.
 * The rule restates the documented 'Tolerance' of MATLAB's pcregistericp (a translation and a rotation difference averaged
 * over the three most recent iterations); the toolbox is not available to compare against, so parity is UNPINNED. */
typedef struct {
    double tol_t;           /* mean translation change, model units                    */
    double tol_r_deg;       /* mean rotation change, degrees                           */
    int    window;          /* updates averaged, 1..16                                 */
} pcreg_icp_stop;
void pcreg_icp_stop_default(pcreg_icp_stop* s);        /* {0.01, 0.5, 3} */
/* pcreg_icp_batch / pcreg_icp_batch_dev with the tolerance stop.  Extra optional outputs: n_iter [nhyp] (pose updates
 * applied) and converged [nhyp] (1 = stopped by the tolerance).  A negative or NaN tolerance or a window outside [1, 16]
 * returns PCREG_ERR_ARG.  Results do not depend on the device count. */
int  pcreg_icp_batch_stop(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld,
                          const double* w_src, const double* T0_16, int64_t nhyp,
                          const pcreg_icp_opts* opts, const pcreg_icp_stop* stop,
                          double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx,
                          double* rmse_hist, int64_t* best, int32_t* n_iter, int32_t* converged);
int  pcreg_icp_batch_stop_dev(const pcreg_model* m, const double* d_src, int64_t ns,
                              const double* d_w_src, const double* d_T0_16, int64_t nhyp,
                              const pcreg_icp_opts* opts, const pcreg_icp_stop* stop,
                              double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status,
                              int32_t* d_idx, double* d_rmse_hist, int64_t* d_best,
                              int32_t* d_n_iter, int32_t* d_converged, void* stream);

/* ---- model normals and the point-to-plane metric --------------------------------------------------------------------
 * Point-to-point ICP converges only linearly on a smooth, locally planar surface (the CT/MRI models of this project are
 * meshes); point-to-plane converges in a few updates (Rusinkiewicz & Levoy 2001; Low 2004).  It needs one unit normal per
 * model point, uploaded or computed on the device.  Normals live with the model (every device replica has its own copy),
 * in original point order. */
/* nrm: n x 3 column-major (ld), float (is_double = 0) or double; each row is normalised in FP64 as
 * n / sqrt((nx*nx + ny*ny) + nz*nz).  A zero or non-finite row returns PCREG_ERR_ARG (and leaves the model's normals alone). */
int  pcreg_model_set_normals(pcreg_model* m, const void* nrm, int is_double, int64_t ld);
/* pcnormals(ptCloud, k) semantics, computed on the device; needs a model built with build_grid = 1 (else PCREG_ERR_ARG).
 * k in [3, 64] and at most the model size (pcnormals' default is 6).  The rule:
 *   neighbourhood  the k nearest model points of each model point, the point itself included (knnsearch semantics: exact FP64
 *                  squared distances, ties broken toward the smaller original index);
 *   normal         the eigenvector of the smallest eigenvalue of the unweighted covariance of those k points about their mean
 *                  (FP64, symmetric 3x3 Jacobi), normalised as in pcreg_model_set_normals;
 *   orientation    pcnormals documents none, so this library fixes one: with a viewpoint (double[3]) the normal is flipped so
 *                  that n . (viewpoint - p) >= 0; with viewpoint == NULL so that n . (p - c) >= 0, c = the centre of the
 *                  model's bounding box (outward on a closed star-shaped model).  The point-to-plane step does not depend on
 *                  the sign.
 * The toolbox is not available to compare against, so parity with pcnormals is UNPINNED. */
int  pcreg_model_compute_normals(pcreg_model* m, int k, const double* viewpoint);
/* out: n x 3 column-major doubles (ld = n).  PCREG_ERR_STATE when the model has no normals. */
int  pcreg_model_get_normals(const pcreg_model* m, double* out);

#define PCREG_ICP_POINT_TO_POINT 0
#define PCREG_ICP_POINT_TO_PLANE 1
/* Batched ICP with a choice of metric, plus the optional tolerance stop (stop == NULL: fixed iterations; n_iter and
 * converged are written only with a stop).  Correspondences, rejection, trimming, weights and rmse (Euclidean,
 * sqrt(sum w d^2 / sum w)) are those of pcreg_icp_batch; only the minimised metric and the pose update differ.
 * POINT_TO_POINT: the results equal pcreg_icp_batch / pcreg_icp_batch_stop bit for bit.
 * POINT_TO_PLANE (needs model normals, else PCREG_ERR_STATE): per pass, for every correspondence with weight w > 0, with
 * q = quickTF(src, T), m = model point, n = its normal and p = the model's pivot (bounding-box centre),
 *   q~ = q - p, m~ = m - p, a = (q~ x n, n) in R^6, b = (m~ - q~) . n;
 * A = sum w a a' and g = sum w a b are FP64 sums; A = L D L' (no pivoting, unknowns (omega, tau) in that order) solves
 * A x = g.  The update is degenerate (status 1, pose frozen as in pcreg_icp_batch) when fewer than 6 correspondences are
 * usable, sum w is not > 0, or any D_k <= 1e-12 max_k A_kk (a flat patch).  Otherwise
 *   R = I + (sin t / t) [omega]x + ((1 - cos t) / t^2) [omega]x^2, t = |omega| (R = I at t = 0),
 *   dT = [R' 0; p - p R' + tau, 1] (row-vector form) and T <- T dT.
 * An unknown metric returns PCREG_ERR_ARG.  Results do not depend on the device count. */
int  pcreg_icp_batch_metric(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld,
                            const double* w_src, const double* T0_16, int64_t nhyp,
                            const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                            double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx,
                            double* rmse_hist, int64_t* best, int32_t* n_iter, int32_t* converged);
int  pcreg_icp_batch_metric_dev(const pcreg_model* m, const double* d_src, int64_t ns,
                                const double* d_w_src, const double* d_T0_16, int64_t nhyp,
                                const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                                double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status,
                                int32_t* d_idx, double* d_rmse_hist, int64_t* d_best,
                                int32_t* d_n_iter, int32_t* d_converged, void* stream);

/* ---- plane-to-plane metric (generalized ICP; Segal, Haehnel & Thrun 2009) -------------------------------------------
 * Point-to-point treats the source as exact and point-to-plane uses only the model's surface; plane-to-plane models both clouds
 * as locally planar, which suits a noisy source (a stereo reconstruction) against a smooth model.  It needs model normals (else
 * PCREG_ERR_STATE) and one normal per source point.  Per pass, correspondences, rejection, trimming, weights and rmse (Euclidean,
 * sqrt(sum w d^2 / sum w)) are those of pcreg_icp_batch; only the minimised metric and the update differ.  With q = quickTF(s, T),
 * R the rotation block of T, p the model's pivot, for every correspondence (s, m) with w > 0:
 *   n_q = n_s R (the source normal carried with the point), n_m = the model normal of m,
 *   C = 2I - (1 - eps)(n_m n_m' + n_q n_q')  (the sum of the two plane covariances I - (1 - eps) n n'; eigenvalues in [2 eps, 2]),
 *   M = C^-1 = adj(C) / det(C) in FP64,  q~ = q - p, m~ = m - p, e = m~ - q~,  J' = [[q~]x; I] (6 x 3),
 *   A = sum w J' M J (FP64, upper triangle) and g = sum w J' M e = sum w (q~ x Me, Me).
 * With M = n n' this is the point-to-plane accumulation (J' n = (q~ x n, n) is its a).  The solve, the degenerate case and the update
 * are those of POINT_TO_PLANE (A x = g by L D L', status 1 and the pose frozen with fewer than 6 usable correspondences, sum w not
 * > 0 or a pivot <= 1e-12 max A_kk; Rodrigues, dT = [R' 0; p - p R' + tau, 1], T <- T dT).
 * Consequences: M depends on the normals only through n n', so flipping the sign of any source or model normal changes no bit of
 * the result; eps = 1 gives M = I/2, i.e. the Gauss-Newton linearised point-to-point step (not the Kabsch one).  This is ONE
 * Gauss-Newton step per correspondence pass with M frozen for that pass; Segal et al. run an inner optimiser instead.  eps = 1e-3
 * is their value and the usual default; an eps that is not finite or outside (0, 1] returns PCREG_ERR_ARG.  pcregistericp's
 * 'planeToPlane' documents no eps, so parity with the toolbox is UNPINNED.
 * src_nrm: ns x 3 column-major, same type and ld as src; each row is normalised in FP64 as pcreg_model_set_normals does, and a NULL
 * pointer or a zero or non-finite row returns PCREG_ERR_ARG (checked on the device before any ICP kernel runs).  stop is optional
 * and checked as in pcreg_icp_batch_stop (n_iter and converged are written only with a stop).  Results do not depend on the device
 * count: the host entry copies the source normals to every device. */
int  pcreg_icp_batch_gicp(const pcreg_model* m, const void* src, int is_double, int64_t ns, int64_t ld,
                          const double* w_src, const void* src_nrm, double eps,
                          const double* T0_16, int64_t nhyp, const pcreg_icp_opts* opts, const pcreg_icp_stop* stop,
                          double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx,
                          double* rmse_hist, int64_t* best, int32_t* n_iter, int32_t* converged);
/* d_src_nrm: float64 column-major, ld = ns, on the device; synchronous with respect to `stream` as pcreg_icp_batch_dev. */
int  pcreg_icp_batch_gicp_dev(const pcreg_model* m, const double* d_src, int64_t ns, const double* d_w_src,
                              const double* d_src_nrm, double eps,
                              const double* d_T0_16, int64_t nhyp, const pcreg_icp_opts* opts, const pcreg_icp_stop* stop,
                              double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx,
                              double* d_rmse_hist, int64_t* d_best, int32_t* d_n_iter, int32_t* d_converged, void* stream);

/* ---- many matching windows in one call ----------------------------------------------------------------------------------
 * The reference registers each matching window of a surface separately (slideMatchingWindow_v2.m:178-198 under parfor,
 * completeExperiment.m:265); pcreg_ransac_batch runs every window's RANSAC in one call, and this entry polishes every window's
 * hypotheses against that window's own source cloud in one call.  A call holds nwin >= 1 windows:
 *   window w has source rows src_offsets[w] .. src_offsets[w + 1] - 1 of src (ns_total x 3 column-major, ns_total =
 *   src_offsets[nwin], same type and ld for src_nrm), its own rows of w_src and src_nrm, and hypotheses hyp_offsets[w] ..
 *   hyp_offsets[w + 1] - 1 of T0_16 (hypotheses grouped by window, as in pcreg_ransac_batch);
 *   the model, opts, metric, gicp_eps and stop are shared.
 * Window w's results equal, bit for bit, what pcreg_icp_batch_metric (metric 0 or 1) / pcreg_icp_batch_gicp (metric 2) returns
 * for its rows, weights, normals and poses alone: T16, rmse, n_used, status, idx, rmse_hist, n_iter and converged.  Results do not
 * depend on the device count.
 * metric: PCREG_ICP_POINT_TO_POINT, _POINT_TO_PLANE or _PLANE_TO_PLANE; src_nrm (and gicp_eps) only with PLANE_TO_PLANE, ignored
 * otherwise.  stop optional (n_iter and converged are written only with a stop).  Per-hypothesis outputs are indexed by the global
 * hypothesis h; idx is ragged and window-major: window w's [H_w][ns_w] block (original source order relative to the window) starts at
 * sum_{v<w} H_v ns_v.  best [nwin]: per window, the first-index arg-min of rmse relative to the window, -1 when the window has no
 * hypothesis or all its rmse are NaN.
 * PCREG_ERR_ARG: null offsets, offsets[0] != 0 or decreasing offsets, nwin < 1, a window with hypotheses but no source rows, an unknown
 * metric, a bad eps or stop, a zero or non-finite source normal.  PCREG_ERR_STATE: metric 1 or 2 on a model without normals.
 * The batch runs as ONE launch of the fused per-hypothesis kernel when the model has a voxel map, opts.nn is the grid and the largest
 * window fits its shared memory (DESIGN.md section 3.3 gives the rule); otherwise, or with PCREG_FUSED=0, it loops over the windows
 * through the single-source path.  pcreg_last_profile then reports out[27] = 1 (fused) or 0 (loop: launches, times and counts summed
 * over the windows). */
#define PCREG_ICP_PLANE_TO_PLANE 2
int  pcreg_icp_batch_windows(const pcreg_model* m, const void* src, int is_double, int64_t ld, const int64_t* src_offsets,
                             const double* w_src, const void* src_nrm, double gicp_eps, const int64_t* hyp_offsets, int64_t nwin,
                             const double* T0_16, const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                             double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                             int64_t* best, int32_t* n_iter, int32_t* converged);
/* The same on device arrays (src, w_src, src_nrm float64 column-major with ld = ns_total), launched on `stream` and synchronous
 * with respect to it as pcreg_icp_batch_dev.  src_offsets and hyp_offsets are HOST arrays (the host sizes the launch from them);
 * d_best is a device int64[nwin]. */
int  pcreg_icp_batch_windows_dev(const pcreg_model* m, const double* d_src, const int64_t* src_offsets, const double* d_w_src,
                                 const double* d_src_nrm, double gicp_eps, const int64_t* hyp_offsets, int64_t nwin,
                                 const double* d_T0_16, const pcreg_icp_opts* opts, int metric, const pcreg_icp_stop* stop,
                                 double* d_T16, double* d_rmse, int32_t* d_n_used, int32_t* d_status, int32_t* d_idx,
                                 double* d_rmse_hist, int64_t* d_best, int32_t* d_n_iter, int32_t* d_converged, void* stream);

/* ---- pose extrapolation (accelerated ICP; Besl & McKay 1992, section IV; pcregistericp's 'Extrapolate') ------------------------
 * When the last updates of a hypothesis keep pointing the same way, the pose jumps further along that direction, by a step from a
 * line fit and a parabola fit of the error against the distance travelled.  Point-to-point only.  The rule (parity with the toolbox is
 * UNPINNED):
 *   c: the hypothesis's source centroid, the unweighted FP64 mean of its window's rows (one fixed-order device reduction per window).
 *   State of a pose T = [R 0; t 1]: x(T) = (qR, qT) in R^7, qR = the unit quaternion (w, x, y, z) of R (Shepperd's largest-diagonal
 *   branch), qT = c R + t (the image of the centroid: moving both clouds by a common rigid motion leaves the rule unchanged).  Sign of
 *   qR: for T_0 w >= 0 (at w = 0 the first nonzero component positive); for every later state the one with qR . qR_prev >= 0.
 *   d(T) = sum w |m - quickTF(s, T)|^2 / sum w over update u's correspondences and weights (the paper's d_k; a closed form of the
 *   update's 17 sums, centred so that a source far from the model's pivot loses no accuracy).
 *   Update u (1-based, not degenerate), K_u = T_{u-1} dT the Kabsch pose: Delta_u = x(K_u) - x_{u-1} (x_{u-1} the stored state),
 *   n_u = |Delta_u|, theta_u = acos(clamp(cos angle(Delta_{u-1}, Delta_u), -1, 1)) in degrees, undefined for u < 2 or a zero norm.
 *   It extrapolates when u >= 3 and theta_u, theta_{u-1} are both defined and < angle_deg: with v = (0, -n_u, -n_u - n_{u-1}) and
 *   D = (d(K_u), d_{u-1}, d_{u-2}), v1 = the zero of the least-squares line through (v_i, D_i), v2 = -b / (2a) the vertex of the
 *   parabola through them, vmax = vmax_scale n_u; dv = v2 if 0 < v2 < v1 < vmax or 0 < v2 < vmax < v1; v1 if 0 < v1 < v2 < vmax,
 *   0 < v1 < vmax < v2 or (v2 < 0 and 0 < v1 < vmax); vmax if v1 > vmax and v2 > vmax; else 0 (strict compares, NaN fails each).
 *   With dv > 0: x' = x(K_u) + dv Delta_u / n_u, qR' renormalised, T_u = [R(qR') 0; qT' - c R' 1]; otherwise T_u = K_u.
 *   Stored: x_u = x' or x(K_u), d_u = d(T_u), Delta_u and n_u as before the jump; n_extrap counts the updates with dv > 0.
 *   An update whose K_u or T_{u-1} is improper (reflection_fix = 0 on data that prefer a reflection) has no quaternion state: it is
 *   not extrapolated (T_u = K_u, nothing stored) and the history restarts: the next update whose K_u and T_{u-1} are both proper
 *   takes T_{u-1} as update 1 takes T_0 (canonical sign, no direction yet).  So a returned pose has the handedness of its Kabsch pose.
 * Correspondences, rejection, trimming, weights, rmse, the degenerate freeze and the winner are unchanged.  The tolerance stop
 * measures the motion from T_{u-1} to the pose written, T_u.  The rule is causal: a hypothesis stopped after k updates returns exactly
 * what the same call with iters = k returns.  Defaults {10, 25} are the paper's; angle_deg outside (0, 180] or a vmax_scale that is not
 * finite and > 0 returns PCREG_ERR_ARG. */
typedef struct {
    double angle_deg;       /* both of the last two direction changes below this: extrapolate  */
    double vmax_scale;      /* the step is at most vmax_scale n_u                              */
} pcreg_icp_extrap;
void pcreg_icp_extrap_default(pcreg_icp_extrap* e);   /* {10, 25} */
/* Point-to-point batched ICP with pose extrapolation, in the windows layout of pcreg_icp_batch_windows (nwin = 1: one source for every
 * hypothesis; arguments, outputs, errors and sharding over the devices as there, metric 0).  stop is optional; ex == NULL returns the
 * bits of pcreg_icp_batch_windows with metric 0.  n_extrap [nhyp] (optional, written only with ex): updates extrapolated. */
int  pcreg_icp_batch_extrap(const pcreg_model* m, const void* src, int is_double, int64_t ld, const int64_t* src_offsets,
                            const double* w_src, const int64_t* hyp_offsets, int64_t nwin, const double* T0_16,
                            const pcreg_icp_opts* opts, const pcreg_icp_stop* stop, const pcreg_icp_extrap* ex,
                            double* T16, double* rmse, int32_t* n_used, int32_t* status, int32_t* idx, double* rmse_hist,
                            int64_t* best, int32_t* n_iter, int32_t* converged, int32_t* n_extrap);
/* The same on device arrays, synchronous with respect to `stream` as pcreg_icp_batch_windows_dev (offsets on the host). */
int  pcreg_icp_batch_extrap_dev(const pcreg_model* m, const double* d_src, const int64_t* src_offsets, const double* d_w_src,
                                const int64_t* hyp_offsets, int64_t nwin, const double* d_T0_16, const pcreg_icp_opts* opts,
                                const pcreg_icp_stop* stop, const pcreg_icp_extrap* ex, double* d_T16, double* d_rmse,
                                int32_t* d_n_used, int32_t* d_status, int32_t* d_idx, double* d_rmse_hist, int64_t* d_best,
                                int32_t* d_n_iter, int32_t* d_converged, int32_t* d_n_extrap, void* stream);

/* Timing / accounting of the most recent pcreg_icp_batch{,_dev,_stop,_stop_dev,_metric,_metric_dev,_gicp,_gicp_dev,_windows,_windows_dev,_extrap,_extrap_dev} or pcreg_nn_search call,
 * measured with CUDA events on the launching stream (bench.py's roofline numbers):
 *   out[0] = NN kernel launches, out[1] = total NN kernel ms, out[2] = NN queries (with the tolerance stop: the queries of
 *   the passes each hypothesis ran, except on the brute-force and map-less grid paths, which still search for stopped
 *   hypotheses and count every pass),
 *   out[3] = (query, model point) pairs evaluated by brute force,
 *   out[4] = update (select + 17-sum + Kabsch) kernel launches, out[5] = their total ms,
 *   out[6] = correspondences reduced (tolerance stop: of the passes run);
 *   grid NN, exact device-side counts: out[7] = model points / out[8] = cell rows visited by the row scan,
 *   out[9] = pyramid nodes popped, out[10] = queries answered from their candidate list, out[11] = queries walked,
 *   out[12] = queries row-scanned, out[13] = list entries read, out[14] = list points gathered,
 *   out[15] = model points / out[16] = leaf cells visited by the walk;
 *   out[17..19] = total ms and out[20..22] = launches of the list-scan / row-scan / walk kernels,
 *   out[23] = queries whose search was skipped by lazy trimming (they are included in out[10]);
 *   after pcreg_get_matches: out[24] = total ms of the score kernel, out[25] = (pair, dimension) terms it evaluated;
 *   after pcreg_align_points: out[24] = ms of the alignment kernel, out[25] = points it processed;
 *   out[26] = 1 when the grid NN ran on the model's Voronoi voxel map: then out[10] = queries answered by the voxel list
 *   scan, out[13] = list entries read, out[14] = points gathered for the FP64 decision, out[17] / out[20] = ms / launches
 *   of the list-scan kernel, and out[11], out[15], out[16], out[9], out[19] describe the pyramid walk of the rest.
 *   out[27] = 1 when the whole ICP ran as the fused per-hypothesis kernel (one launch; out[1] = out[17] = its ms);
 *   out[28..31] = share of a block's cycles in its four phases (NN, trim selection, 17 sums + reduction, pose update).
 * Collected only when enabled: the counters add atomics to the kernels, so timed runs keep it off.
 * enabled = 1: event times + work counters; 2: event times only (kernel times undisturbed by the counter atomics). */
int  pcreg_set_profiling(int enabled);
int  pcreg_last_profile(double out[32]);

#ifdef __cplusplus
}
#endif
#endif /* PCREG_H */
