// pcreg_internal.h -- host-side state shared by the translation units of libpcreg_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string>
#include <vector>
#include <memory>
#include <new>
#include <exception>

#include "../../include/pcreg.h"

namespace pcreg {

// ---- error plumbing --------------------------------------------------------------------------
void set_error(const char* fmt, ...);
struct CudaFail { cudaError_t e; const char* what; const char* file; int line; };

#define PCREG_CUDA(call)                                                                      \
    do {                                                                                      \
        cudaError_t _e = (call);                                                              \
        if (_e != cudaSuccess) throw ::pcreg::CudaFail{_e, #call, __FILE__, __LINE__};        \
    } while (0)

// Bumps the launch counter and checks the launch error (no sync).
void count_launch(int n = 1);
#define PCREG_LAUNCHED()                                                                      \
    do {                                                                                      \
        ::pcreg::count_launch();                                                              \
        PCREG_CUDA(cudaGetLastError());                                                       \
    } while (0)

struct ArgError { std::string msg; };
#define PCREG_REQUIRE(cond, msg)                                                              \
    do { if (!(cond)) throw ::pcreg::ArgError{msg}; } while (0)
struct StateError { std::string msg; };     // the handle lacks what the call needs (PCREG_ERR_STATE)

// Every extern "C" body is wrapped in these: no C++ exception crosses the ABI.
#define PCREG_API_BEGIN try {
#define PCREG_API_END                                                                                         \
    }                                                                                                         \
    catch (const ::pcreg::CudaFail& f) {                                                                      \
        ::pcreg::set_error("CUDA error %d (%s) in %s at %s:%d", (int)f.e, cudaGetErrorString(f.e), f.what, f.file, f.line); \
        cudaGetLastError();                                                                                   \
        return PCREG_ERR_CUDA;                                                                                \
    }                                                                                                         \
    catch (const ::pcreg::ArgError& a) { ::pcreg::set_error("%s", a.msg.c_str()); return PCREG_ERR_ARG; }     \
    catch (const ::pcreg::StateError& a) { ::pcreg::set_error("%s", a.msg.c_str()); return PCREG_ERR_STATE; } \
    catch (const std::bad_alloc&) { ::pcreg::set_error("host allocation failed"); return PCREG_ERR_ALLOC; }   \
    catch (...) { ::pcreg::set_error("unknown C++ exception"); return PCREG_ERR_STATE; }

// Runs f on the calling thread and maps the library's exceptions to a status code (worker threads of the multi-device
// entry points: no exception may leave a std::thread).
template <typename F>
int guarded(F&& f) {
    PCREG_API_BEGIN
    f();
    return PCREG_OK;
    PCREG_API_END
}

// ---- library context: one per selected device ("slot" k = the k-th device handed to pcreg_init) ------
// Host threads pick their slot with use_slot(); the thread that called pcreg_init works on slot 0, the
// multi-device entry points (pcreg_icp_batch, pcreg_ransac_batch) run one worker thread per slot.
constexpr int PCREG_MAX_DEVICES = 16;
struct PoolBlock { void* p; size_t bytes; bool used; };
struct Context {
    bool initialised = false;
    int  slot = 0;
    int  device = 0;
    int  sm_count = 148;
    size_t smem_optin = 0;
    size_t total_mem = 0;                // device memory, bytes
    bool profiling = false;
    bool profiling_counters = true;      // pcreg_set_profiling(2): event times only (the counters add atomics to the kernels)
    double profile[32] = {0};
    std::vector<cudaEvent_t> events;     // reusable timing events (profiling mode)
    std::vector<cudaStream_t> streams;   // internal streams of the two-lane ICP loop
    void* pinned[2] = {nullptr, nullptr};   // bounce buffers of h2d_columns (allocated on first use)
    cudaEvent_t pinned_ev[2] = {nullptr, nullptr};
    std::vector<PoolBlock> pool;            // caching device allocator of this device
};
int  num_slots();                        // devices selected by pcreg_init
void use_slot(int slot);                 // bind the calling host thread to a slot (+ cudaSetDevice)
int  current_slot();
cudaEvent_t pooled_event(size_t i);      // i-th reusable event, created on first use
cudaStream_t lane_stream(int i);         // i-th internal stream (non-blocking), created on first use
Context& ctx();
void require_init();

// Caching device allocator: cudaMalloc / cudaFree cost milliseconds for the half-gigabyte scratch a
// batch needs, so released blocks are kept and reused (best fit within 2x).  Blocks are only ever
// released after the stream that used them has been synchronised.
void* pool_alloc(size_t bytes);
void pool_free(void* p);
void pool_trim(size_t keep_bytes);

// RAII device buffer on the caching allocator.
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    explicit DevBuf(size_t count) { alloc(count); }
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; } return *this; }
    ~DevBuf() { release(); }
    void alloc(size_t count) {
        release();
        n = count;
        if (count == 0) return;
        p = (T*)pool_alloc(count * sizeof(T));
    }
    // On an error path (stack unwinding) kernels queued before the throw may still use the buffer: drain the device before
    // the block goes back to the pool, so that the next call cannot be handed memory that is still being written.
    void release() {
        if (p) {
            if (std::uncaught_exceptions() > 0) cudaDeviceSynchronize();
            pool_free(p);
        }
        p = nullptr; n = 0;
    }
    size_t bytes() const { return n * sizeof(T); }
};

// ---- model handle --------------------------------------------------------------------------------
// Level-0 sorted point record of the grid: one 32-byte sector per point.
struct __align__(32) GridPoint { double x, y, z; int32_t orig; int32_t pad; };
struct __align__(32) ModelPointD { double x, y, z, pad; };

constexpr int GRID_MAX_LEVELS = 12;

struct GridView {               // passed by value to kernels
    const GridPoint* pts;       // sorted by level-0 cell
    const int32_t* cell_start;  // [ncell0 + 1]
    const uint8_t* mask[GRID_MAX_LEVELS];   // mask[l], l >= 1: 8-bit child occupancy of level-l cells
    int32_t dims[GRID_MAX_LEVELS][3];       // dims[l] of level l (level 0 = fine cells)
    int32_t nlevels;            // root is level nlevels-1 (dims 1x1x1)
    double origin[3];
    double cell;                // level-0 edge
    double inv_cell;
};

// Candidate ("Verlet") lists of the grid NN path, one per query of the current hypothesis chunk: every model
// point within R_list = r0 + skin of the position q0 the query had when its list was built.  A later ICP pass
// scans the list and accepts the result when (best list distance) + |q - q0| < R_list (nn_grid.cu).
struct CandView {               // passed by value to kernels
    float4* hdr;                // [nq] (q0 - grid origin) in FP32, w = R_list (rounded down)
    int2* cnt;                  // [nq] x = list length (-1 = no list), y = float bits of the level scale's lower end.  nullptr: disabled
    int32_t* list;              // [nq][cap] (position into GridView::pts) << 8 | distance level at build time
    float inv_level;            // 255 / (2 skin): levels per model unit
    int32_t cap;
    int32_t* ext;               // [nq] extension slot of the query (-1: none): entries cap.. of long lists
    int32_t* ext_list;          // [ext_slots][ext_cap]
    unsigned int* ext_count;    // slots handed out so far
    int32_t ext_cap, ext_slots;
    float gap_cells;            // a building search is exhaustive within (best distance + gap), in cell units
    double skin;                // model units, <= gap_cells * cell: margin of the list around the best distance
    const float* delta;         // [nhyp] or null: displacement bound of the last pose update (build only when small)
    float build_max_delta;
};

// Voronoi voxel map (nn_vox.cu): for every voxel of a uniform grid over the padded model bounding box, a
// conservative superset of the model points that are the nearest neighbour of SOME location inside the voxel.
// A query reads the short list of its voxel (FP32 offsets from the voxel centre, contiguous) and decides in FP64.
struct VoxView {                // passed by value to kernels
    const float4* ent;          // entries: (p - voxel centre) rounded to FP32, w = bits of the int32 position into GridView::pts
    const uint2* hdr;           // [brick-ordered voxels] x = first entry, y = entries (0: no list -> pyramid walk)
    int32_t dims[3];            // voxels per axis
    int32_t tiles[3];           // 4 x 4 x 4 bricks per axis (storage order of hdr)
    double origin[3];           // lower corner of voxel (0,0,0)
    double s, inv_s;            // voxel edge
    float band_abs;             // absolute term of the FP32 error band of the list scan
};

}  // namespace pcreg

struct pcreg_model {
    int slot = 0;               // device slot this copy lives on
    std::vector<pcreg_model*> replicas;     // slot-0 handle only: the copies on slots 1.. (replicas[k-1] = slot k)
    const pcreg_model* on_slot(int k) const { return k == 0 ? this : replicas[(size_t)k - 1]; }
    int64_t n = 0;              // points
    int64_t n_pad = 0;          // padded to a multiple of the brute tile
    double pivot[3] = {0, 0, 0};        // subtracted before the FP32 conversion and before the 17 sums
    double bbox_lo[3] = {0, 0, 0}, bbox_hi[3] = {0, 0, 0};
    float  max_norm = 0.f;      // max |m32| over the model (FP32 error bound of the brute scan)
    pcreg::DevBuf<float4> m4;               // shuffled scan order: (x,y,z relative to pivot, |.|^2)
    pcreg::DevBuf<int32_t> perm;            // perm[scan position] = original index
    pcreg::DevBuf<pcreg::ModelPointD> md;   // original order, FP64
    pcreg::DevBuf<pcreg::ModelPointD> nrm;  // unit normals {nx, ny, nz, 0}, original order (empty: none; point-to-plane ICP)
    // grid
    bool has_grid = false;
    pcreg::GridView grid{};
    pcreg::DevBuf<pcreg::GridPoint> g_pts;
    pcreg::DevBuf<int32_t> g_cell_start;
    std::vector<pcreg::DevBuf<uint8_t>> g_masks;
    int64_t g_occupied = 0;
    // Voronoi voxel map (built on top of the grid's sorted point array)
    bool has_vox = false;
    pcreg::VoxView vox{};
    pcreg::DevBuf<float4> v_ent;
    pcreg::DevBuf<uint2> v_hdr;
    int64_t v_voxels = 0, v_listed = 0, v_entries = 0, v_too_long = 0, v_no_room = 0, v_max_len = 0;
    double v_build_ms = 0.0;
    int64_t v_far = 0;          // voxels outside the band (band-limited map)
    double v_band = 0.0;
};

namespace pcreg {

// ---- internal launchers (implemented in the .cu files) ---------------------------------------------
constexpr int BRUTE_TILE = 1024;            // model points per shared-memory tile (16 KB as float4)

// Per-call scratch of the brute path (partial results of the model splits); grows on demand.
struct NNScratch {
    DevBuf<double> pd2;      // [nsplit][nq]
    DevBuf<int32_t> pidx;    // [nsplit][nq]
    DevBuf<float> pmin;      // [nsplit0][nq] sub-sample bound pass
};

// Nearest neighbour of quickTF(src_i, T_h) for every (h, i): exact FP64 decision.
//   d_T   : [nhyp][16] row-major row-vector poses (device)
//   prev  : optional [nhyp*ns] previous correspondences (warm start), may be nullptr
//   out   : idx [nhyp*ns], d2 [nhyp*ns]
void nn_brute_launch(const pcreg_model* m, const double* d_sx, const double* d_sy, const double* d_sz,
                     int64_t ns, const double* d_T, int64_t nhyp, const int32_t* d_prev,
                     int32_t* d_idx, double* d_d2, NNScratch& scratch, cudaStream_t st);
// Per-call scratch of the grid path: the work list handed from the direct kernel to the walk kernel.
struct GridScratch {
    DevBuf<int32_t> worklist;       // [nq] direct -> walk
    DevBuf<int32_t> worklist0;      // [nq] list scan -> direct
    DevBuf<unsigned int> count;     // [2]
    DevBuf<unsigned long long> cursor;   // [1] chunk cursor of the row-scan kernel
    // profiling: event marks between the kernels of a pass (kind 0 = list scan starts, 1 = row scan starts,
    // 2 = walk starts, 3 = pass ends); events are drawn from the pool through the caller's cursor
    struct Mark { int kind; cudaEvent_t ev; };
    std::vector<Mark>* timing = nullptr;
    size_t* ev_cursor = nullptr;
};
// cl: candidate lists of this chunk or nullptr; scan_lists: lists may exist (a build pass has run)
void nn_grid_launch(const pcreg_model* m, const double* d_sx, const double* d_sy, const double* d_sz,
                    int64_t ns, const double* d_T, int64_t nhyp, const int32_t* d_prev,
                    int32_t* d_idx, double* d_d2, unsigned long long* d_visit_counters, GridScratch& scratch,
                    const CandView* cl, bool scan_lists, const double* d_skip_thr /*[nhyp] or null: lazy trimming*/, cudaStream_t st,
                    const int32_t* d_stop_iter = nullptr /*[nhyp] or null: voxel-map path skips hypotheses with stop_iter >= 0*/);

// Tolerance stop of the ICP loop (pcreg_icp_stop; the rule is icp_stop_update in pcreg_icp.cuh)
constexpr int ICP_STOP_WINDOW_MAX = 16;
struct IcpStopRule { double tol_t, tol_r_deg; int window; };
// Pose extrapolation of the point-to-point loop (pcreg_icp_extrap; the rule is extrap_step in pcreg_math.cuh)
struct IcpExtrapRule { double angle_deg, vmax_scale; };

// Outputs of the covariance pass (pcreg_icp_covariance; the ICP_M_COV kernels, selected by cov != nullptr), indexed by the
// hypothesis of the launch; null pointers in every other call.
struct IcpCovOut {
    double* cov;                // [nhyp][36] row-major, about ref
    double* info;               // [nhyp][36] or null
    double* sigma2;             // [nhyp]
    int32_t* status;            // [nhyp] 1: degenerate (cov and tre NaN)
    double* tre;                // [nhyp][ntarget] or null
    const double* targets;      // [3][ntarget] column-major model-frame points, device
    int32_t ntarget;
    double ref[3];
};
// the same outputs from hypothesis h0 on (a chunk or a window of the launch)
inline IcpCovOut cov_out_at(const IcpCovOut& c, int64_t h0) {
    IcpCovOut o = c;
    o.cov += h0 * 36; o.sigma2 += h0; o.status += h0;
    if (o.info) o.info += h0 * 36;
    if (o.tre) o.tre += h0 * o.ntarget;
    return o;
}

// Select / weight / 17 sums / Kabsch / compose, one block per hypothesis.
struct IcpUpdateArgs {
    const pcreg::ModelPointD* md;
    double pivot[3];
    const double* sx; const double* sy; const double* sz; const double* w_src;
    int64_t ns;
    double* T;                  // [nhyp][16] row-major, updated in place when `update`
    const int32_t* idx; const double* d2;
    unsigned long long* keys;   // [nhyp*ns] scratch (KNN mode)
    const int32_t* tie_order;   // [ns] or null: tie_order[original index] = position in the (sorted) source arrays
    float* delta;               // [nhyp] or null: out, upper bound of the displacement of any source point by this update
    const double* src_stats;    // [4] centroid + radius of the source cloud (for delta)
    double* skip_thr;           // [nhyp] or null: out, residual above which a query cannot be selected in the next pass
    int mode; double k_frac; double R_w; double thDist2; int reflection_fix;
    int update;                 // 1: apply the pose update; 0: score only (final pass)
    int32_t* frozen;            // [nhyp] status flags (1 = frozen)
    double* rmse; int32_t* n_used;        // [nhyp] written every pass
    double* rmse_hist; int hist_stride; int hist_col;   // optional; hist_col is also the pass index
    // tolerance stop (stop_iter == nullptr: none, the k_icp_update<*, false> instantiations).  An intermediate pass leaves a
    // stopped hypothesis alone; the final pass scores it and fills its history from the column its own final pass would have had.
    int32_t* stop_iter;         // [nhyp] updates applied when the hypothesis stopped (converged or frozen), -1 while it runs
    double* stop_ring;          // [nhyp][2 * ICP_STOP_WINDOW_MAX] motion of the last `window` updates
    IcpStopRule stop;
    int32_t* n_iter; int32_t* converged;   // [nhyp] optional, written by the final pass
    const pcreg::ModelPointD* nrm;         // model normals (original order): the point-to-plane metric (k_icp_update<*, *, 1>)
    // plane-to-plane metric (k_icp_update<*, *, 2>; null otherwise): unit source normals in the order of sx / sy / sz, covariance epsilon
    const double* snx; const double* sny; const double* snz; double gicp_eps;
    // pose extrapolation (ex_state == nullptr: none; else the k_icp_update<*, 2, 0> instantiations, which need stop_iter as well)
    IcpExtrapRule ex;
    double* ex_state;           // [nhyp][EXTRAP_STATE], zero before the first pass
    const double* ex_cen;       // [3] source centroid
    int32_t* n_extrap;          // [nhyp] optional, written by the final pass
    IcpCovOut cov;              // the covariance pass (k_icp_update<*, 0, 3>; cov.cov null otherwise)
};
void icp_update_launch(const IcpUpdateArgs& a, int64_t nhyp, cudaStream_t st);
// d_seg (optional, device [nseg + 1]): one arg-min per segment of the rmse array, each relative to its segment
void icp_argmin_launch(const double* d_rmse, int64_t nhyp, int64_t* d_best, cudaStream_t st, const int64_t* d_seg = nullptr, int64_t nseg = 1);

// getLocalPoints.m batched over centres with the neighbourhoods left on the device (local_points.cu)
struct LocalPointsDev {
    std::vector<int64_t> counts, offsets;       // per centre: sphere count; rows offsets[k]..offsets[k+1]-1 (empty if rejected)
    std::vector<int32_t> status;                // 1 where getLocalPoints returns []
    DevBuf<double> pts;                         // [3][nel] points relative to their centre, original model order
    DevBuf<int64_t> d_offsets;                  // offsets on the device
    int64_t ntotal = 0, nel = 1;
};
void local_points_device(const pcreg_model* m, const double* centres, int64_t nc, int64_t ld, double R, int64_t min_points,
                         int64_t max_points, LocalPointsDev& out, cudaStream_t st);

void grid_build(pcreg_model* m, const pcreg_model_opts& o, cudaStream_t st);
// Voronoi voxel map on top of the grid (nn_vox.cu); leaves m->has_vox false when the model is too dense for the budget
void vox_build(pcreg_model* m, const pcreg_model_opts& o, cudaStream_t st);
struct GridArgs;
// list scan of every query's voxel; queries without a list are appended to a.worklist (then walked by nn_grid.cu)
void nn_vox_launch(const pcreg_model* m, const GridArgs& a, cudaStream_t st);
// Upload of a column-major host matrix (ncols columns of `rows` doubles, column stride ld_src) from PAGEABLE memory
// into a device matrix with column stride ld_dst: columns are packed into two alternating pinned bounce buffers and
// sent asynchronously, so the host-side packing of one chunk overlaps the DMA of the previous one (a plain
// cudaMemcpy2D from pageable memory stages row by row at ~2 GB/s).  Returns after the last chunk is queued on st.
void h2d_columns(double* d_dst, int64_t ld_dst, const double* h_src, int64_t ld_src, int64_t rows, int64_t ncols, cudaStream_t st);
// MATLAB column-major 4x4 <-> internal row-major 4x4, batched (a transpose either way)
void transpose16_launch(const double* d_in, double* d_out, int64_t n, cudaStream_t st);

}  // namespace pcreg
