// normals.cu -- unit normals of the model cloud (include/pcreg.h: pcreg_model_set_normals / _compute_normals / _get_normals),
// the input of the point-to-plane ICP metric.
//
// pcnormals(ptCloud, k) semantics on the device: the k nearest model points of every model point (the point itself included),
// the covariance of that neighbourhood about its mean, the eigenvector of its smallest eigenvalue.  The neighbourhood is exact
// (knnsearch: FP64 squared distances in dist2_exact's order, ties toward the smaller original index), found by the
// branch-and-bound walk of the occupancy pyramid (walk_search, pcreg_grid.cuh) with a sorted k-best list in place of the one best
// candidate and the k-th distance as the pruning bound.  One thread per model point, the points taken in grid (cell) order so
// that the walks of a warp stay in one region.  The Voronoi voxel map answers only k = 1 and is not used here.
#include <math.h>
#include <float.h>
#include <vector>
#include <thread>

#include "pcreg_internal.h"
#include "pcreg_dev.cuh"
#include "pcreg_grid.cuh"
#include "pcreg_math.cuh"

namespace pcreg {

constexpr int NRM_KMAX = 64;
constexpr int NRM_THREADS = 128;

// the k nearest model points of grid point t (sorted by (d2, original index)) -> covariance -> normal -> out[orig]
__global__ void __launch_bounds__(NRM_THREADS) k_model_normals(const GridView G, int64_t n, int k, int has_vp, double vx, double vy,
                                                                double vz, double cx, double cy, double cz, ModelPointD* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * NRM_THREADS + threadIdx.x;
    if (t >= n) return;
    const GridPoint self = G.pts[t];
    const double qx = self.x, qy = self.y, qz = self.z;
    const float fx = __double2float_rn((qx - G.origin[0]) * G.inv_cell);
    const float fy = __double2float_rn((qy - G.origin[1]) * G.inv_cell);
    const float fz = __double2float_rn((qz - G.origin[2]) * G.inv_cell);
    const double inv_cell2 = G.inv_cell * G.inv_cell;
    double kd[NRM_KMAX];
    int32_t ko[NRM_KMAX], kp[NRM_KMAX];     // original index (the tie rule) and position in G.pts of each list entry
    int cnt = 0;
    float bound = FLT_MAX;                  // k-th distance in squared cell units, rounded up (FLT_MAX until the list is full)

    unsigned long long stack[GRID_STACK];
    int sp = 0;
    stack[sp++] = pack_entry(0.f, G.nlevels - 1, 0, 0, 0);
    while (sp > 0) {
        const unsigned long long e = stack[--sp];
        const float lbf = __uint_as_float((unsigned)(e >> 34) << 1);
        if (lbf > bound) continue;
        const unsigned lo32 = (unsigned)e;
        const int level = (int)((e >> 30) & 0xF);
        const int ix = (int)(lo32 & 1023u), iy = (int)((lo32 >> 10) & 1023u), iz = (int)((lo32 >> 20) & 1023u);
        if (level == 0) {
            const int64_t c = ((int64_t)iz * G.dims[0][1] + iy) * G.dims[0][0] + ix;
            const int32_t s0 = G.cell_start[c], s1 = G.cell_start[c + 1];
            bool changed = false;
            for (int32_t p = s0; p < s1; ++p) {
                const GridPoint gp = G.pts[p];
                const double d = dist2_exact(gp.x, gp.y, gp.z, qx, qy, qz);
                if (cnt == k && !(d < kd[k - 1] || (d == kd[k - 1] && gp.orig < ko[k - 1]))) continue;
                int j = cnt < k ? cnt : k - 1;           // insertion into the sorted list, the last entry drops out when full
                while (j > 0 && (kd[j - 1] > d || (kd[j - 1] == d && ko[j - 1] > gp.orig))) {
                    kd[j] = kd[j - 1]; ko[j] = ko[j - 1]; kp[j] = kp[j - 1];
                    --j;
                }
                kd[j] = d; ko[j] = gp.orig; kp[j] = p;
                if (cnt < k) ++cnt;
                changed = true;
            }
            if (changed && cnt == k) bound = best_ub_cells(kd[k - 1], inv_cell2);
            continue;
        }
        const int64_t c = ((int64_t)iz * G.dims[level][1] + iy) * G.dims[level][0] + ix;
        unsigned m = G.mask[level][c];
        const float edge = (float)(1 << (level - 1));
        const float bx = (float)(2 * ix) * edge, by = (float)(2 * iy) * edge, bz = (float)(2 * iz) * edge;
        float ax0 = axis_lb(fx, bx, edge), ax1 = axis_lb(fx, bx + edge, edge);
        float ay0 = axis_lb(fy, by, edge), ay1 = axis_lb(fy, by + edge, edge);
        float az0 = axis_lb(fz, bz, edge), az1 = axis_lb(fz, bz + edge, edge);
        ax0 *= ax0; ax1 *= ax1; ay0 *= ay0; ay1 *= ay1; az0 *= az0; az1 *= az1;
        const unsigned oct = (fx >= bx + edge ? 1u : 0u) | (fy >= by + edge ? 2u : 0u) | (fz >= bz + edge ? 4u : 0u);
        if (oct & 1u) m = ((m & 0xAAu) >> 1) | ((m & 0x55u) << 1);
        if (oct & 2u) m = ((m & 0xCCu) >> 2) | ((m & 0x33u) << 2);
        if (oct & 4u) m = ((m & 0xF0u) >> 4) | ((m & 0x0Fu) << 4);
        while (m) {
            const int tt = 31 - __clz(m);                          // far first, so the near octant is popped first
            m &= ~(1u << tt);
            const int kk = tt ^ (int)oct;
            const float lb = ((((kk & 1) ? ax1 : ax0) + ((kk & 2) ? ay1 : ay0)) + ((kk & 4) ? az1 : az0)) * (1.f - 6e-7f);
            if (lb <= bound) {
                if (sp >= GRID_STACK) __trap();            // unreachable (static_assert in pcreg_grid.cuh): never drop a node silently
                stack[sp++] = pack_entry(lb, level - 1, 2 * ix + (kk & 1), 2 * iy + ((kk >> 1) & 1), 2 * iz + (kk >> 2));
            }
        }
    }

    // unweighted covariance of the neighbourhood about its mean (list order), smallest eigenpair
    double mx = 0.0, my = 0.0, mz = 0.0;
    for (int j = 0; j < cnt; ++j) { const GridPoint gp = G.pts[kp[j]]; mx += gp.x; my += gp.y; mz += gp.z; }
    mx /= (double)cnt; my /= (double)cnt; mz /= (double)cnt;
    double C[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = 0; j < cnt; ++j) {
        const GridPoint gp = G.pts[kp[j]];
        const double dx = gp.x - mx, dy = gp.y - my, dz = gp.z - mz;
        C[0] += dx * dx; C[1] += dx * dy; C[2] += dx * dz;
        C[4] += dy * dy; C[5] += dy * dz; C[8] += dz * dz;
    }
    C[3] = C[1]; C[6] = C[2]; C[7] = C[5];
    double w[3], V[9];
    eigsym3(C, w, V);
    eigsort3(w, V, +1);
    double nx = V[0], ny = V[3], nz = V[6];
    const double nr = sqrt((nx * nx + ny * ny) + nz * nz);
    nx /= nr; ny /= nr; nz /= nr;
    const double dot = has_vp ? nx * (vx - qx) + ny * (vy - qy) + nz * (vz - qz) : nx * (qx - cx) + ny * (qy - cy) + nz * (qz - cz);
    if (dot < 0.0) { nx = -nx; ny = -ny; nz = -nz; }
    ModelPointD o;
    o.x = nx; o.y = ny; o.z = nz; o.pad = 0.0;
    out[self.orig] = o;
}

// the same normals on every device replica of the model: slot 0 keeps `d0` (already on it) or receives `h`, the other slots
// receive `h` (host copy, original order).  Returns the first failing slot's status.
static int store_normals(pcreg_model* m, DevBuf<ModelPointD>* d0, const std::vector<ModelPointD>& h) {
    const int nrep = (int)m->replicas.size();
    std::vector<int> rc((size_t)nrep + 1, PCREG_OK);
    auto upload = [&](int k) {
        pcreg_model* r = const_cast<pcreg_model*>(m->on_slot(k));
        DevBuf<ModelPointD> buf((size_t)r->n);
        PCREG_CUDA(cudaMemcpyAsync(buf.p, h.data(), buf.bytes(), cudaMemcpyHostToDevice, 0));
        PCREG_CUDA(cudaStreamSynchronize(0));
        r->nrm = std::move(buf);
    };
    std::vector<std::thread> workers;
    for (int k = 1; k <= nrep; ++k) workers.emplace_back([&, k]() { rc[k] = guarded([&]() { use_slot(k); upload(k); }); });
    rc[0] = guarded([&]() {
        use_slot(0);
        if (d0) m->nrm = std::move(*d0);
        else upload(0);
    });
    for (auto& w : workers) w.join();
    use_slot(0);
    for (int r : rc) if (r != PCREG_OK) return r;
    return PCREG_OK;
}

}  // namespace pcreg

using namespace pcreg;

extern "C" {

int pcreg_model_set_normals(pcreg_model* m, const void* nrm, int is_double, int64_t ld) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(m && nrm, "pcreg_model_set_normals: null pointer");
    PCREG_REQUIRE(ld >= m->n, "pcreg_model_set_normals: ld must be >= the model size");
    std::vector<ModelPointD> h((size_t)m->n);
    for (int64_t i = 0; i < m->n; ++i) {
        double v[3];
        for (int a = 0; a < 3; ++a) v[a] = is_double ? ((const double*)nrm)[a * ld + i] : (double)((const float*)nrm)[a * ld + i];
        const double r = sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
        PCREG_REQUIRE(std::isfinite(r) && r > 0.0, "pcreg_model_set_normals: zero or non-finite normal");
        h[i].x = v[0] / r; h[i].y = v[1] / r; h[i].z = v[2] / r; h[i].pad = 0.0;
    }
    return store_normals(m, nullptr, h);
    PCREG_API_END
}

int pcreg_model_compute_normals(pcreg_model* m, int k, const double* viewpoint) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(m, "pcreg_model_compute_normals: null pointer");
    PCREG_REQUIRE(m->has_grid, "pcreg_model_compute_normals: the model has no grid (create it with build_grid = 1)");
    PCREG_REQUIRE(k >= 3 && k <= NRM_KMAX, "pcreg_model_compute_normals: k must be in [3, 64]");
    PCREG_REQUIRE(k <= m->n, "pcreg_model_compute_normals: k exceeds the number of model points");
    use_slot(0);
    cudaStream_t st = 0;
    DevBuf<ModelPointD> d((size_t)m->n);
    const double* vp = viewpoint;
    k_model_normals<<<(unsigned)((m->n + NRM_THREADS - 1) / NRM_THREADS), NRM_THREADS, 0, st>>>(
        m->grid, m->n, k, vp ? 1 : 0, vp ? vp[0] : 0.0, vp ? vp[1] : 0.0, vp ? vp[2] : 0.0, m->pivot[0], m->pivot[1], m->pivot[2], d.p);
    PCREG_LAUNCHED();
    std::vector<ModelPointD> h(m->replicas.empty() ? 0 : (size_t)m->n);
    if (!h.empty()) PCREG_CUDA(cudaMemcpyAsync(h.data(), d.p, d.bytes(), cudaMemcpyDeviceToHost, st));
    PCREG_CUDA(cudaStreamSynchronize(st));
    return store_normals(m, &d, h);
    PCREG_API_END
}

int pcreg_model_get_normals(const pcreg_model* m, double* out) {
    PCREG_API_BEGIN
    require_init();
    PCREG_REQUIRE(m && out, "pcreg_model_get_normals: null pointer");
    if (!m->nrm.p) throw StateError{"pcreg_model_get_normals: the model has no normals"};
    use_slot(0);
    std::vector<ModelPointD> h((size_t)m->n);
    PCREG_CUDA(cudaMemcpy(h.data(), m->nrm.p, m->nrm.bytes(), cudaMemcpyDeviceToHost));
    for (int64_t i = 0; i < m->n; ++i) { out[i] = h[i].x; out[m->n + i] = h[i].y; out[2 * m->n + i] = h[i].z; }
    return PCREG_OK;
    PCREG_API_END
}

}  // extern "C"
