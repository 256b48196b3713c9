// nn_brute.cu -- tiled brute-force nearest neighbour for sm_100a: FP32 scan on the FMA pipe,
// exact FP64 decision.
//
// What it replaces: the NN correspondence step of the ICP loop BASELINE.json's north_star names.
// The reference has no such code (SURVEY.md section 0); semantics are MATLAB knnsearch(X,Y,'K',1):
// Euclidean, FP64, ties -> smallest index (the reference's only literal 1-NN loop is
// ColorCodeModel.m:15-18).  Queries are q = quickTF(src_i, T_h) (quickTF.m:5-7), computed on the fly,
// never materialised.
//
// Algorithm
//   scan value   d'(j) = |m_j|^2 - 2 q.m_j   (3 FFMA per pair, |m|^2 in the float4 w lane; all
//                coordinates relative to the model pivot), i.e. d^2 - |q|^2 in FP32.
//   fast path    per group of G model points a thread keeps only the group minimum of d' for each of
//                its Q register-resident queries (FMNMX3), no index tracking.
//   slow path    a group whose minimum is <= (best d' so far + 2E) is re-scanned; every point inside
//                that band is evaluated EXACTLY in FP64 with the oracle's formula and operation order
//                on the original coordinates, and competes on (d2, original index).  E bounds the FP32
//                error of d' against the true FP64 distance (derivation in DESIGN.md), so the true
//                nearest neighbour -- and every exact tie of it -- is always inside the band: the
//                returned index and d2 are the FP64 brute-force answers, bit for bit.  A query so far away
//                that d' or E could overflow (2E > BRUTE_MAX_TWO_E) gets an infinite band: all points in FP64.
//   bound        the band needs a good initial "best so far": the previous ICP iteration's
//                correspondence when there is one, else a pure-min pass over a 1/8 sub-sample (the
//                scan order is a random permutation, so the head of the array is a random sample).
//   tiles        model tiles of 1024 float4 (16 KB) are staged in shared memory by the TMA engine
//                (cp.async.bulk + mbarrier, double-buffered); all 256 threads read them as broadcast
//                LDS.128.  Few queries (C2: 10 k) are spread over the SMs by splitting the MODEL across
//                blockIdx.y; partial (d2, idx) winners are merged by a small kernel.
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <algorithm>

#include "pcreg_internal.h"
#include "pcreg_dev.cuh"

namespace pcreg {

#ifndef BRUTE_PACKED
#define BRUTE_PACKED 1
#endif
constexpr int BRUTE_THREADS = 256;
constexpr int BRUTE_G = 16;                 // group size of the fast path
constexpr float BRUTE_ERR_COEF = 7.2e-7f;   // 12 * 2^-24: E = coef * (|q32| + max|m32|)^2
// Largest band 2E a query may have.  Above it (a query some 1e18 model radii away, or beyond the float range) the scan
// values |d'| <= 2 (|q32| + max|m32|)^2 could overflow, and with them the band: such a query scans with q32 = 0 and an
// infinite band instead, so every model point is decided in FP64 (brute_prologue).
constexpr float BRUTE_MAX_TWO_E = 1.0e30f;

__device__ __forceinline__ float fmin3(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

struct BruteArgs {
    const float4* m4; const int32_t* perm; const ModelPointD* md;
    const double* sx; const double* sy; const double* sz; int64_t ns;
    const double* T; int64_t nq;
    double px, py, pz; float max_norm;
    int64_t p_begin;            // scanned range of scan positions [p_begin, p_end)  (multiples of the group size)
    int64_t p_end;
    int64_t split_len;          // scan positions per blockIdx.y (multiple of the group size)
    const int32_t* prev;        // [nq] or null
    const float* bound_in;      // [nbound][nq] or null
    int nbound;
    float* pmin;                // PURE_MIN output [gridDim.y][nq]
    double* pd2; int32_t* pidx; // exact output [gridDim.y][nq]
};

// FP32 error band of one query: 2E with E = coef * (|q32| + max|m32|)^2, from the scan coefficients
// (ax,ay,az) = -2 * q32.  One function so that the prologue and the slow path agree bit for bit.
__device__ __forceinline__ float brute_two_e(float ax, float ay, float az, float max_norm) {
    const float qn = 0.5f * __fsqrt_ru(__fmaf_ru(ax, ax, __fmaf_ru(ay, ay, __fmul_ru(az, az))));
    const float s = __fadd_ru(qn, max_norm);
    return __fmul_ru(__fmul_ru(2.02f * BRUTE_ERR_COEF, s), s);
}

// Scan coefficients (ax,ay,az) = -2 q32 of one query and its band 2E; a query whose band exceeds BRUTE_MAX_TWO_E gets zero
// coefficients and an infinite band (its scan values are then |m|^2, finite, and every point lies inside the band).
__device__ __forceinline__ float brute_prologue(double qx, double qy, double qz, const BruteArgs& a, float& ax, float& ay, float& az) {
    ax = -2.f * __double2float_rn(qx - a.px); ay = -2.f * __double2float_rn(qy - a.py); az = -2.f * __double2float_rn(qz - a.pz);
    const float twoE = brute_two_e(ax, ay, az, a.max_norm);
    if (twoE <= BRUTE_MAX_TWO_E) return twoE;
    ax = ay = az = 0.f;
    return INFINITY;
}

// Re-scan one group for one query; exact FP64 evaluation of everything inside the band.  The exact
// running winner (d2, original index) lives in the kernel's output arrays (global memory): the slow path is
// rare, and keeping that state out of registers leaves the hot loop with 4 registers per query.
// Returns the tightened threshold.
__device__ __noinline__ float nn_slow(const float4* __restrict__ grp, int64_t jbase, float ax, float ay, float az,
                                      float thr, int64_t g, int64_t o, const BruteArgs& a) {
    const int64_t h = g / a.ns, i = g - h * a.ns;
    double qx, qy, qz;
    quick_tf(a.T + h * 16, a.sx[i], a.sy[i], a.sz[i], qx, qy, qz);
    const float twoE = thr == INFINITY ? INFINITY : brute_two_e(ax, ay, az, a.max_norm);     // INFINITY: see brute_prologue
    double best64 = a.pd2[o];
    int32_t bidx = a.pidx[o];
#pragma unroll 1
    for (int j = 0; j < BRUTE_G; ++j) {
        const float4 m = grp[j];
        float d = fmaf(ax, m.x, m.w);
        d = fmaf(ay, m.y, d);
        d = fmaf(az, m.z, d);
        if (d <= thr) {
            const int32_t orig = a.perm[jbase + j];
            if (orig >= 0) {
                const ModelPointD p = a.md[orig];
                const double d64 = dist2_exact(p.x, p.y, p.z, qx, qy, qz);
                if (d64 < best64 || (d64 == best64 && (bidx < 0 || orig < bidx))) { best64 = d64; bidx = orig; }
                const float cand = __fadd_ru(d, twoE);
                if (cand < thr) thr = cand;
            }
        }
    }
    a.pd2[o] = best64;
    a.pidx[o] = bidx;
    return thr;
}

constexpr int BRUTE_STAGES = 4;             // shared-memory ring of model tiles
constexpr int BRUTE_PREFETCH = 2;           // tiles in flight ahead of the consumer (ring slack = STAGES - PREFETCH - 1 tiles)
constexpr int BRUTE_WARPS = BRUTE_THREADS / 32;
constexpr size_t BRUTE_SMEM = (size_t)BRUTE_STAGES * BRUTE_TILE * sizeof(float4) + 2 * BRUTE_STAGES * sizeof(uint64_t);

template <int Q, bool PURE_MIN>
__global__ void __launch_bounds__(BRUTE_THREADS, 2) k_nn_brute(const __grid_constant__ BruteArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4* tiles = reinterpret_cast<float4*>(smem_raw);                                        // [STAGES][TILE]
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)BRUTE_STAGES * BRUTE_TILE * sizeof(float4));
    uint64_t* empty = full + BRUTE_STAGES;

    const int tid = threadIdx.x, lane = tid & 31;
    const int64_t qbase = (int64_t)blockIdx.x * (BRUTE_THREADS * Q);
    const int64_t r_begin = a.p_begin + (int64_t)blockIdx.y * a.split_len;
    const int64_t r_end = min(a.p_end, r_begin + a.split_len);
    const int nt = r_end > r_begin ? (int)((r_end - r_begin + BRUTE_TILE - 1) / BRUTE_TILE) : 0;

    if (tid == 0) {
        for (int s = 0; s < BRUTE_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], BRUTE_WARPS); }
        mbar_fence_init();
    }
    __syncthreads();
    // producer (thread 0): tile t -> stage t % STAGES, after every warp released the stage's previous tile
    auto issue_tile = [&](int t) {
        const int st = t % BRUTE_STAGES;
        if (t >= BRUTE_STAGES) mbar_wait(&empty[st], (uint32_t)(((t / BRUTE_STAGES) - 1) & 1));
        const int64_t start = r_begin + (int64_t)t * BRUTE_TILE;
        const uint32_t bytes = (uint32_t)(min((int64_t)BRUTE_TILE, r_end - start) * (int64_t)sizeof(float4));
        mbar_expect_tx(&full[st], bytes);
        bulk_g2s(tiles + (size_t)st * BRUTE_TILE, a.m4 + start, bytes, &full[st]);
    };
    if (tid == 0)
        for (int t = 0; t < BRUTE_PREFETCH && t < nt; ++t) issue_tile(t);

    // ---- per-thread query state: 4 registers per query in the hot loop ----
    float ax[Q], ay[Q], az[Q], thr[Q];
#pragma unroll
    for (int k = 0; k < Q; ++k) {
        const int64_t g = qbase + (int64_t)k * BRUTE_THREADS + tid;
        ax[k] = ay[k] = az[k] = 0.f;
        thr[k] = PURE_MIN ? FLT_MAX : -FLT_MAX;           // PURE_MIN: thr is the running minimum itself
        if (g < a.nq) {
            const int64_t h = g / a.ns, i = g - h * a.ns;
            double qx, qy, qz;
            quick_tf(a.T + h * 16, a.sx[i], a.sy[i], a.sz[i], qx, qy, qz);
            const float twoE = brute_prologue(qx, qy, qz, a, ax[k], ay[k], az[k]);
            if (!PURE_MIN) {
                const int64_t o = (int64_t)blockIdx.y * a.nq + g;
                a.pd2[o] = INFINITY;
                a.pidx[o] = -1;
                float bound = FLT_MAX;
                if (a.prev) {
                    const int32_t p = a.prev[g];
                    if (p >= 0) {
                        const ModelPointD mp = a.md[p];
                        const float mx = __double2float_rn(mp.x - a.px), my = __double2float_rn(mp.y - a.py), mz = __double2float_rn(mp.z - a.pz);
                        const float mw = __double2float_rn((double)mx * (double)mx + (double)my * (double)my + (double)mz * (double)mz);
                        float d = fmaf(ax[k], mx, mw);
                        d = fmaf(ay[k], my, d);
                        d = fmaf(az[k], mz, d);
                        bound = d;
                    }
                } else if (a.bound_in) {
                    for (int b = 0; b < a.nbound; ++b) bound = fminf(bound, a.bound_in[(int64_t)b * a.nq + g]);
                }
                thr[k] = twoE == INFINITY ? INFINITY : (bound < FLT_MAX) ? __fadd_ru(bound, twoE) : FLT_MAX;
            }
        }
    }

    // ---- stream the model tiles through the ring ----
#pragma unroll 1
    for (int it = 0; it < nt; ++it) {
        const int st = it % BRUTE_STAGES;
        if (tid == 0 && it + BRUTE_PREFETCH < nt) issue_tile(it + BRUTE_PREFETCH);
        mbar_wait(&full[st], (uint32_t)((it / BRUTE_STAGES) & 1));
        const float4* __restrict__ tp = tiles + (size_t)st * BRUTE_TILE;
        const int64_t tstart = r_begin + (int64_t)it * BRUTE_TILE;
        const int tlen = (int)min((int64_t)BRUTE_TILE, r_end - tstart);
#pragma unroll 1
        for (int g0 = 0; g0 < tlen; g0 += BRUTE_G) {
            float gm[Q];
#pragma unroll
            for (int jj = 0; jj < BRUTE_G; jj += 2) {
                const float4 m0 = tp[g0 + jj], m1 = tp[g0 + jj + 1];
#if BRUTE_PACKED
                // packed FP32 FMA (fma.rn.f32x2, FFMA2 in SASS): one instruction serves the same model point for TWO queries of this
                // thread -- half the issue slots per FMA, which is what the scalar form is short of (issue 78 %, FMA pipe 61 %).
                // Each half is an ordinary IEEE fma, so d' and with it the error band and the results are unchanged.
                const float2 x0 = make_float2(m0.x, m0.x), y0 = make_float2(m0.y, m0.y), z0 = make_float2(m0.z, m0.z), w0 = make_float2(m0.w, m0.w);
                const float2 x1 = make_float2(m1.x, m1.x), y1 = make_float2(m1.y, m1.y), z1 = make_float2(m1.z, m1.z), w1 = make_float2(m1.w, m1.w);
#pragma unroll
                for (int k = 0; k < Q; k += 2) {
                    const float2 a2x = make_float2(ax[k], ax[k + 1]), a2y = make_float2(ay[k], ay[k + 1]), a2z = make_float2(az[k], az[k + 1]);
                    float2 d0 = __ffma2_rn(a2x, x0, w0);
                    float2 d1 = __ffma2_rn(a2x, x1, w1);
                    d0 = __ffma2_rn(a2y, y0, d0);
                    d1 = __ffma2_rn(a2y, y1, d1);
                    d0 = __ffma2_rn(a2z, z0, d0);
                    d1 = __ffma2_rn(a2z, z1, d1);
                    if (PURE_MIN)      { thr[k] = fmin3(thr[k], d0.x, d1.x); thr[k + 1] = fmin3(thr[k + 1], d0.y, d1.y); }
                    else if (jj == 0)  { gm[k] = fminf(d0.x, d1.x); gm[k + 1] = fminf(d0.y, d1.y); }
                    else               { gm[k] = fmin3(gm[k], d0.x, d1.x); gm[k + 1] = fmin3(gm[k + 1], d0.y, d1.y); }
                }
#else
#pragma unroll
                for (int k = 0; k < Q; ++k) {
                    float d0 = fmaf(ax[k], m0.x, m0.w);
                    float d1 = fmaf(ax[k], m1.x, m1.w);
                    d0 = fmaf(ay[k], m0.y, d0);
                    d1 = fmaf(ay[k], m1.y, d1);
                    d0 = fmaf(az[k], m0.z, d0);
                    d1 = fmaf(az[k], m1.z, d1);
                    if (PURE_MIN)      thr[k] = fmin3(thr[k], d0, d1);
                    else if (jj == 0)  gm[k] = fminf(d0, d1);
                    else               gm[k] = fmin3(gm[k], d0, d1);
                }
#endif
            }
            if (!PURE_MIN) {
                bool hit = false;
#pragma unroll
                for (int k = 0; k < Q; ++k) hit |= (gm[k] <= thr[k]);
                if (hit) {
                    const int64_t jbase = tstart + g0;
#pragma unroll
                    for (int k = 0; k < Q; ++k) {
                        if (gm[k] <= thr[k]) {
                            const int64_t g = qbase + (int64_t)k * BRUTE_THREADS + tid;
                            thr[k] = nn_slow(tp + g0, jbase, ax[k], ay[k], az[k], thr[k], g, (int64_t)blockIdx.y * a.nq + g, a);
                        }
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);     // this warp is done with the stage
    }

#pragma unroll
    for (int k = 0; k < Q; ++k) {
        const int64_t g = qbase + (int64_t)k * BRUTE_THREADS + tid;
        if (g < a.nq) {
            if (PURE_MIN) a.pmin[(int64_t)blockIdx.y * a.nq + g] = thr[k];
        }
    }
}

// merge the per-split winners on (d2, original index)
__global__ void k_nn_merge(const double* __restrict__ pd2, const int32_t* __restrict__ pidx, int nsplit, int64_t nq,
                           int32_t* __restrict__ idx, double* __restrict__ d2) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= nq) return;
    double bd = INFINITY;
    int32_t bi = -1;
    for (int s = 0; s < nsplit; ++s) {
        const double d = pd2[(int64_t)s * nq + g];
        const int32_t i = pidx[(int64_t)s * nq + g];
        if (i >= 0 && (d < bd || (d == bd && (bi < 0 || i < bi)))) { bd = d; bi = i; }
    }
    idx[g] = bi;
    if (d2) d2[g] = bd;
}

template <int Q>
static void brute_run(const pcreg_model* m, BruteArgs a, const int32_t* d_prev, int32_t* d_idx, double* d_d2,
                      NNScratch& sc, cudaStream_t st) {
    const int64_t nq = a.nq;
    const int64_t qblocks = (nq + BRUTE_THREADS * Q - 1) / (BRUTE_THREADS * Q);
    const int slots = ctx().sm_count * 2;                  // co-resident blocks (2 per SM)
    // (function attributes are per device: set on every launch, it costs nothing next to the kernel)
    PCREG_CUDA(cudaFuncSetAttribute(k_nn_brute<Q, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BRUTE_SMEM));
    PCREG_CUDA(cudaFuncSetAttribute(k_nn_brute<Q, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BRUTE_SMEM));
    // Few query blocks: split the MODEL range so that all blocks fit in ONE wave with equal work
    // (split boundaries are multiples of the group size, not of the tile).  Many query blocks: no split.
    auto plan_split = [&](int64_t npts, int& nsplit, int64_t& len) {
        int64_t want = qblocks >= slots ? 1 : slots / qblocks;
        want = std::max<int64_t>(1, std::min<int64_t>(want, npts / (4 * BRUTE_G)));
        len = ((npts + want - 1) / want + BRUTE_G - 1) / BRUTE_G * BRUTE_G;
        nsplit = (int)((npts + len - 1) / len);
    };
    a.prev = d_prev;
    a.bound_in = nullptr; a.nbound = 0;
    if (!d_prev) {
        // bound pass: pure minimum of d' over the first 1/8 of the (randomly ordered) scan array
        const int64_t nsub = std::max<int64_t>(BRUTE_G, (m->n_pad / 8) / BRUTE_G * BRUTE_G);
        int ns0; int64_t len0;
        plan_split(nsub, ns0, len0);
        if (sc.pmin.n < (size_t)ns0 * nq) sc.pmin.alloc((size_t)ns0 * nq);
        BruteArgs b = a;
        b.p_begin = 0; b.p_end = nsub; b.split_len = len0; b.pmin = sc.pmin.p;
        dim3 grid((unsigned)qblocks, (unsigned)ns0);
        k_nn_brute<Q, true><<<grid, BRUTE_THREADS, BRUTE_SMEM, st>>>(b);
        PCREG_LAUNCHED();
        a.bound_in = sc.pmin.p; a.nbound = ns0;
    }
    int nsplit; int64_t len;
    plan_split(m->n_pad, nsplit, len);
    a.p_begin = 0; a.p_end = m->n_pad; a.split_len = len;
    if (nsplit == 1) {
        a.pd2 = d_d2; a.pidx = d_idx;
        if (!d_d2) { if (sc.pd2.n < (size_t)nq) sc.pd2.alloc((size_t)nq); a.pd2 = sc.pd2.p; }
    } else {
        if (sc.pd2.n < (size_t)nsplit * nq) sc.pd2.alloc((size_t)nsplit * nq);
        if (sc.pidx.n < (size_t)nsplit * nq) sc.pidx.alloc((size_t)nsplit * nq);
        a.pd2 = sc.pd2.p; a.pidx = sc.pidx.p;
    }
    dim3 grid((unsigned)qblocks, (unsigned)nsplit);
    k_nn_brute<Q, false><<<grid, BRUTE_THREADS, BRUTE_SMEM, st>>>(a);
    PCREG_LAUNCHED();
    if (nsplit > 1) {
        k_nn_merge<<<(unsigned)((nq + 255) / 256), 256, 0, st>>>(sc.pd2.p, sc.pidx.p, nsplit, nq, d_idx, d_d2);
        PCREG_LAUNCHED();
    }
}

void nn_brute_launch(const pcreg_model* m, const double* d_sx, const double* d_sy, const double* d_sz, int64_t ns,
                     const double* d_T, int64_t nhyp, const int32_t* d_prev, int32_t* d_idx, double* d_d2,
                     NNScratch& sc, cudaStream_t st) {
    BruteArgs a{};
    a.m4 = m->m4.p; a.perm = m->perm.p; a.md = m->md.p;
    a.sx = d_sx; a.sy = d_sy; a.sz = d_sz; a.ns = ns; a.T = d_T; a.nq = nhyp * ns;
    a.px = m->pivot[0]; a.py = m->pivot[1]; a.pz = m->pivot[2]; a.max_norm = m->max_norm;
    PCREG_REQUIRE(a.nq > 0, "nn_brute: no queries");
    PCREG_REQUIRE((a.nq + BRUTE_THREADS * 4 - 1) / (BRUTE_THREADS * 4) < 2147483647LL, "nn_brute: too many queries in one launch");
    static int force_q = -1;
    if (force_q < 0) { const char* e = getenv("PCREG_BRUTE_Q"); force_q = e ? atoi(e) : 0; }
    const bool wide = force_q ? (force_q == 8) : true;    // 8 queries per thread measured faster at every size (profiles/)
    if (wide) brute_run<8>(m, a, d_prev, d_idx, d_d2, sc, st);
    else                                                    brute_run<4>(m, a, d_prev, d_idx, d_d2, sc, st);
}

}  // namespace pcreg
