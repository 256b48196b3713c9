// pcreg_dev.cuh -- device-side helpers: exactly-rounded FP64 primitives that mirror the oracle's
// operation order, warp/block reductions, mbarrier + bulk-copy (TMA 1-D) wrappers for sm_100a.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pcreg {

// ---- exact arithmetic in the oracle's order (no FMA contraction) ------------------------------
// quickTF.m:5-7  [p 1]*T, column c:  ((x*T[0][c] + y*T[1][c]) + z*T[2][c]) + T[3][c]
// T is row-major 4x4 (row-vector convention).
__device__ __forceinline__ void quick_tf(const double* __restrict__ T, double x, double y, double z,
                                         double& qx, double& qy, double& qz) {
    qx = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, T[0]), __dmul_rn(y, T[4])), __dmul_rn(z, T[8])), T[12]);
    qy = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, T[1]), __dmul_rn(y, T[5])), __dmul_rn(z, T[9])), T[13]);
    qz = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, T[2]), __dmul_rn(y, T[6])), __dmul_rn(z, T[10])), T[14]);
}

// ((mx-qx)^2 + (my-qy)^2) + (mz-qz)^2  -- the one distance formula (oracle/nn_brute.c)
__device__ __forceinline__ double dist2_exact(double mx, double my, double mz, double qx, double qy, double qz) {
    const double dx = __dsub_rn(mx, qx), dy = __dsub_rn(my, qy), dz = __dsub_rn(mz, qz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// vecnorm(p,2,2) of one row: sqrt((x^2 + y^2) + z^2)
__device__ __forceinline__ double norm3_exact(double x, double y, double z) {
    return __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)));
}

// ---- reductions ------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum of NV doubles per thread; result valid in every thread (via shared memory).
// `scratch` must hold NV * 32 doubles.  Deterministic (fixed tree).
template <int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = warp_sum(v[k]);
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NV; ++k) scratch[k * 32 + warp] = v[k];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            double x = (lane < nwarp) ? scratch[k * 32 + lane] : 0.0;
            x = warp_sum(x);
            if (lane == 0) scratch[k * 32] = x;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = scratch[k * 32];
    __syncthreads();
}

// block_sum of NV doubles and one per-thread count, reduced as one more double in the same pass (exact: a count is an
// integer far below 2^53).  Every sum goes through the same tree as in block_sum<NV>.  `scratch` must hold (NV + 1) * 32
// doubles.  Returns the block's count in every thread.
template <int NV>
__device__ __forceinline__ long long block_sum_count(double (&v)[NV], long long count, double* scratch) {
    double x[NV + 1];
#pragma unroll
    for (int k = 0; k < NV; ++k) x[k] = v[k];
    x[NV] = (double)count;
    block_sum<NV + 1>(x, scratch);
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = x[k];
    return (long long)x[NV];
}

__device__ __forceinline__ long long block_sum_ll(long long v, long long* scratch /*[32]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    if (warp == 0) {
        long long x = (lane < nwarp) ? scratch[lane] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) scratch[0] = x;
    }
    __syncthreads();
    const long long r = scratch[0];
    __syncthreads();
    return r;
}

// ---- mbarrier + 1-D bulk copy (TMA engine, UBLKCP in SASS) -----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }
}
// global -> shared bulk copy, completion counted in bytes on `bar`.  dst/src 16-byte aligned,
// bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// order-preserving map of a non-negative double onto uint64 (plain bit pattern)
__device__ __forceinline__ unsigned long long dbits(double x) { return (unsigned long long)__double_as_longlong(x); }

// ---- block-wide K-th smallest selection with MATLAB's stable tie rule -------------------------------
// keys[0..n): order-preserving uint64 keys (KEY_NOSEL for excluded elements).  Selects the K smallest
// keys, ties broken by LOWER INDEX (MATLAB sort is stable: AlignPoints_KNN.m:24).  After the call
//   selected(i)  <=>  keys[i] < vK  ||  (all_eq && keys[i] == vK)  ||  keys[i] == KEY_SEL
// (when the K-th value is shared by more elements than fit, the equal keys are rewritten in place to
// KEY_SEL / KEY_NOSEL in index order).  MSB-first 8-bit radix select: 8 histogram passes.
constexpr unsigned long long KEY_NOSEL = ~0ull;
constexpr unsigned long long KEY_SEL = ~0ull - 1ull;

struct RadixSelShared {
    int hist[256];
    unsigned long long prefix;
    long long remaining;
    int count_eq;
    int warp_cnt[32];
    int run_eq;
};

// `order` (optional): order[r] = array position of the element whose tie-breaking rank is r (the array may
// be stored in a permuted order, e.g. spatially sorted source points); nullptr = array order.
__device__ __forceinline__ void block_radix_select(unsigned long long* __restrict__ keys, long long n, long long K,
                                                   RadixSelShared& sh, unsigned long long& vK, bool& all_eq,
                                                   const int32_t* __restrict__ order = nullptr) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    if (K <= 0) { vK = 0ull; all_eq = false; return; }        // nothing selected
    __syncthreads();
    if (tid == 0) { sh.prefix = 0ull; sh.remaining = K; }
    unsigned long long mask = 0ull;
    for (int pass = 7; pass >= 0; --pass) {
        for (int b = tid; b < 256; b += nthr) sh.hist[b] = 0;
        __syncthreads();
        const unsigned long long prefix = sh.prefix;
        for (long long i = tid; i < n; i += nthr) {
            const unsigned long long key = keys[i];
            if ((key & mask) == prefix) atomicAdd(&sh.hist[(int)((key >> (8 * pass)) & 255ull)], 1);
        }
        __syncthreads();
        if (tid == 0) {
            long long rem = sh.remaining;
            int b = 0;
            for (; b < 255; ++b) {
                if (rem <= sh.hist[b]) break;
                rem -= sh.hist[b];
            }
            sh.remaining = rem;
            sh.prefix = prefix | ((unsigned long long)b << (8 * pass));
            sh.count_eq = sh.hist[b];
        }
        mask |= 0xFFull << (8 * pass);
        __syncthreads();
    }
    vK = sh.prefix;
    const long long need_eq = sh.remaining;        // how many keys equal to vK belong to the first K
    all_eq = (need_eq == (long long)sh.count_eq);
    if (!all_eq) {
        if (tid == 0) sh.run_eq = 0;
        __syncthreads();
        const int lane = tid & 31, warp = tid >> 5, nwarp = (nthr + 31) >> 5;
        for (long long base = 0; base < n; base += nthr) {
            const long long r = base + tid;
            const long long i = (r < n) ? (order ? (long long)order[r] : r) : n;
            const bool eq = i < n && keys[i] == vK;
            const unsigned bal = __ballot_sync(0xffffffffu, eq);
            if (lane == 0) sh.warp_cnt[warp] = __popc(bal);
            __syncthreads();
            int off = sh.run_eq;
            for (int w = 0; w < warp; ++w) off += sh.warp_cnt[w];
            const int rank = off + __popc(bal & ((1u << lane) - 1u));
            if (eq) keys[i] = ((long long)rank < need_eq) ? KEY_SEL : KEY_NOSEL;
            __syncthreads();
            if (tid == 0) { int t = 0; for (int w = 0; w < nwarp; ++w) t += sh.warp_cnt[w]; sh.run_eq += t; }
            __syncthreads();
        }
    }
    __syncthreads();
}
__device__ __forceinline__ bool key_selected(unsigned long long key, unsigned long long vK, bool all_eq) {
    return (key < vK) || (all_eq && key == vK) || key == KEY_SEL;
}

}  // namespace pcreg
