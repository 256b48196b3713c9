// pcreg_select.cuh -- fast block-wide "K smallest" selection for the ICP trim (AlignPoints_KNN.m:20-26
// rule: keep the round(k*n) smallest residuals, MATLAB's stable sort breaks ties by lower index).
//
// Residuals are continuous, so instead of eight 8-bit radix passes (whose leading passes put every key
// into one or two bins and serialise on shared-memory atomics) the K-th value is located with ONE
// histogram of SEL_BINS bins under a monotone map of the key, the few keys of the boundary bin are
// collected, and the K-th is ranked among them exactly on the full 64-bit key.  Falls back to the radix
// select (pcreg_dev.cuh) when the boundary bin is crowded (heavy duplicates).  Exact ties at the boundary
// are resolved in ORIGINAL index order, as in block_radix_select.  The map only decides how many keys
// share the boundary bin: any non-decreasing map gives the same, exact selection.
//
// Two steps, so that a caller can fill the histogram in the loop that produces its keys:
//   fill     one atomicAdd per included key into sh.hist[map(key)] (sh.hist is all zero before);
//   finish   block_hist_finish: boundary scan, candidates, ranking, fallback, tie rule; it leaves sh.hist
//            all zero again.
// block_hist_select is the two steps for keys already in memory, with the linear map over [kmin, kmax].
#pragma once
#include "pcreg_dev.cuh"

namespace pcreg {

constexpr int SEL_BINS = 2048;
constexpr int SEL_CAP = 1024;
#ifndef SEL_UNROLL
#define SEL_UNROLL 4
#endif

struct HistSelShared {
    int hist[SEL_BINS];
    unsigned long long cand[SEL_CAP];
    int warp_tot[32];           // boundary scan: per-warp bin totals
    int ncand;
    int bin;                    // boundary bin
    long long before;           // keys in lower bins
    unsigned long long vK;
    long long need_eq;
    int count_eq;
    RadixSelShared radix;       // fallback + tie resolution scratch
};

__device__ __forceinline__ int sel_clamp_bin(long long b) { return b < 0 ? 0 : (b >= SEL_BINS ? SEL_BINS - 1 : (int)b); }

// Linear map of [kmin, kmax] (as doubles) onto the bins.
struct SelBinsLinear {
    double rmin, scale;
    __device__ __forceinline__ int operator()(unsigned long long key) const {
        int b = (int)((__longlong_as_double((long long)key) - rmin) * scale);
        return b < 0 ? 0 : (b >= SEL_BINS ? SEL_BINS - 1 : b);
    }
};

// Range-free map: the key is the bit pattern of a non-negative double, so (key >> shift) - base, clamped, is
// monotone.  shift 45 = 1/128 octave per bin (16 octaves in view), shift 48 = 1/16 octave (128 octaves).
struct SelBinsShift {
    int shift;
    long long base;
    // 16 octaves centred on the exponent of `centre` (a key near the expected K-th); centre 0: the fixed
    // 1/16-octave window over [2^-64, 2^64)
    __device__ __forceinline__ static SelBinsShift around(unsigned long long centre) {
        SelBinsShift m;
        if (centre == 0ull) { m.shift = 48; m.base = (long long)(1023 - 64) << 4; }
        else                { m.shift = 45; m.base = ((long long)(centre >> 52) - 8) << 7; }
        return m;
    }
    __device__ __forceinline__ int operator()(unsigned long long key) const { return sel_clamp_bin((long long)(key >> shift) - base); }
};

// keys[0..n): bit patterns of non-negative doubles (KEY_NOSEL = excluded); sh.hist holds the count of every included key
// under `map`, complete in every thread (a barrier after the fill).  K = k_of_total(number of included keys) (block-uniform,
// at most that number; <= 0: nothing selected).  Leaves sh.hist all zero.
template <class Map, class KOf>
__device__ __forceinline__ void block_hist_finish(unsigned long long* __restrict__ keys, long long n, const Map& map, KOf k_of_total,
                                                  HistSelShared& sh, unsigned long long& vK, bool& all_eq, const int32_t* __restrict__ order) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nwarp = (nthr + 31) >> 5;
    // ---- boundary bin: every thread sums its run of bins, a block exclusive scan gives its prefix ----
    const int per = (SEL_BINS + nthr - 1) / nthr;
    const int b0 = tid * per < SEL_BINS ? tid * per : SEL_BINS, b1 = b0 + per < SEL_BINS ? b0 + per : SEL_BINS;
    int mine = 0;
    for (int b = b0; b < b1; ++b) mine += sh.hist[b];
    int inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) sh.warp_tot[warp] = inc;
    if (tid == 0) sh.ncand = 0;
    __syncthreads();
    long long excl = (long long)inc - mine, total = 0;
    for (int w = 0; w < nwarp; ++w) {
        const int t = sh.warp_tot[w];
        if (w < warp) excl += t;
        total += t;
    }
    const long long K = k_of_total(total);
    if (K > 0 && excl < K && K <= excl + mine) {           // the one thread whose run holds the K-th key
        long long cum = excl;
        int b = b0;
        for (;; ++b) {
            if (cum + sh.hist[b] >= K) break;
            cum += sh.hist[b];
        }
        sh.bin = b;
        sh.before = cum;
    }
    for (int b = b0; b < b1; ++b) sh.hist[b] = 0;       // only this thread reads its run: zero for the next fill
    if (K <= 0) { vK = 0ull; all_eq = false; return; }
    __syncthreads();
    // ---- the boundary bin's keys ----
    const int bstar = sh.bin;
    // SEL_UNROLL keys per trip, loaded before any is used: with keys in global memory (k_icp_update) a pass over them is
    // bound by the load latency of one key per thread otherwise
    for (long long i0 = tid; i0 < n; i0 += (long long)SEL_UNROLL * nthr) {
        unsigned long long kk[SEL_UNROLL];
#pragma unroll
        for (int u = 0; u < SEL_UNROLL; ++u) { const long long i = i0 + (long long)u * nthr; kk[u] = i < n ? keys[i] : KEY_NOSEL; }
#pragma unroll
        for (int u = 0; u < SEL_UNROLL; ++u) {
            const unsigned long long key = kk[u];
            if (key == KEY_NOSEL) continue;
            if (map(key) == bstar) {
                const int pos = atomicAdd(&sh.ncand, 1);
                if (pos < SEL_CAP) sh.cand[pos] = key;
            }
        }
    }
    __syncthreads();
    const int nc = sh.ncand;
    if (nc > SEL_CAP) {                                   // crowded boundary bin: exact radix select instead (block-uniform)
        block_radix_select(keys, n, K, sh.radix, vK, all_eq, order);
        return;
    }
    // ---- rank of the K-th key inside the boundary bin ----
    const long long kk = K - sh.before;                   // 1-based
    for (int t = tid; t < nc; t += nthr) {
        const unsigned long long c = sh.cand[t];
        int less = 0, eq = 0;
        for (int j = 0; j < nc; ++j) {
            const unsigned long long o = sh.cand[j];
            less += o < c ? 1 : 0;
            eq += o == c ? 1 : 0;
        }
        if ((long long)less < kk && kk <= (long long)(less + eq)) {       // every holder of that key writes the same values
            sh.vK = c;
            sh.need_eq = kk - less;
            sh.count_eq = eq;
        }
    }
    __syncthreads();
    vK = sh.vK;
    const long long need_eq = sh.need_eq;
    all_eq = (need_eq == (long long)sh.count_eq);
    if (!all_eq) {
        // stable tie rule: rank the keys equal to vK in ORIGINAL index order, keep the first need_eq (each round ends in a
        // barrier, so the rewritten keys are visible when this returns)
        RadixSelShared& rs = sh.radix;
        if (tid == 0) rs.run_eq = 0;
        __syncthreads();
        for (long long base = 0; base < n; base += nthr) {
            const long long r = base + tid;
            const long long i = (r < n) ? (order ? (long long)order[r] : r) : n;
            const bool eq = i < n && keys[i] == vK;
            const unsigned bal = __ballot_sync(0xffffffffu, eq);
            if (lane == 0) rs.warp_cnt[warp] = __popc(bal);
            __syncthreads();
            int off = rs.run_eq;
            for (int w = 0; w < warp; ++w) off += rs.warp_cnt[w];
            const int rank = off + __popc(bal & ((1u << lane) - 1u));
            if (eq) keys[i] = ((long long)rank < need_eq) ? KEY_SEL : KEY_NOSEL;
            __syncthreads();
            if (tid == 0) { int t = 0; for (int w = 0; w < nwarp; ++w) t += rs.warp_cnt[w]; rs.run_eq += t; }
            __syncthreads();
        }
    }
}

// keys[0..n): bit patterns of non-negative doubles (KEY_NOSEL = excluded); kmin/kmax: min / max over the
// included keys (block-uniform); K >= 1 and K <= number of included keys.
__device__ __forceinline__ void block_hist_select(unsigned long long* __restrict__ keys, long long n, long long K,
                                                  unsigned long long kmin, unsigned long long kmax, HistSelShared& sh,
                                                  unsigned long long& vK, bool& all_eq, const int32_t* __restrict__ order) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    if (K <= 0) { vK = 0ull; all_eq = false; return; }
    const double rmin = __longlong_as_double((long long)kmin), rmax = __longlong_as_double((long long)kmax);
    if (!(rmax > rmin) || !(rmax - rmin < 1.0e300)) {
        block_radix_select(keys, n, K, sh.radix, vK, all_eq, order);
        return;
    }
    const SelBinsLinear map{rmin, (double)SEL_BINS / (rmax - rmin)};
    for (int b = tid; b < SEL_BINS; b += nthr) sh.hist[b] = 0;
    __syncthreads();
    for (long long i0 = tid; i0 < n; i0 += (long long)SEL_UNROLL * nthr) {
        unsigned long long kk[SEL_UNROLL];
#pragma unroll
        for (int u = 0; u < SEL_UNROLL; ++u) { const long long i = i0 + (long long)u * nthr; kk[u] = i < n ? keys[i] : KEY_NOSEL; }
#pragma unroll
        for (int u = 0; u < SEL_UNROLL; ++u) {
            const unsigned long long key = kk[u];
            if (key != KEY_NOSEL) atomicAdd(&sh.hist[map(key)], 1);
        }
    }
    __syncthreads();
    block_hist_finish(keys, n, map, [K](long long) { return K; }, sh, vK, all_eq, order);
}

}  // namespace pcreg
