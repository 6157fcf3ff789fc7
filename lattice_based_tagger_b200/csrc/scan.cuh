// scan.cuh — device exclusive scan of 32-bit counts (CSR offsets of the lattice, path offsets)
// and the kernel that packs the per-sentence best paths into one contiguous output array.
#pragma once
#include "cuda_compat.cuh"
#include <stdint.h>

#include "../../include/lt_b200.h"

namespace lt {

constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* warp_sums, uint32_t& block_total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = (lane < kScanThreads / 32) ? warp_sums[lane] : 0u;
        uint32_t wi = w;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t t = __shfl_up_sync(0xFFFFFFFFu, wi, d);
            if (lane >= d) wi += t;
        }
        if (lane < kScanThreads / 32) warp_sums[lane] = wi - w;
        if (lane == kScanThreads / 32 - 1) warp_sums[kScanThreads / 32] = wi;
    }
    __syncthreads();
    block_total = warp_sums[kScanThreads / 32];
    uint32_t r = warp_sums[warp] + incl - v;
    __syncthreads();
    return r;
}

// pass 1: per-tile sums
__global__ void __launch_bounds__(kScanThreads) scan_tile_sums(const uint32_t* __restrict__ in, int64_t n, uint32_t* __restrict__ sums) {
    __shared__ uint32_t ws[kScanThreads / 32 + 1];
    const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
    uint32_t local = 0;
    #pragma unroll
    for (int i = 0; i < kScanItems; ++i)
        if (base + i < n) local += in[base + i];
    uint32_t total;
    block_exclusive_scan(local, ws, total);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

// pass 2: exclusive scan of the tile sums by one block
__global__ void __launch_bounds__(kScanThreads) scan_sums(uint32_t* __restrict__ sums, int64_t n_tiles) {
    __shared__ uint32_t ws[kScanThreads / 32 + 1];
    uint32_t carry = 0;
    for (int64_t base = 0; base < n_tiles; base += kScanThreads) {
        const int64_t i = base + threadIdx.x;
        uint32_t v = (i < n_tiles) ? sums[i] : 0u;
        uint32_t total;
        uint32_t ex = block_exclusive_scan(v, ws, total);
        if (i < n_tiles) sums[i] = carry + ex;
        carry += total;
    }
}

// pass 3: exclusive scan inside each tile + tile offset
__global__ void __launch_bounds__(kScanThreads) scan_apply(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int64_t n,
                                                          const uint32_t* __restrict__ sums) {
    __shared__ uint32_t ws[kScanThreads / 32 + 1];
    const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
    uint32_t v[kScanItems];
    uint32_t local = 0;
    #pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
        v[i] = (base + i < n) ? in[base + i] : 0u;
        local += v[i];
    }
    uint32_t total;
    uint32_t run = block_exclusive_scan(local, ws, total) + sums[blockIdx.x];
    #pragma unroll
    for (int i = 0; i < kScanItems; ++i) {
        if (base + i < n) out[base + i] = run;
        run += v[i];
    }
}

// Small inputs: the whole exclusive scan by one CTA (one launch instead of three).
constexpr int kScanSmallThreads = 1024;
constexpr int64_t kScanSmallMax = 64 * 1024;
__global__ void __launch_bounds__(kScanSmallThreads) scan_small(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int64_t n) {
    __shared__ uint32_t warp_sums[33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t per = (n + kScanSmallThreads - 1) / kScanSmallThreads;
    const int64_t lo = (int64_t)threadIdx.x * per, hi = (lo + per < n) ? lo + per : n;
    uint32_t local = 0;
    for (int64_t i = lo; i < hi; ++i) local += in[i];
    uint32_t incl = local;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = warp_sums[lane];
        uint32_t wi = w;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, wi, d);
            if (lane >= d) wi += t;
        }
        warp_sums[lane] = wi - w;
    }
    __syncthreads();
    uint32_t run = warp_sums[warp] + incl - local;
    for (int64_t i = lo; i < hi; ++i) {
        const uint32_t v = in[i];
        out[i] = run;
        run += v;
    }
}

// Prologue of a batch: zeroes the control words and work counters (instead of separate memsets) and
// computes the WORK ORDER — sentence indices by raw length, longest first, so that the persistent warps
// of the lattice / beam kernels pull the expensive sentences early and the launch tail stays short
// (C2: 0.571 ms per step against 0.620 ms in input order).
// The CTAs do not talk to each other: CTA g of G sorts the sentences g, g + G, g + 2G, ... (histogram of
// clamped lengths, scan, scatter; the order inside a length bucket is arbitrary, results do not depend on
// it) and its r-th longest goes to position r * G + g — the G sorted sequences interleaved, a permutation
// whatever the lengths are.  One CTA = the exact order.  Measured on C2 (r2l): the exact order by one CTA
// makes the two big kernels 5.5 us faster than 32 interleaved sequences do and costs as much in the
// prologue itself; 4 CTAs are the best of both by a microsecond.
constexpr int kOrderBins = 1024;
constexpr int kPrologueMaxCtas = 4;
__host__ __device__ inline int prologue_ctas(int n_sent) {
    const int want = (n_sent + 2047) / 2048;
    return want < 1 ? 1 : (want > kPrologueMaxCtas ? kPrologueMaxCtas : want);
}
__global__ void __launch_bounds__(1024) batch_prologue(const int32_t* __restrict__ sent_off, int32_t n_sent,
                                                       uint32_t* __restrict__ order, unsigned int* __restrict__ ctl, int n_ctl,
                                                       unsigned long long* __restrict__ counters, int n_counters) {
    const int G = (int)gridDim.x, g = (int)blockIdx.x;
    if (g == 0) {
        if ((int)threadIdx.x < n_ctl) ctl[threadIdx.x] = 0;
        if ((int)threadIdx.x < n_counters) counters[threadIdx.x] = 0;
    }
    if (order == nullptr) return;
    __shared__ uint32_t bins[kOrderBins];
    __shared__ uint32_t warp_sums[32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    bins[t] = 0;
    __syncthreads();
    for (int64_t s = (int64_t)g + (int64_t)t * G; s < n_sent; s += (int64_t)blockDim.x * G) {
        int len = sent_off[s + 1] - sent_off[s];
        len = len < 0 ? 0 : (len >= kOrderBins ? kOrderBins - 1 : len);
        atomicAdd(&bins[kOrderBins - 1 - len], 1u);          // bin 0 = longest
    }
    __syncthreads();
    // exclusive scan of the 1024 bins: warp scans + scan of the warp totals
    const uint32_t v = bins[t];
    uint32_t incl = v;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += u;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = warp_sums[lane];
        uint32_t wi = w;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, wi, d);
            if (lane >= d) wi += u;
        }
        warp_sums[lane] = wi - w;
    }
    __syncthreads();
    bins[t] = warp_sums[warp] + incl - v;           // start of every bin
    __syncthreads();
    for (int64_t s = (int64_t)g + (int64_t)t * G; s < n_sent; s += (int64_t)blockDim.x * G) {
        int len = sent_off[s + 1] - sent_off[s];
        len = len < 0 ? 0 : (len >= kOrderBins ? kOrderBins - 1 : len);
        const uint32_t r = atomicAdd(&bins[kOrderBins - 1 - len], 1u);
        order[(int64_t)r * G + g] = (uint32_t)s;
    }
}

// lt_tables_update_weights: weight i goes to the slot of the hashed feature table that holds feature i
// (slot = 0x8000'0000 | ... marks a dense-table weight, 0xFFFF'FFFF a dropped feature: both are skipped here)
struct WeightSlot { uint64_t fp; double w; };
template <typename Slot>
__global__ void scatter_weights(Slot* __restrict__ table, const uint32_t* __restrict__ dst, const double* __restrict__ w, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t d = dst[i];
        if (d & 0x80000000u) continue;
        table[d].w = w[i];
    }
}

// zeroes the beam stage's queue cursor and counters when a lattice is searched a second time
__global__ void beam_reset(unsigned int* __restrict__ queue, unsigned long long* __restrict__ counters, int n_counters) {
    if (threadIdx.x == 0) *queue = 0;
    if ((int)threadIdx.x < n_counters) counters[threadIdx.x] = 0;
}

// best paths: reversed per-sentence scratch -> contiguous forward order
__global__ void pack_paths(const lt_edge* __restrict__ tmp, const int32_t* __restrict__ sent_off,
                           const uint32_t* __restrict__ path_off, int32_t n_sent, lt_edge* __restrict__ out) {
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    for (int s = blockIdx.x * warps_per_block + (threadIdx.x >> 5); s < n_sent; s += gridDim.x * warps_per_block) {
        const uint32_t o0 = path_off[s], o1 = path_off[s + 1];
        const int W = (int)(o1 - o0);
        const int s0 = sent_off[s];
        const uint4* src = reinterpret_cast<const uint4*>(tmp + s0);
        uint4* dst = reinterpret_cast<uint4*>(out + o0);
        for (int i = lane; i < W; i += 32) dst[i] = src[W - 1 - i];
    }
}

// Batches of up to kPackScanMax sentences: offsets AND packing in one launch.  CTA g owns the contiguous
// sentence range [g * per, (g + 1) * per): it sums the path lengths in front of its range itself (at most
// 256 KB of L2-resident counts, read side by side — cheaper than a scan launch of its own plus the gap
// behind it), scans its own range, writes path_off and moves its paths.
constexpr int kPackScanThreads = 256;
constexpr int64_t kPackScanMax = 64 * 1024;
__global__ void __launch_bounds__(kPackScanThreads) pack_paths_scan(const lt_edge* __restrict__ tmp, const int32_t* __restrict__ sent_off,
                                                                    const int32_t* __restrict__ path_len, uint32_t* __restrict__ path_off,
                                                                    int32_t n_sent, int32_t per, lt_edge* __restrict__ out) {
    __shared__ uint32_t warp_sums[kPackScanThreads / 32 + 1];
    __shared__ uint32_t s_off[kPackScanThreads + 1];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int r0 = (int)blockIdx.x * per;
    const int r1 = min(n_sent, r0 + per);
    if (r0 >= n_sent) return;
    // words in front of this CTA's range
    uint32_t local = 0;
    for (int i = t; i < r0; i += kPackScanThreads) local += (uint32_t)path_len[i];
    #pragma unroll
    for (int d = 16; d; d >>= 1) local += __shfl_xor_sync(0xFFFFFFFFu, local, d);
    if (lane == 0) warp_sums[warp] = local;
    __syncthreads();
    uint32_t carry = 0;
    #pragma unroll
    for (int w = 0; w < kPackScanThreads / 32; ++w) carry += warp_sums[w];
    __syncthreads();
    for (int base = r0; base < r1; base += kPackScanThreads) {
        const int s = base + t;
        const uint32_t v = (s < r1) ? (uint32_t)path_len[s] : 0u;
        uint32_t incl = v;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += u;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        uint32_t before = 0, total = 0;
        #pragma unroll
        for (int w = 0; w < kPackScanThreads / 32; ++w) {
            const uint32_t x = warp_sums[w];
            before += (w < warp) ? x : 0u;
            total += x;
        }
        const uint32_t off = carry + before + incl - v;
        s_off[t] = off;
        if (s < r1) {
            path_off[s] = off;
            if (s == n_sent - 1) path_off[n_sent] = off + v;      // (the last sentence's owner alone)
        }
        if (t == kPackScanThreads - 1) s_off[kPackScanThreads] = carry + total;
        __syncthreads();
        // this tile's paths: one warp per sentence
        const int tile_n = min(kPackScanThreads, r1 - base);
        for (int i = warp; i < tile_n; i += kPackScanThreads / 32) {
            const uint32_t o0 = s_off[i];
            const int W = (int)(((i + 1 < tile_n) ? s_off[i + 1] : s_off[kPackScanThreads]) - o0);
            const uint4* src = reinterpret_cast<const uint4*>(tmp + sent_off[base + i]);
            uint4* dst = reinterpret_cast<uint4*>(out + o0);
            for (int k = lane; k < W; k += 32) dst[k] = src[W - 1 - k];
        }
        carry += total;
        __syncthreads();
    }
}

// all survivors (k-best): path r of sentence s sits reversed at tmp[sent_off[s] * K + r * raw_len(s)]
__global__ void pack_paths_k(const lt_edge* __restrict__ tmp, const int32_t* __restrict__ sent_off,
                             const uint32_t* __restrict__ path_off, int32_t n_sent, int32_t K, lt_edge* __restrict__ out) {
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    const int64_t total = (int64_t)n_sent * K;
    for (int64_t i = blockIdx.x * warps_per_block + (threadIdx.x >> 5); i < total; i += (int64_t)gridDim.x * warps_per_block) {
        const int s = (int)(i / K), r = (int)(i - (int64_t)s * K);
        const uint32_t o0 = path_off[i], o1 = path_off[i + 1];
        const int W = (int)(o1 - o0);
        if (W == 0) continue;
        const int s0 = sent_off[s], raw = sent_off[s + 1] - s0;
        const uint4* src = reinterpret_cast<const uint4*>(tmp + (size_t)s0 * K + (size_t)r * raw);
        uint4* dst = reinterpret_cast<uint4*>(out + o0);
        for (int w = lane; w < W; w += 32) dst[w] = src[W - 1 - w];
    }
}

}  // namespace lt
