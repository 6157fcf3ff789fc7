// train.cuh — the update kernels of a mini-batch perceptron step (lt_trainer_step).
//
// perceptron_kernel (paths.cuh) leaves one count per feature hit: a slot of the hashed table, or feat_slots + an
// offset into the dense blocks.  The trainer keeps the weights in coefficient space (w[n_coef], indexed like the
// encoder's feature_dic, which may map several features to one coefficient) and the step goes
//   hit counts --(feat_dst, feat_coef)--> acc[n_coef] --> w += acc, u += (t-1) * acc --(feat_coef)--> the tables,
// three grid-stride passes of O(n_feat), O(n_coef) and O(n_feat).  Every count is an integer, so the atomic sums
// and w, u (doubles holding integers below 2^53 plus w_0) do not depend on the order of the adds.
#pragma once
#include "tables.cuh"

namespace lt {

constexpr uint32_t kFeatDstNone = 0xFFFFFFFFu, kFeatDstDense = 0x80000000u;

// offsets of the corpus sentences [first, first + count] rebased to the slice that starts at corpus_off[first]
__global__ void __launch_bounds__(256) rebase_offsets(const int32_t* __restrict__ corpus_off, int32_t first, int32_t count,
                                                      int32_t* __restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= count; i += gridDim.x * blockDim.x)
        out[i] = corpus_off[first + i] - corpus_off[first];
}

// acc[feat_coef[i]] += the count of feature i's hit, for every desc feature the trainer trains
__global__ void __launch_bounds__(256) gather_coef_counts(const unsigned long long* __restrict__ counts, const uint32_t* __restrict__ dst,
                                                          const int64_t* __restrict__ feat_coef, int64_t n_feat, uint32_t feat_slots,
                                                          unsigned long long* __restrict__ acc) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_feat; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = feat_coef[i];
        const uint32_t d = dst[i];
        if (c < 0 || d == kFeatDstNone) continue;
        const unsigned long long v = counts[(d & kFeatDstDense) ? feat_slots + (d & ~kFeatDstDense) : d];
        if (v) atomicAdd(acc + c, v);     // two's complement: negative counts add as well
    }
}

// w += acc, u += (t - 1) * acc, acc = 0
__global__ void __launch_bounds__(256) apply_coef_delta(unsigned long long* __restrict__ acc, int64_t n_coef, long long t_minus_1,
                                                        double* __restrict__ w, double* __restrict__ u) {
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_coef; c += (int64_t)gridDim.x * blockDim.x) {
        const long long d = (long long)acc[c];
        if (d == 0) continue;
        w[c] = __dadd_rn(w[c], (double)d);
        u[c] = __dadd_rn(u[c], (double)(t_minus_1 * d));
        acc[c] = 0ull;
    }
}

// the tables' weight of every trained feature := w[feat_coef[i]]: a hashed slot's weight field or a dense entry
__global__ void __launch_bounds__(256) scatter_coef(FeatSlot* __restrict__ table, double* __restrict__ dense, const uint32_t* __restrict__ dst,
                                                    const int64_t* __restrict__ feat_coef, int64_t n_feat, const double* __restrict__ w) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_feat; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = feat_coef[i];
        const uint32_t d = dst[i];
        if (c < 0 || d == kFeatDstNone) continue;
        if (d & kFeatDstDense)
            dense[d & ~kFeatDstDense] = w[c];
        else
            table[d].w = w[c];
    }
}

}  // namespace lt
