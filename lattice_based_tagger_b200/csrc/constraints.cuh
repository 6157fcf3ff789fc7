// constraints.cuh — preparation of a constrained beam search (lt_batch_set_constraints, include/lt_b200.h).
//
// Runs between the lattice and the beam kernel, only when a constraint set is bound.  One warp per sentence writes
//   * the search's status of the sentence: the lattice's, or LT_SENT_BAD_CONSTRAINT when a constraint ends beyond
//     its last syllable;
//   * one descriptor per end position e (at the sentence's unit offset + e - 1, as the CSR rows), read by the
//     constrained copy of beam_kernel (beam_positions.inc):
//       bits 0..3   the largest span the constraints leave open for e: e - (first open begin), 0 strictly inside a
//                   constrained span.  Clamping the window's jmax to it blocks every span that overlaps a constraint
//                   without being it (rule 1) and moves the unknown-after-unknown begin to the first open begin (rule 3)
//       bit 4       e ends a constraint (whose span is then the only open one)
//       bit 5       ... with a tag that no lattice edge of that span has: the span's word is the forced word
//       bit 6       is_l of the constraint's begin (the forced word's is_l)
//       bits 8..15  the constraint's tag, LT_NO_TAG for any word
// Everything is derived from the lattice as it stands, so a grow-and-rerun or an imported lattice gives the same.
#pragma once
#include "lattice.cuh"

namespace lt {

constexpr uint32_t kConsSpanMask = 0xFu;
constexpr uint32_t kConsEnd = 1u << 4;
constexpr uint32_t kConsForced = 1u << 5;
constexpr uint32_t kConsIsL = 1u << 6;
constexpr int kConsTagShift = 8;
constexpr int kConsWarps = 8;                         // warps per CTA of constraint_prep_kernel
constexpr int kConsMaxUnits = 4096;                   // >= any sentence a search holds (lt_tables_max_sentence_units)

struct ConstraintArgs {
    const uint16_t* text;
    const int32_t* sent_off;
    int32_t n_sent;
    const int32_t* status;        // the lattice's
    const uint32_t* flags;        // lattice overflow flags: the lattice is incomplete and will be rebuilt
    const uint2* pos;
    const lt_edge* edges;
    const lt_constraint* cons;
    const int64_t* cons_off;      // [n_sent + 1]
    int32_t* search_status;       // [n_sent] out
    uint32_t* desc;               // [n_units] out
};

__global__ void __launch_bounds__(kConsWarps * 32) constraint_prep_kernel(const __grid_constant__ ConstraintArgs A) {
    __shared__ uint32_t s_isl[kConsWarps][kConsMaxUnits / 32];     // is_l per syllable of the warp's sentence
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    if (A.flags[kFlagEdgeOverflow] | A.flags[kFlagStageOverflow]) return;
    uint32_t* isl = s_isl[warp];
    const int64_t n_warps = (int64_t)gridDim.x * kConsWarps;
    for (int64_t s = (int64_t)blockIdx.x * kConsWarps + warp; s < A.n_sent; s += n_warps) {
        const int s0 = __ldg(A.sent_off + s), s1 = __ldg(A.sent_off + s + 1);
        const int st = __ldg(A.status + s);
        const int64_t c0 = __ldg(A.cons_off + s), nc = __ldg(A.cons_off + s + 1) - c0;
        const lt_constraint* C = A.cons + c0;
        // syllables and their is_l (first syllable of an eojeol), as the beam kernel stages them
        const int raw_len = (st == LT_SENT_OK) ? (s1 - s0) : 0;
        // (a sentence with status LT_SENT_OK has at most lt_tables_max_sentence_units() <= kConsMaxUnits units)
        for (int w = lane; w < (raw_len + 31) / 32; w += 32) isl[w] = 0;
        __syncwarp();
        int L = 0;
        for (int base = 0; base < raw_len; base += 32) {
            const int idx = base + lane;
            const bool valid = idx < raw_len;
            const uint32_t c = valid ? (uint32_t)__ldg(A.text + s0 + idx) : 0x20u;
            const bool keep = valid && c != 0x20u;
            const bool is_l = keep && (idx == 0 || __ldg(A.text + s0 + idx - 1) == 0x20u);
            const unsigned km = __ballot_sync(kFull, keep);
            const int p = L + __popc(km & lt_mask);
            // lanes whose syllables share a word of bits combine by OR
            if (is_l) atomicOr(isl + (p >> 5), 1u << (p & 31));
            L += __popc(km);
        }
        __syncwarp();
        const bool bad = st == LT_SENT_OK && nc > 0 && (int)C[nc - 1].e > L;
        if (lane == 0) A.search_status[s] = bad ? LT_SENT_BAD_CONSTRAINT : st;
        if (st != LT_SENT_OK || bad) continue;
        for (int e = 1 + lane; e <= L; e += 32) {
            // the last constraint that begins before e
            int64_t lo = 0, hi = nc;          // first index with b >= e
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if ((int)C[mid].b < e) lo = mid + 1; else hi = mid;
            }
            uint32_t d = (uint32_t)(e < LT_WINDOW ? e : LT_WINDOW);
            if (lo > 0) {
                const lt_constraint c = C[lo - 1];
                if (e < (int)c.e) {
                    d = 0;                                           // strictly inside: every span is blocked
                } else if (e == (int)c.e) {
                    const uint32_t tag = c.tag;
                    d = (uint32_t)(c.e - c.b) | kConsEnd | (tag << kConsTagShift);
                    if ((isl[c.b >> 5] >> (c.b & 31)) & 1u) d |= kConsIsL;
                    if (tag != LT_NO_TAG) {
                        const uint2 bucket = __ldg(A.pos + s0 + e - 1);
                        bool found = false;
                        for (uint32_t k = 0; k < bucket.y && !found; ++k) {
                            const lt_edge ed = A.edges[bucket.x + k];
                            found = ed.b == c.b && ed.tag0 == tag;
                        }
                        if (!found) d |= kConsForced;
                    }
                } else if (e - (int)c.e < (int)d) {
                    d = (uint32_t)(e - (int)c.e);                    // the constraint's end is the window's left edge
                }
            }
            A.desc[s0 + e - 1] = d;
        }
        __syncwarp();
    }
}

}  // namespace lt
