// evaluate.cuh — the best paths of the batch's last search against gold paths: word-level matches, whether
// each gold path lies in the search space, and the score the model gives it (lt_evaluate).
//
// One warp per sentence (grid stride over sentences), lanes over words in chunks of 32, like
// perceptron_kernel.  Per sentence:
//   1. matching: each predicted word binary-searches the gold path by b (gold b strictly increasing, checked
//      when the path set was created) and compares (b, e), the tags and the morpheme hashes; ballots count.
//   2. reachability (beam_search, beam/beam.py:5-61, oracle/lattice_oracle.py:beam_search): each gold word is
//      checked in order — tiling of [0, L) (the previous word's end carried by a shuffle across chunks), the
//      window, then the CSR bucket of its end position (lattice edges with its b, tags compared before any
//      hashing; the first edge equal on b, e, tags and morphemes is its image, or the beam's unknown word where
//      the span has no edge), and an unknown word after an unknown word only from the window's earliest begin
//      (beam.py:44-45).  The first failed check is the word's reason code; a ballot decides the sentence.
//   3. the image of a reachable gold path (lattice records, in batch scratch) is scored by walk_words with
//      path_increment: bit for bit lt_pathset_eval on the image, and the search's score when the image is the
//      path the search found.
#pragma once
#include "paths.cuh"

namespace lt {

struct EvaluateArgs {
    SearchAndGold sg;
    const double* scores;       // of the best paths
    const uint2* pos;           // lattice CSR: pos[sent_off[s] + e - 1] = (first edge, count) of the edges ending at e
    const lt_edge* edges;
    lt_edge* image;             // scratch: the image of gold word w [gold n_words]
    uint8_t* sent_class;        // [n_sent] LT_EVAL_*
    int32_t* counts;            // [LT_EVAL_N_COUNTS * n_sent]
    double* gold_scores;        // [n_sent]
    uint8_t* word_reason;       // [gold n_words] LT_GOLD_*
};

__device__ __forceinline__ bool h2_same(H2 x, H2 y) { return x.a == y.a && x.b == y.b; }

__device__ __forceinline__ int warp_count(bool x) { return __popc(__ballot_sync(kFull, x)); }

__device__ __forceinline__ lt_edge unknown_record(int b, int e) {
    lt_edge r{};
    r.b = (uint16_t)b;
    r.e = (uint16_t)e;
    r.len = (uint16_t)(e - b);
    r.tag0 = LT_TAG_UNK;
    r.tag1 = LT_NO_TAG;
    r.rule = LT_NO_RULE;
    r.flags = LT_EDGE_UNK;
    return r;
}

__global__ void __launch_bounds__(256) evaluate_kernel(const __grid_constant__ DevTables T, const __grid_constant__ EvaluateArgs A) {
    const int lane = threadIdx.x & 31;
    const int warps = (int)(gridDim.x * blockDim.x) >> 5;
    for (int s = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); s < A.sg.n_sent; s += warps) {
        const bool ok = A.sg.status[s] == LT_SENT_OK;
        const int64_t go = A.sg.gold_off[s];
        const int G = (int)(A.sg.gold_off[s + 1] - go);
        const lt_edge* gold = A.sg.gold_edges + go;
        const int s0 = A.sg.sent_off[s], s1 = A.sg.sent_off[s + 1];
        const lt_edge* pred = A.sg.path_edges + A.sg.path_off[s];
        const int P = ok ? (int)(A.sg.path_off[s + 1] - A.sg.path_off[s]) : 0;
        uint16_t* ch = A.sg.ch + s0;
        uint64_t* ha = A.sg.ha + s0 + s;
        uint64_t* hb = A.sg.hb + s0 + s;
        const int L = ok ? stage_sentence_hashes(A.sg.text, s0, s1, lane, ch, ha, hb) : 0;
        const SentView pv{ch, ha, hb, nullptr, A.sg.imp};
        const SentView gv{nullptr, nullptr, nullptr, nullptr, A.sg.gold_hashes};

        // ---- 1. predicted words against the gold word with the same b ----
        int n_seg = 0, n_tag = 0, n_full = 0, n_pu = 0, n_um = 0;
        for (int base = 0; base < P; base += 32) {
            const int w = base + lane;
            bool two = false, seg = false, tag = false, full = false, u0 = false, u1 = false;
            if (w < P) {
                EdgeView k;
                unpack_edge(ldg16(pred + w), k);
                two = k.tag1 != LT_NO_TAG;
                int lo = 0, hi = G;             // first gold word with b >= k.b
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if ((int)(ldg16(gold + mid).x & 0xFFFFu) < k.b) lo = mid + 1;
                    else hi = mid;
                }
                if (lo < G) {
                    EdgeView g;
                    unpack_edge(ldg16(gold + lo), g);
                    seg = g.b == k.b && g.e == k.e;
                    if (seg) {
                        edge_hashes_inline<1>(T, pv, k, true);
                        edge_hashes_inline<1>(T, gv, g, true);
                        tag = k.tag0 == g.tag0 && k.tag1 == g.tag1;
                        u0 = k.tag0 == g.tag0 && h2_same(k.mk, g.mk);
                        u1 = two && k.tag1 == g.tag1 && h2_same(k.m1, g.m1);
                        full = tag && h2_same(k.mk, g.mk) && h2_same(k.m1, g.m1);
                    }
                }
            }
            n_seg += warp_count(seg);
            n_tag += warp_count(tag);
            n_full += warp_count(full);
            n_pu += warp_count(w < P) + warp_count(two);
            n_um += warp_count(u0) + warp_count(u1);
        }

        // ---- 2. is each gold word in the search space; its image ----
        bool reach = ok && (G > 0 || L == 0);
        int n_gu = 0, prev_e = 0;
        uint32_t prev_t = LT_TAG_BOS;
        for (int base = 0; base < G; base += 32) {
            const int w = base + lane;
            const bool valid = w < G;
            EdgeView g{};
            g.tag0 = LT_TAG_BOS;
            g.tag1 = LT_NO_TAG;
            if (valid) unpack_edge(ldg16(gold + w), g);
            n_gu += warp_count(valid) + warp_count(g.tag1 != LT_NO_TAG);
            // the word before: its end (tiling) and its tag (unknown after unknown), carried across chunks
            int pe = __shfl_up_sync(kFull, g.e, 1);
            uint32_t pt = __shfl_up_sync(kFull, g.tag0, 1);
            if (lane == 0) { pe = prev_e; pt = prev_t; }
            uint32_t reason = LT_GOLD_UNCHECKED;
            if (ok && valid) {
                if (g.b != pe || g.e > L || (w == G - 1 && g.e != L)) {
                    reason = LT_GOLD_BREAKS_TILING;
                } else if (g.e - g.b > LT_WINDOW) {
                    reason = LT_GOLD_BEYOND_WINDOW;
                } else {
                    edge_hashes_inline<1>(T, gv, g, true);
                    const uint2 bucket = A.pos[s0 + g.e - 1];
                    bool span = false;
                    lt_edge img{};
                    reason = LT_GOLD_NOT_IN_LATTICE;
                    for (uint32_t i = 0; i < bucket.y; ++i) {
                        const uint4 raw = ldg16(A.edges + bucket.x + i);
                        EdgeView c;
                        unpack_edge(raw, c);
                        if (c.b != g.b) {
                            if (c.b > g.b) break;       // the bucket is sorted by b
                            continue;
                        }
                        span = true;
                        if (c.tag0 != g.tag0 || c.tag1 != g.tag1) continue;
                        edge_hashes_inline<1>(T, pv, c, true);
                        if (h2_same(c.mk, g.mk) && h2_same(c.m1, g.m1)) {
                            memcpy(&img, &raw, sizeof img);
                            reason = LT_GOLD_OK;
                            break;
                        }
                    }
                    // a span without any edge: the beam's unknown word (beam.py:36-38)
                    if (!span && g.tag0 == LT_TAG_UNK && g.tag1 == LT_NO_TAG && h2_same(g.mk, sub_hash(T, pv, g.b, g.e)) &&
                        h2_same(g.m1, H2{0, 0})) {
                        img = unknown_record(g.b, g.e);
                        reason = LT_GOLD_OK;
                    }
                    if (reason == LT_GOLD_OK && g.tag0 == LT_TAG_UNK && pt == LT_TAG_UNK && g.b != max(0, g.e - LT_WINDOW))
                        reason = LT_GOLD_UNK_AFTER_UNK;
                    if (reason == LT_GOLD_OK) A.image[go + w] = img;
                }
            }
            reach = reach && __ballot_sync(kFull, valid && reason != LT_GOLD_OK) == 0u;
            if (valid && A.word_reason) A.word_reason[go + w] = (uint8_t)reason;
            prev_e = __shfl_sync(kFull, g.e, 31);
            prev_t = __shfl_sync(kFull, g.tag0, 31);
        }

        // ---- 3. the image's score: Sequence.add in word order, as path_eval_kernel ----
        double image_score = 0.0;
        if (reach) {
            __syncwarp();       // the image records other lanes wrote
            const lt_edge* img = A.image + go;
            walk_words(T, G, lane, [&](int w, EdgeView& k) {
                unpack_edge(*reinterpret_cast<const uint4*>(img + w), k);
                edge_hashes_inline<1>(T, pv, k, true);
            }, [&](int w, bool valid, const EdgeView& k, const PathCtx& c) {
                uint32_t hit[9];
                const double inc = valid ? path_increment(T, k, c, -1, hit) : 0.0;
                const int m = min(32, G - (w - lane));
                for (int l = 0; l < m; ++l) image_score = __dadd_rn(__dadd_rn(image_score, __shfl_sync(kFull, inc, l)), 0.0);
            });
        }

        if (lane == 0) {
            const bool exact = ok && P == G && n_full == G;
            uint8_t cls;
            if (!ok) cls = LT_EVAL_FAILED;
            else if (exact) cls = LT_EVAL_CORRECT;
            else if (!reach) cls = LT_EVAL_UNREACHABLE;
            else cls = image_score > A.scores[s] ? LT_EVAL_SEARCH_ERROR : LT_EVAL_MODEL_ERROR;
            A.sent_class[s] = cls;
            if (A.counts) {
                int32_t* out = A.counts + (int64_t)LT_EVAL_N_COUNTS * s;
                out[LT_EVAL_GOLD_WORDS] = G;
                out[LT_EVAL_PRED_WORDS] = P;
                out[LT_EVAL_SEG] = n_seg;
                out[LT_EVAL_TAG] = n_tag;
                out[LT_EVAL_FULL] = n_full;
                out[LT_EVAL_GOLD_UNITS] = n_gu;
                out[LT_EVAL_PRED_UNITS] = n_pu;
                out[LT_EVAL_UNIT_MATCH] = n_um;
            }
            if (A.gold_scores) A.gold_scores[s] = reach ? image_score : __longlong_as_double(0x7FF8000000000000ll);
        }
        __syncwarp();
    }
}

}  // namespace lt
