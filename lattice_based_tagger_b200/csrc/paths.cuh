// paths.cuh — scoring and featurizing word paths the search did not produce itself.
//
// The beam kernel (beam.cuh) evaluates the transitions of the paths it grows; the kernels here evaluate
// GIVEN paths with the same arithmetic: a caller's path set (lt_pathset_eval: a gold analysis, candidates
// from elsewhere) and, for the perceptron step, the best paths of the batch's last search next to the gold
// paths (lt_perceptron_delta).
//
// One warp per path, lanes over words in chunks of 32.  A lane forms its word's transition context from the
// two words before it (shuffles, carried across chunk boundaries; BOS before the first word) as exactly the
// hash products the beam keeps per ring entry (beam_positions.inc, step 5): p1 = wj * M1, pp = wj * M1 + wi * M2,
// c1 = contextual morpheme * M1, has_i, the context flag and min(8, len_j).  The keys q0..q8 are then the
// beam's, the score program runs in the candidate loop's order and the trigram weights are summed by
// numpy_order_sum9.  Each hit also names where its weight lives — a slot of the hashed table, or
// feat_slots + an offset (in doubles) into the dense blocks — the index space of the perceptron's count
// buffer, mapped to lt_tables_desc order through the table builder's feat_dst.
#pragma once
#include "beam.cuh"

namespace lt {

constexpr uint32_t kNoHit = 0xFFFFFFFFu;

// context of a word's transition: what the beam keeps for the hypothesis the word extends
struct PathCtx {
    H2 p1, pp, c1;
    uint32_t tj, ul;
    bool has_i, j_unk, ctx8;
};

// SimpleTrigramFeatureScore.score (score_funcs.py:137-144) of scorer f for one transition, with the place of
// every weight that fires (kNoHit where a template does not fire), templates in order 0..8.
__device__ __forceinline__ double trigram_hits(const DevTables& T, int f, const EdgeView& k, H2 e0, H2 g0, const PathCtx& c,
                                               uint32_t (&hit)[9]) {
    const int NT = T.n_tags;
    const uint32_t blk_bytes = (uint32_t)dense_block_bytes(NT);
    const uint32_t dbase = (uint32_t)(T.feat_mask + 1) + (uint32_t)T.func_dense[f] * (blk_bytes / 8);
    const DenseView D = dense_view(T.dense + (size_t)T.func_dense[f] * blk_bytes, NT);
    const uint32_t tk = k.tag0, tj = c.tj;
    const uint32_t hk = feature_head32(tk, 0);
    FKey q[9];
    q[0] = feature_key_sum32(T.seeds[f][0], hk, h2_add(e0, c.p1));
    q[1] = feature_key_sum32(T.seeds[f][1], hk, c.p1);
    q[2] = feature_key_sum32(T.seeds[f][2], feature_head32(tj, tk), e0);
    q[4] = feature_key_sum(T.seeds[f][4], feature_head(k.len, 0), H2{0, 0});
    q[5] = feature_key_sum32(T.seeds[f][5], feature_head32(tk, (k.flags & LT_EDGE_IS_L) ? 1u : 0u), e0);
    q[7] = feature_key_sum32(T.seeds[f][7], 0u, h2_add(e0, c.pp));
    q[8] = feature_key_sum32(T.seeds[f][8], 0u, h2_add(g0, c.c1));
    const bool hashed4 = k.len >= (uint32_t)kT4Dense;
    const uint32_t probe = 0x7u | (hashed4 ? 1u << 4 : 0u) | (1u << 5) | (c.has_i ? 1u << 7 : 0u) | (c.ctx8 ? 1u << 8 : 0u);
    double w[9];
    uint32_t present = 0;
    #pragma unroll
    for (int i = 0; i < 9; ++i) {
        w[i] = 0.0;
        hit[i] = kNoHit;
        if ((probe >> i) & 1u) {
            const FeatProbe p = feat_first(T, q[i]);
            if (feat_resolve(T, q[i], p, w[i])) {
                present |= 1u << i;
                hit[i] = feat_hit_slot(T, q[i], p);
            }
        }
    }
    if ((D.m3[tj] >> tk) & 1u) {
        w[3] = D.t3[tj * NT + tk];
        present |= 1u << 3;
        hit[3] = dbase + tj * NT + tk;
    }
    if (!hashed4 && ((D.m4[k.len >> 5] >> (k.len & 31)) & 1u)) {
        w[4] = D.t4[k.len];
        present |= 1u << 4;
        hit[4] = dbase + NT * NT + k.len;
    }
    if (c.j_unk && ((D.m6[0] >> c.ul) & 1u)) {
        w[6] = D.t6[c.ul];
        present |= 1u << 6;
        hit[6] = dbase + NT * NT + kT4Dense + c.ul;
    }
    return numpy_order_sum9(w, present);
}

// The score program over one transition (the beam's candidate loop, beam_positions.inc: score += f(...) per
// scorer in order); the hits of scorer `func` (a trigram scorer, or -1 for none) go to `hit`.
__device__ __forceinline__ double path_increment(const DevTables& T, const EdgeView& k, const PathCtx& c, int func, uint32_t (&hit)[9]) {
    const H2 e0 = h2_mul(k.wk, kM0a, kM0b), g0 = h2_mul(k.mk, kM0a, kM0b);
    double inc = 0.0;
    #pragma unroll
    for (int i = 0; i < 9; ++i) hit[i] = kNoHit;
    #pragma unroll 1
    for (int f = 0; f < T.n_funcs; ++f) {
        const int kind = T.funcs[f].kind;
        double val;
        if (kind == LT_FUNC_TRIGRAM) {
            uint32_t h[9];
            val = trigram_hits(T, f, k, e0, g0, c, h);
            if (f == func) {
                #pragma unroll
                for (int i = 0; i < 9; ++i) hit[i] = h[i];
            }
        } else {
            double unused;
            edge_score_body(T, T.dense, k, e0, g0, f, kind, H2{0, 0}, H2{0, 0}, T.seeds[f][9], val, unused);
        }
        inc = __dadd_rn(inc, val);
    }
    return inc;
}

// The features of scorer `func` alone on one transition (no score): the perceptron's counting.
__device__ __forceinline__ void path_hits(const DevTables& T, const EdgeView& k, const PathCtx& c, int func, uint32_t (&hit)[9]) {
    const H2 e0 = h2_mul(k.wk, kM0a, kM0b), g0 = h2_mul(k.mk, kM0a, kM0b);
    trigram_hits(T, func, k, e0, g0, c, hit);
}

__device__ __forceinline__ H2 shfl_up_h2(H2 x, int d) {
    return H2{__shfl_up_sync(kFull, x.a, d), __shfl_up_sync(kFull, x.b, d)};
}
__device__ __forceinline__ H2 shfl_h2(H2 x, int src) {
    return H2{__shfl_sync(kFull, x.a, src), __shfl_sync(kFull, x.b, src)};
}

// One path of n words with one warp: word w (lane w % 32 of chunk w / 32) is loaded with its hashes by
// load(w, word) and handed to visit(w, valid, word, context).  Every lane calls visit once per chunk.
template <class Load, class Visit>
__device__ __forceinline__ void walk_words(const DevTables& T, int n, int lane, Load load, Visit visit) {
    // words base-1 (j of lane 0) and base-2 (i of lane 0, j... of lane 1): BOS, then nothing, before the path
    H2 w1 = T.bos, mo1 = T.bos, w2{0, 0}, mo2{0, 0};
    uint32_t t1 = LT_TAG_BOS, len1 = 0, t2 = LT_TAG_BOS;
    for (int base = 0; base < n; base += 32) {
        const int w = base + lane;
        const bool valid = w < n;
        EdgeView k{};
        k.tag0 = LT_TAG_BOS;
        k.tag1 = LT_NO_TAG;
        if (valid) load(w, k);
        H2 wj = shfl_up_h2(k.wk, 1), mj = shfl_up_h2(k.mk, 1);
        uint32_t tj = __shfl_up_sync(kFull, k.tag0, 1), lenj = __shfl_up_sync(kFull, k.len, 1);
        H2 wi = shfl_up_h2(k.wk, 2), mi = shfl_up_h2(k.mk, 2);
        uint32_t ti = __shfl_up_sync(kFull, k.tag0, 2);
        if (lane == 0) { wj = w1; mj = mo1; tj = t1; lenj = len1; wi = w2; mi = mo2; ti = t2; }
        if (lane == 1) { wi = w1; mi = mo1; ti = t1; }
        PathCtx c;
        c.has_i = w >= 1;       // word_i is None only for the first word (beam.py: BOS has no predecessor)
        const bool jctx = tj < 32u && ((kCtxMask >> tj) & 1u);
        const bool ictx = c.has_i && ti < 32u && ((kCtxMask >> ti) & 1u);
        c.p1 = h2_mul(wj, kM1a, kM1b);
        c.pp = c.has_i ? h2_add(c.p1, h2_mul(wi, kM2a, kM2b)) : H2{0, 0};
        c.c1 = jctx ? h2_mul(mj, kM1a, kM1b) : (ictx ? h2_mul(mi, kM1a, kM1b) : H2{0, 0});
        c.ctx8 = k.tag0 < 32u && ((kCtxMask >> k.tag0) & 1u) && (jctx || ictx);
        c.tj = tj;
        c.j_unk = tj == LT_TAG_UNK;
        c.ul = lenj < 8u ? lenj : 8u;
        visit(w, valid, k, c);
        w1 = shfl_h2(k.wk, 31); mo1 = shfl_h2(k.mk, 31);
        t1 = __shfl_sync(kFull, k.tag0, 31); len1 = __shfl_sync(kFull, k.len, 31);
        w2 = shfl_h2(k.wk, 30); mo2 = shfl_h2(k.mk, 30);
        t2 = __shfl_sync(kFull, k.tag0, 30);
    }
}

// walk_words over the records edges[0 .. n) (read-only for the kernel's lifetime), hashed by
// edge_hashes_inline: strings of LT_EDGE_EXPLICIT words from v.imp, the others from the sentence's prefix
// hashes in v.
template <class Visit>
__device__ __forceinline__ void walk_path(const DevTables& T, const lt_edge* edges, int n, const SentView& v, int lane, Visit visit) {
    walk_words(T, n, lane, [&](int w, EdgeView& k) {
        unpack_edge(ldg16(edges + w), k);
        edge_hashes_inline<1>(T, v, k, true);
    }, visit);
}

// A sentence's syllables (spaces dropped) into ch[0 .. L) and their prefix hashes into ha / hb[0 .. L], as the
// beam kernel stages them, in global scratch; -> L.
__device__ __forceinline__ int stage_sentence_hashes(const uint16_t* text, int s0, int s1, int lane, uint16_t* ch,
                                                     uint64_t* ha, uint64_t* hb) {
    const unsigned lt_mask = (1u << lane) - 1u;
    int L = 0;
    for (int base = 0; base < s1 - s0; base += 32) {
        const bool in = base + lane < s1 - s0;
        const uint32_t cu = in ? (uint32_t)text[s0 + base + lane] : 0x20u;
        const bool keep = in && cu != 0x20u;
        const unsigned km = __ballot_sync(kFull, keep);
        if (keep) ch[L + __popc(km & lt_mask)] = (uint16_t)cu;
        L += __popc(km);
    }
    __syncwarp();
    prefix_hashes_inline(ch, L, lane, ha, hb);
    __syncwarp();
    return L;
}

struct PathEvalArgs {
    const lt_edge* edges;       // the path set's words
    const int64_t* off;         // [n_paths + 1]
    const H2* hashes;           // (word, morph0, morph1) per LT_EDGE_EXPLICIT record
    int32_t n_paths;
    int32_t func;               // scorer whose hits are listed, -1: none
    double* scores;             // [n_paths]
    int32_t* feat;              // [9 * n_words] desc indices of the hits of word w, template order, or nullptr
    uint8_t* nfeat;             // [n_words]
    const int32_t* hit_feat;    // hit -> lt_tables_desc index of its feature (-1: none)
};

__global__ void __launch_bounds__(256) path_eval_kernel(const __grid_constant__ DevTables T, const __grid_constant__ PathEvalArgs A) {
    const int lane = threadIdx.x & 31;
    const int warps = (int)(gridDim.x * blockDim.x) >> 5;
    const SentView v{nullptr, nullptr, nullptr, nullptr, A.hashes};
    for (int p = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); p < A.n_paths; p += warps) {
        const int64_t o = A.off[p];
        const int n = (int)(A.off[p + 1] - o);
        double s = 0.0;
        walk_path(T, A.edges + o, n, v, lane, [&](int w, bool valid, const EdgeView& k, const PathCtx& c) {
            uint32_t hit[9];
            const double inc = valid ? path_increment(T, k, c, A.func, hit) : 0.0;
            // Sequence.add in word order, with the beam's -0.0 normalisation (beam_positions.inc)
            const int m = min(32, n - (w - lane));
            for (int l = 0; l < m; ++l) s = __dadd_rn(__dadd_rn(s, __shfl_sync(kFull, inc, l)), 0.0);
            if (valid && A.feat) {
                const int64_t gw = o + w;
                int cnt = 0;
                #pragma unroll
                for (int i = 0; i < 9; ++i) {
                    const int32_t d = hit[i] != kNoHit ? A.hit_feat[hit[i]] : -1;
                    if (d >= 0) A.feat[9 * gw + cnt++] = d;
                }
                A.nfeat[gw] = (uint8_t)cnt;
            }
        });
        if (lane == 0) A.scores[p] = s;
    }
}

// What the perceptron and evaluation kernels read of the batch's last search and of the gold path set.
struct SearchAndGold {
    const uint16_t* text;       // the batch's sentences (the last search)
    const int32_t* sent_off;
    int32_t n_sent;
    const int32_t* status;
    const uint32_t* path_off;   // best paths of the last search
    const lt_edge* path_edges;
    const H2* imp;              // an imported lattice's string hashes, or nullptr
    const lt_edge* gold_edges;  // gold path set, one path per sentence
    const int64_t* gold_off;
    const H2* gold_hashes;
    uint16_t* ch;               // scratch: syllables [n_units], prefix hashes [n_units + n_sent]
    uint64_t* ha;
    uint64_t* hb;
};

struct PerceptronArgs {
    SearchAndGold sg;
    int32_t func;               // the trigram scorer whose features are counted
    unsigned long long* counts; // per hit, two's complement
    uint8_t* differs;           // [n_sent]
    unsigned long long* n_differ;
};

// One warp per sentence: does the prediction differ from the gold path (trainer/train.py:_same_path on
// b, e, morph0, morph1, tag0, tag1), and if so count +1 per gold hit and -1 per predicted hit.
__global__ void __launch_bounds__(256) perceptron_kernel(const __grid_constant__ DevTables T, const __grid_constant__ PerceptronArgs A) {
    const int lane = threadIdx.x & 31;
    const int warps = (int)(gridDim.x * blockDim.x) >> 5;
    for (int s = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); s < A.sg.n_sent; s += warps) {
        const int st = A.sg.status[s];
        const int64_t go = A.sg.gold_off[s];
        const int G = (int)(A.sg.gold_off[s + 1] - go);
        const int s0 = A.sg.sent_off[s], s1 = A.sg.sent_off[s + 1];
        const lt_edge* pred = A.sg.path_edges + A.sg.path_off[s];
        const int P = (st == LT_SENT_OK) ? (int)(A.sg.path_off[s + 1] - A.sg.path_off[s]) : 0;
        uint16_t* ch = A.sg.ch + s0;
        uint64_t* ha = A.sg.ha + s0 + s;
        uint64_t* hb = A.sg.hb + s0 + s;
        if (st == LT_SENT_OK) stage_sentence_hashes(A.sg.text, s0, s1, lane, ch, ha, hb);
        const SentView pv{ch, ha, hb, nullptr, A.sg.imp};
        const SentView gv{nullptr, nullptr, nullptr, nullptr, A.sg.gold_hashes};
        bool differ = st != LT_SENT_OK || P != G;
        for (int base = 0; base < P && !differ; base += 32) {
            const int w = base + lane;
            bool mismatch = false;
            if (w < P) {
                EdgeView k, g;
                unpack_edge(ldg16(pred + w), k);
                edge_hashes_inline<1>(T, pv, k, true);
                unpack_edge(ldg16(A.sg.gold_edges + go + w), g);
                edge_hashes_inline<1>(T, gv, g, true);
                mismatch = k.b != g.b || k.e != g.e || k.tag0 != g.tag0 || k.tag1 != g.tag1 || k.mk.a != g.mk.a || k.mk.b != g.mk.b ||
                           k.m1.a != g.m1.a || k.m1.b != g.m1.b;
            }
            differ = __ballot_sync(kFull, mismatch) != 0u;
        }
        if (differ) {
            auto count = [&](unsigned long long delta) {
                return [&, delta](int, bool valid, const EdgeView& k, const PathCtx& c) {
                    if (!valid) return;
                    uint32_t hit[9];
                    path_hits(T, k, c, A.func, hit);
                    #pragma unroll
                    for (int i = 0; i < 9; ++i)
                        if (hit[i] != kNoHit) atomicAdd(A.counts + hit[i], delta);
                };
            };
            walk_path(T, A.sg.gold_edges + go, G, gv, lane, count(1ull));
            if (st == LT_SENT_OK) walk_path(T, pred, P, pv, lane, count(~0ull));     // -1
        }
        if (lane == 0) {
            A.differs[s] = differ ? 1 : 0;
            if (differ) atomicAdd(A.n_differ, 1ull);
        }
        __syncwarp();
    }
}

// counts per hit -> delta in lt_tables_desc order (dst: lt_tables::feat_dst)
__global__ void __launch_bounds__(256) gather_counts(const unsigned long long* __restrict__ counts, const uint32_t* __restrict__ dst,
                                                     int64_t n, uint32_t feat_slots, long long* __restrict__ delta) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t d = dst[i];
        long long v = 0;
        if (d != 0xFFFFFFFFu) v = (long long)counts[(d & 0x80000000u) ? feat_slots + (d & 0x7FFFFFFFu) : d];
        delta[i] = v;
    }
}

}  // namespace lt
