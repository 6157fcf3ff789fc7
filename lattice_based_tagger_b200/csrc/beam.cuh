// beam.cuh — transition scoring + fixed-window beam search kernel.
//
// Replaces beam_search / Beam / Sequence (beam/beam.py:5-124) and the score functions
// (beam/score_funcs.py:18-144) with their feature templates (features/feature.py:76-121).
//
// One warp per sentence (atomic work queue).  Hypotheses are back-pointer entries in a shared-
// memory ring of the last 9 end positions (window 8, beam.py:30).  An entry holds its score and the
// hash products of its last two words that the NEXT transition's feature keys are sums of
// (hash.cuh: keys are additive), so a transition costs additions, not string hashing.
//
// Per end position e the warp
//   1. makes sure the edges of e's CSR bucket are PREPARED: per edge the word/morpheme hash
//      products and everything of the score that depends on the edge alone — RegularizationScore,
//      the preference scorers, templates 4 and 5 (SURVEY App. B2).  Dictionary edges are prepared
//      32 consecutive edges at a time into a ring cache (the buckets of consecutive positions are
//      adjacent in HBM, so one full-warp pass serves many positions), unknown words 4 positions x 8
//      spans at a time;
//   2. counts edges per span and candidates per span; an unknown word after an unknown word is
//      allowed only from the window's first begin (beam.py:44-45), such candidates are never
//      enumerated;
//   3. enumerates candidates in the reference's generation order — begin ascending, parent rank
//      ascending, edge order ascending (beam.py:30-48) — 32 at a time, one per lane, and scores
//      each: score program in BeamScoreFunctions order, every fp64 add in the reference's
//      association (SURVEY App. A Q6); templates 0,1,2,7,8 are gathered from the feature table
//      (a cuckoo table: both slots of a key loaded at once), template 3/6 come from shared memory;
//   4. keeps the best `beam` candidates on the order-preserving integer image of the fp64 score
//      with ties resolved towards the earlier candidate, which is exactly the stable sort of
//      Beam.append (beam.py:83-86): rank counting (beam <= 16), a sorting network (<= 32) or two
//      sorted runs of 32 merged by sorting networks (<= 64);
//   5. writes the survivors as new ring entries and one back-pointer each (shared memory when the
//      host finds room, HBM otherwise).
// The best path is recovered from the back-pointers and written as 16-byte edge records.
//
// The kernel is instantiated per top-K method, beam size, sentence-array size and score program
// (beam_kernel<MODE, KT, UC, PROG>): with those fixed every shared-memory array sits at a constant
// offset and the scorer loop unrolls with its template seeds as immediates — in this latency-bound
// kernel dynamically indexed constant loads and spilled address arithmetic were the largest costs.
// Steps 1-5, the position loop, live in beam_positions.inc and are compiled into the kernel TWICE: once for any
// sentence, once without the code (and the out-of-line calls) that only buckets beyond the edge cache need —
// see the note at the top of that file.
#pragma once
#include "constraints.cuh"
#include "lattice.cuh"
#include "tables.cuh"

namespace lt {

constexpr int kRing = LT_WINDOW + 1;
constexpr int kEdgeRing = 64;                 // prepared dictionary edges: ring over the global edge index
#ifndef LT_BUCKET_CACHED
#define LT_BUCKET_CACHED 64
#endif
constexpr int kBucketCached = LT_BUCKET_CACHED;   // bucket-local edge indices below this are served from the ring (<= kEdgeRing)
static_assert(kBucketCached <= kEdgeRing, "a cached bucket must fit the ring");
constexpr int kUnkBlock = 4;                  // end positions whose unknown words are prepared together
constexpr int kCacheSlots = kEdgeRing + kUnkBlock * LT_WINDOW;
constexpr int kRankMaxBeam = 16;              // beams up to this size select by rank counting, larger ones by sorting network
constexpr uint32_t kCtxMask = (1u << LT_TAG_NOUN) | (1u << LT_TAG_ADVERB) | (1u << LT_TAG_ADJECTIVE) | (1u << LT_TAG_VERB);

// entry meta bits
constexpr uint32_t kMetaTagMask = 0xFFu;
constexpr uint32_t kMetaHasI = 1u << 8;
constexpr uint32_t kMetaHasCtx = 1u << 9;
constexpr uint32_t kMetaUnkLenShift = 12;     // min(8, len_j), 4 bits

struct BeamArgs {
    const uint16_t* text;
    const int32_t* sent_off;
    int32_t n_sent;
    int32_t units;              // shared-memory elements per sentence array: >= longest sentence + 8, a multiple of 8
    int32_t beam;
    int32_t warps;              // warps per CTA
    const uint2* pos;           // [n_units] (first edge, edge count) per (sentence, end position)
    const lt_edge* edges;
    const int32_t* status;      // from the lattice pass
    const uint32_t* flags;      // lattice overflow flags (lattice.cuh)
    uint64_t* trail;            // [(n_units) * beam] back-pointers
    lt_edge* path_tmp;          // [n_units] best path, reversed, at the sentence's offset
    int32_t* path_len;          // [n_sent]
    double* scores;             // [n_sent]
    unsigned long long* counters;   // [3]=T [4]=F [5]=Bk [6]=W
    unsigned int* queue;
    const uint32_t* order;      // queue position -> sentence index (longest first), or nullptr
    int32_t trail_smem;         // back-pointers in shared memory (4 B) instead of `trail` (8 B)
    const H2* imp;              // imported lattices: 3 hashes (word, morph0, morph1) per LT_EDGE_EXPLICIT edge
    // all survivors of the last position (beam_search's return value, beam.py:59-61) instead of matures[0] only:
    int32_t kbest;              // 1: also write every survivor's path
    lt_edge* kb_tmp;            // [n_units * beam] path r of sentence s, reversed, at sent_off[s] * beam + r * (raw length)
    int32_t* kb_len;            // [n_sent * beam] words of survivor r (0 beyond the survivors)
    double* kb_scores;          // [n_sent * beam]
    int32_t* kb_count;          // [n_sent] survivors (1 for an empty sentence: [BOS, EOS])
    const uint32_t* cdesc;      // constrained search: [n_units] position descriptors (constraints.cuh)
};

// Prepared edges (shared memory, struct of arrays).  Slots [0, kEdgeRing): dictionary edges at
// (global edge index % kEdgeRing); slots kEdgeRing + ((e - 1) % kUnkBlock) * 8 + (span - 1): the
// unknown word of (end position e, span).
struct EdgeCache {
    H2* e0;            // word hash   * M0
    H2* g0;            // morph0 hash * M0 (dictionary edges only: an unknown word is its own morpheme)
    double* kval;      // 2 doubles per scorer: score-program values that depend on the edge only
    uint32_t* meta;    // tag0 | len << 8 (16 bits) | flags << 24
    uint32_t* present; // bit f*2: template 4 present, bit f*2+1: template 5 present (scorer f); bits 24..31: min(255, e - b)
};

// doubles per edge in kval (stride 2 * n_funcs): for scorer f: [2f] = REG / MPREF / WPREF value or
// template-4 weight, [2f+1] = template-5 weight

// The back-pointer trail takes 4 bytes per kept entry in shared memory when the host finds that it
// does not cost residency (BeamArgs::trail_smem); otherwise 8-byte records go to HBM.
// Per-warp shared memory, in this order so that most arrays sit at compile-time offsets:
//   fixed part      edge cache (e0, g0, meta, present), selection pool, per-span tables, counters
//   beam part       ring entries: score, p1, pp, c1, meta, non-unknown ranks        (kRing * beam each)
//   sentence part   ha, hb, CSR row, syllables                                       (units each)
//   kval            edge-only score values, 2 doubles per scorer and cache slot
//   trail           back-pointers, units * beam (when they live in shared memory)
// `units` >= longest sentence of the batch + 8 (a multiple of 8); the common sizes are template
// parameters of the kernel, so that every array but the trail sits at a constant offset.
constexpr size_t kBeamFixedBytes = (size_t)kCacheSlots * 16 + (size_t)kEdgeRing * 16 + 32 * 8 + 64 * 8 +
                                   (size_t)kCacheSlots * 8 + (5 * 16 + 32 + 8) * 4;
static_assert(kBeamFixedBytes % 16 == 0, "fixed part keeps 16-byte alignment");
__host__ __device__ inline size_t beam_ring_bytes(int beam) {
    return (((size_t)kRing * beam * (8 + 48 + 4 + 1)) + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t beam_sentence_bytes(int units) { return (size_t)units * (8 + 8 + 8 + 2); }
// doubles of edge-only score values per cache slot: two per scorer
__host__ __device__ inline int beam_kval_doubles(int n_funcs, bool /*reg_tri*/) { return 2 * (n_funcs > 0 ? n_funcs : 1); }
__host__ __device__ inline size_t beam_warp_smem(int units, int beam, int kval_doubles, bool trail_smem) {
    const size_t bytes = kBeamFixedBytes + beam_ring_bytes(beam) + beam_sentence_bytes(units) + (size_t)kCacheSlots * 8 * (size_t)kval_doubles +
                         (trail_smem ? (size_t)units * beam * 4 : 0);
    return (bytes + 15) & ~(size_t)15;
}
// sentence-array sizes with their own kernel instantiation
__host__ __device__ inline int beam_units_class(int lcap) {
    const int need = lcap + 8;
    return need <= 64 ? 64 : (need <= 128 ? 128 : 0);
}

// candidate payload = shared-memory trail entry: (LT_WINDOW - span) << 27 | parent rank << 20 | bucket-local edge index
constexpr uint32_t kPayUnk = 0xFFFFFu;        // edge index of an unknown word

// HBM trail entry: edge reference (global edge index, or kTrailUnk) | span << 32 | parent rank << 40
constexpr uint32_t kTrailUnk = 0xFFFFFFFFu;

struct DenseView {
    const double* t3;
    const double* t4;
    const double* t6;
    const uint32_t* m3;
    const uint32_t* m4;
    const uint32_t* m6;
};

__device__ __forceinline__ DenseView dense_view(const unsigned char* blk, int nt) {
    DenseView d;
    d.t3 = reinterpret_cast<const double*>(blk);
    d.t4 = d.t3 + nt * nt;
    d.t6 = d.t4 + kT4Dense;
    d.m3 = reinterpret_cast<const uint32_t*>(d.t6 + 16);
    d.m4 = d.m3 + nt;
    d.m6 = d.m4 + 2;
    return d;
}

// numpy's ndarray.sum() association for the <= 9 surviving weights (SURVEY §8c / App. A Q6)
__device__ __forceinline__ double numpy_order_sum9(const double (&v)[9], uint32_t present) {
    const int n = __popc(present);
    if (n < 8) {
        double s = 0.0;
        #pragma unroll
        for (int i = 0; i < 9; ++i)
            if ((present >> i) & 1u) s = __dadd_rn(s, v[i]);
        return s;
    }
    // exactly one of nine missing (n == 8) or none (n == 9): first eight present values -> lanes
    int missing = (n == 9) ? 9 : (__ffs(~present & 0x1FFu) - 1);
    double r[8];
    #pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = (j < missing) ? v[j] : v[j + 1];
    double s = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    if (n == 9) s = __dadd_rn(s, v[8]);
    return s;
}

struct EdgeView {
    int b, e;
    uint32_t len, tag0, tag1, rule, split, flags;
    H2 wk, mk, m1;      // hashes of word, morph0, morph1
};

__device__ __forceinline__ void unpack_edge(uint4 raw, EdgeView& k) {
    k.b = (int)(raw.x & 0xFFFFu);
    k.e = (int)(raw.x >> 16);
    k.len = raw.y & 0xFFFFu;
    k.tag0 = (raw.y >> 16) & 0xFFu;
    k.tag1 = (raw.y >> 24) & 0xFFu;
    k.rule = raw.z;
    k.split = raw.w & 0xFFFFu;
    k.flags = (raw.w >> 16) & 0xFFu;
}

__device__ __forceinline__ void unknown_edge(int b, int e, EdgeView& k) {
    k.b = b; k.e = e;
    k.len = (uint32_t)(e - b); k.tag0 = LT_TAG_UNK; k.tag1 = LT_NO_TAG; k.rule = LT_NO_RULE;
    k.split = 0; k.flags = LT_EDGE_UNK;
}

// IMP: the batch may hold an imported lattice (lt_lattice_import) — only the all-survivors kernels (KB = 1)
// are launched on one, so the throughput instantiations compile the test out.
template <int IMP>
__device__ __forceinline__ void edge_hashes_inline(const DevTables& T, const SentView& v, EdgeView& k, bool need_m1) {
    if (IMP != 0 && (k.flags & LT_EDGE_EXPLICIT)) {
        // imported lattice (lt_lattice_import): the strings of this word were hashed on the host
        const H2* h = v.imp + 3 * (size_t)k.rule;
        k.wk = h[0];
        k.mk = h[1];
        k.m1 = h[2];
        return;
    }
    k.wk = sub_hash(T, v, k.b, k.e);
    k.mk = k.wk;
    k.m1 = H2{0, 0};
    if (k.flags & LT_EDGE_LEMMA) {
        const int p = k.b + (int)k.split;
        if (k.rule == LT_NO_RULE) {
            k.mk = sub_hash(T, v, k.b, p + 1);
            if (need_m1) k.m1 = sub_hash(T, v, p + 1, k.e);
        } else {
            RuleRec rec = rule_load(T, k.rule);
            H2 pre = (p > k.b) ? sub_hash(T, v, k.b, p) : H2{0, 0};
            k.mk = h2_concat(pre, rec.stem, pow_at(T, rec.stem_len));
            if (need_m1) {
                int from = p + ((k.flags & LT_EDGE_SKIP2) ? 2 : 1);
                H2 suf{0, 0};
                uint32_t sl = 0;
                if (from < k.e) { suf = sub_hash(T, v, from, k.e); sl = (uint32_t)(k.e - from); }
                k.m1 = h2_concat(rec.eomi, suf, pow_at(T, sl));
            }
        }
    }
}
// (out of line where code size matters more than the call: the kernels' any-sentence copies)
template <int IMP>
__device__ __noinline__ void edge_hashes(const DevTables& T, const SentView& v, EdgeView& k, bool need_m1) {
    edge_hashes_inline<IMP>(T, v, k, need_m1);
}

// Everything of a transition's score that depends on the edge alone (SURVEY App. B2), for scorer f:
//   REG / MPREF / WPREF: a = the scorer's value;  TRIGRAM: a = template 4 weight, b2 = template 5
//   weight, presence bits 0 / 1.
__device__ __forceinline__ uint32_t edge_score_body(const DevTables& T, const unsigned char* dense_blk, const EdgeView& k,
                                                    H2 e0, H2 g0, int f, int kind, H2 seed4, H2 seed5, H2 seed_pref,
                                                    double& a, double& b2) {
    uint32_t present = 0;
    const uint32_t tk = k.tag0;
    const lt_func& fn = T.funcs[f];
    a = 0.0;
    b2 = 0.0;
    if (kind == LT_FUNC_REG) {
        // score_funcs.py:65-73
        if (tk == LT_TAG_UNK) a = __dmul_rn(fn.p[0], __dadd_rn((double)k.len, 0.1));
        else a = __dmul_rn(fn.p[1], (double)k.len);
        a = __dadd_rn(0.0, a);
        if (k.len == 1 && tk == LT_TAG_NOUN) a = __dadd_rn(a, fn.p[2]);
    } else if (kind == LT_FUNC_MPREF) {
        // score_funcs.py:84-88
        FKey k0 = feature_key_sum32(seed_pref, feature_head32(tk, 0), g0);
        FeatProbe s0 = feat_first(T, k0);
        if (k.tag1 != LT_NO_TAG) {
            FKey k1 = feature_key_sum32(seed_pref, feature_head32(k.tag1, 0), h2_mul(k.m1, kM0a, kM0b));
            FeatProbe s1 = feat_first(T, k1);
            feat_resolve(T, k1, s1, b2);
        }
        feat_resolve(T, k0, s0, a);
        if (k.tag1 != LT_NO_TAG) a = __dadd_rn(a, b2);
        b2 = 0.0;
    } else if (kind == LT_FUNC_WPREF) {
        // score_funcs.py:99-100
        FKey k0 = feature_key_sum32(seed_pref, feature_head32(tk, 0), e0);
        FeatProbe s0 = feat_first(T, k0);
        feat_resolve(T, k0, s0, a);
    } else {
        // templates 4 (wk.len) and 5 (wk.word, wk.tag0, wk.is_l), features/feature.py:100,104
        const DenseView D = dense_view(dense_blk, T.n_tags);
        FKey q5 = feature_key_sum32(seed5, feature_head32(tk, (k.flags & LT_EDGE_IS_L) ? 1u : 0u), e0);
        FeatProbe s5 = feat_first(T, q5);
        if (k.len >= (uint32_t)kT4Dense) {
            FKey q4 = feature_key_sum(seed4, feature_head(k.len, 0), H2{0, 0});
            FeatProbe s4 = feat_first(T, q4);
            if (feat_resolve(T, q4, s4, a)) present |= 1u;
        } else if ((D.m4[k.len >> 5] >> (k.len & 31)) & 1u) {
            a = D.t4[k.len];
            present |= 1u;
        }
        if (feat_resolve(T, q5, s5, b2)) present |= 2u;
    }
    return present;
}

// any score program: kind, dense block and seeds of scorer f read from the tables
__device__ __noinline__ uint32_t edge_score(const DevTables& T, const unsigned char* dense_smem, const EdgeView& k,
                                            H2 e0, H2 g0, int f, double& a, double& b2) {
    const int kind = T.funcs[f].kind;
    const unsigned char* dense_blk = dense_smem;
    if (kind == LT_FUNC_TRIGRAM) dense_blk += (size_t)T.func_dense[f] * dense_block_bytes(T.n_tags);
    return edge_score_body(T, dense_blk, k, e0, g0, f, kind, T.seeds[f][4], T.seeds[f][5], T.seeds[f][9], a, b2);
}

// numpy's association from eight surviving weights on (SURVEY §8c): rare, so the nine weights are
// simply gathered again and summed by numpy_order_sum9.
// (inline: a call in the candidate loop costs more than the code, see beam_positions.inc)
__device__ __forceinline__ double trigram_sum_tree(const DevTables& T, const unsigned char* dense_blk, int NT, int f, FKey q0, FKey q1,
                                                FKey q2, FKey q7, FKey q8, uint32_t tj, uint32_t tk, uint32_t epresent,
                                                double val4, double val5, bool j_unk, uint32_t ul, bool has_i, bool ctx8) {
    const DenseView D = dense_view(dense_blk, NT);
    double w[9];
    uint32_t present = 0;
    #pragma unroll
    for (int i = 0; i < 9; ++i) w[i] = 0.0;
    if (feat_resolve(T, q0, feat_first(T, q0), w[0])) present |= 1u << 0;
    if (feat_resolve(T, q1, feat_first(T, q1), w[1])) present |= 1u << 1;
    if (feat_resolve(T, q2, feat_first(T, q2), w[2])) present |= 1u << 2;
    if ((D.m3[tj] >> tk) & 1u) { w[3] = D.t3[tj * NT + tk]; present |= 1u << 3; }
    if ((epresent >> (2 * f)) & 1u) { w[4] = val4; present |= 1u << 4; }
    if ((epresent >> (2 * f + 1)) & 1u) { w[5] = val5; present |= 1u << 5; }
    if (j_unk && ((D.m6[0] >> ul) & 1u)) { w[6] = D.t6[ul]; present |= 1u << 6; }
    if (has_i && feat_resolve(T, q7, feat_first(T, q7), w[7])) present |= 1u << 7;
    if (ctx8 && feat_resolve(T, q8, feat_first(T, q8), w[8])) present |= 1u << 8;
    return numpy_order_sum9(w, present);
}

// order-preserving integer image of an fp64 score (larger score -> larger key); 0 is "no candidate"
__device__ __forceinline__ uint64_t sortable(double s) {
    uint64_t bits = (uint64_t)__double_as_longlong(s);
    return bits ^ ((bits >> 63) ? 0xFFFFFFFFFFFFFFFFull : 0x8000000000000000ull);
}
__device__ __forceinline__ double unsortable(uint64_t key) {
    uint64_t bits = key ^ ((key >> 63) ? 0x8000000000000000ull : 0xFFFFFFFFFFFFFFFFull);
    return __longlong_as_double((long long)bits);
}

#ifndef LT_BEAM_MINB
#define LT_BEAM_MINB 1
#endif
#ifndef LT_BEAM_MAXW
#define LT_BEAM_MAXW 16        // largest CTA in warps (with LT_BEAM_MINB: the register budget the kernels are compiled for:
                               // 512 threads x 1 CTA = 128 registers, as 256 x 2 before).  One CTA of 13 warps is what fits an SM
                               // when a warp takes 16.5 KB of shared memory (beam 10, 128-element arrays): 13 resident warps
                               // instead of 3 x 4 — C3 sample 3.34 -> 3.19 ms, C5 sample 4.14 -> 3.96 ms (r3f)
#endif
#ifndef LT_BEAM_REG_WARPS
#define LT_BEAM_REG_WARPS 16   // warps per SM that budget allows (the host's residency estimate)
#endif
constexpr int kBeamMaxWarpsC = LT_BEAM_MAXW;
#ifndef LT_PROBE_SPLIT
#define LT_PROBE_SPLIT 1       // 1: generic kernels issue the loads of templates 7 and 8 after templates 0..2 are consumed
#endif
// (launch bounds: 128 registers per thread for every instantiation.  Compiling the small-beam instantiations for
// 5 resident 4-warp CTAs — 96 registers, with the shared-memory diet that makes room for the fifth — spills ~120
// bytes per thread and runs 16 % slower than 4 CTAs at 128 registers: profiles/README.md, r2d.)
constexpr int beam_max_threads(int, int, int, int) { return kBeamMaxWarpsC * 32; }
constexpr int beam_min_blocks(int, int, int, int) { return LT_BEAM_MINB; }
constexpr int kBeamWarps = 4;                 // preferred warps per CTA of the beam kernel
constexpr int kBeamMaxWarps = kBeamMaxWarpsC;              // largest CTA (128 registers per thread whatever the shape)

// Edge prep: hash products and the edge-only part of the score program into cache slot `slot`.
template <int PROG, int IMP, bool LEAN = false>
__device__ __forceinline__ void prep_edge(const DevTables& T, const SentView& v, const unsigned char* dense_smem,
                                          EdgeView& k, bool need_m1, int nf, int kvs, const EdgeCache& C, uint32_t slot) {
    if constexpr (LEAN) edge_hashes_inline<IMP>(T, v, k, need_m1);
    else edge_hashes<IMP>(T, v, k, need_m1);
    const H2 e0 = h2_mul(k.wk, kM0a, kM0b), g0 = h2_mul(k.mk, kM0a, kM0b);
    uint32_t present = 0;
    if (PROG == 1) {
        // (RegularizationScore, SimpleTrigramFeatureScore): both scorers inline, the trigram seeds as immediates,
        // the regulariser computed while the template-5 probe is in flight
        double reg, unused, w4, w5;
        const uint32_t tri = edge_score_body(T, dense_smem, k, e0, g0, 1, LT_FUNC_TRIGRAM, feature_seed(4u, 1u), feature_seed(5u, 1u),
                                             H2{0, 0}, w4, w5);
        edge_score_body(T, dense_smem, k, e0, g0, 0, LT_FUNC_REG, H2{0, 0}, H2{0, 0}, H2{0, 0}, reg, unused);
        (void)unused;
        present = tri << 2;
        C.kval[slot * 4 + 0] = reg;
        C.kval[slot * 4 + 1] = 0.0;
        C.kval[slot * 4 + 2] = w4;
        C.kval[slot * 4 + 3] = w5;
    } else {
        #pragma unroll 1
        for (int f = 0; f < nf; ++f) {
            double a, b2;
            present |= edge_score(T, dense_smem, k, e0, g0, f, a, b2) << (2 * f);
            C.kval[slot * kvs + 2 * f] = a;
            C.kval[slot * kvs + 2 * f + 1] = b2;
        }
    }
    C.e0[slot] = e0;
    if (slot < (uint32_t)kEdgeRing) C.g0[slot] = g0;
    C.meta[slot] = k.tag0 | (k.len << 8) | (k.flags << 24);
    const uint32_t span = (uint32_t)(k.e - k.b);
    C.present[slot] = present | ((span < 255u ? span : 255u) << 24);
}

// MODE selects the top-K of a position's candidates:
//   2  rank by counting (beam <= kRankMaxBeam): every candidate counts the pool entries that beat it
//   1  32-lane bitonic sorting network per chunk + bitonic merge with the kept list (beam <= 32)
//   0  two kept entries per lane = two sorted runs of 32, chunks merged into them by sorting networks (beam 33..64)
// KT: the beam size, UC: the sentence-array size when known at compile time (array offsets become
// constants, which is what keeps the kernel's address arithmetic out of registers); 0 = A.beam / A.units.
// PROG: 1 = the score program is exactly (RegularizationScore, SimpleTrigramFeatureScore) — the
// scorer loop of a candidate unrolls, the template seeds become immediates; 0 = read it from T.
// KB: 1 = every survivor of the last position is written out as well (lt_beam_kbest); 0 compiles that out of
// the instantiations the throughput path runs.
// TS: back-pointers in shared memory (1) or HBM (0) known at compile time; -1 = A.trail_smem.
// CONS: 1 = constrained search (lt_batch_set_constraints): the position loop reads A.cdesc and A.status is the search's
// status; only the generic instantiations (KT = UC = PROG = 0) have such a copy.
template <int MODE, int KT, int UC, int PROG, int KB = 0, int TS = -1, int CONS = 0>
__global__ void __launch_bounds__(beam_max_threads(KT, UC, PROG, KB), beam_min_blocks(KT, UC, PROG, KB)) beam_kernel(const __grid_constant__ DevTables T, const __grid_constant__ BeamArgs A) {
    static_assert(CONS == 0 || (KT == 0 && UC == 0 && PROG == 0), "only the generic instantiations have a constrained copy");
    constexpr int KR = (MODE == 0) ? 2 : 1;      // kept entries per lane
    LT_DYN_SMEM(smem_raw);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int K = KT ? KT : A.beam;
    const int NT = T.n_tags;

    // CTA-shared dense tables (tag x tag matrix, length vectors)
    const size_t dense_bytes = ((size_t)T.n_tri * dense_block_bytes(NT) + 15) & ~(size_t)15;
    unsigned char* dense_smem = smem_raw;
    for (size_t i = threadIdx.x * 4; i < (size_t)T.n_tri * dense_block_bytes(NT); i += blockDim.x * 4)
        *reinterpret_cast<uint32_t*>(dense_smem + i) = *reinterpret_cast<const uint32_t*>(T.dense + i);
    __syncthreads();
    if (A.flags[kFlagEdgeOverflow] | A.flags[kFlagStageOverflow]) {
        // lattice incomplete: the host grows the buffer and reruns; the path lengths the scan / pack kernels
        // behind this launch read must still be defined
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= A.n_sent; i += (int64_t)gridDim.x * blockDim.x)
            A.path_len[i] = 0;
        return;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) A.path_len[A.n_sent] = 0;      // the scan runs over n_sent + 1 entries

    const bool trail_smem = TS < 0 ? A.trail_smem != 0 : TS != 0;
    // instantiations of the throughput path carry a second copy of the position loop without the big-bucket code
    constexpr bool kLeanCopy = (PROG == 1 && KB == 0);
    const int units = UC ? UC : A.units;
    const int RK = kRing * K;
    const int kvs = beam_kval_doubles(T.n_funcs, PROG == 1);   // kval stride
    unsigned char* wbase = smem_raw + dense_bytes + (size_t)warp * beam_warp_smem(units, K, kvs, trail_smem);
    // fixed part
    EdgeCache C;
    C.e0 = reinterpret_cast<H2*>(wbase);
    C.g0 = C.e0 + kCacheSlots;
    uint64_t* s_newkey = reinterpret_cast<uint64_t*>(C.g0 + kEdgeRing);   // [32] selected keys by rank
    uint64_t* s_pool = s_newkey + 32;               // [64] selection pool: kept entries, then the chunk's lanes
    C.meta = reinterpret_cast<uint32_t*>(s_pool + 64);
    C.present = C.meta + kCacheSlots;
    uint32_t* s_cnt = C.present + kCacheSlots;      // [9] edges per span
    uint32_t* s_gstart = s_cnt + 16;                // [9] bucket-local index of the span's first edge
    uint32_t* s_tlist = s_gstart + 16;              // [8] spans that generate candidates, in generation order: first candidate << 4 | span
    uint32_t* s_nbeam = s_tlist + 16;               // [kRing] entries per ring slot
    uint32_t* s_nnon = s_nbeam + 16;                // [kRing] entries per ring slot that do not end in an unknown word
    uint32_t* s_newpay = s_nnon + 16;               // [32] selected payloads by rank
    uint32_t* s_acc = s_newpay + 32;                // [4] work counters of this warp: T, F, Bk, W (+ 4 spare)
    // beam part
    double* e_score = reinterpret_cast<double*>(wbase + kBeamFixedBytes);
    H2* e_p1 = reinterpret_cast<H2*>(e_score + RK);             // wj * M1
    H2* e_pp = e_p1 + RK;                                       // wj * M1 + wi * M2
    H2* e_c1 = e_pp + RK;                                       // contextual morph * M1
    uint32_t* e_meta = reinterpret_cast<uint32_t*>(e_c1 + RK);
    uint8_t* s_nonunk = reinterpret_cast<uint8_t*>(e_meta + RK);   // [kRing * K] ranks of the non-unknown entries, ascending
    // sentence part
    uint64_t* ha = reinterpret_cast<uint64_t*>(wbase + kBeamFixedBytes + beam_ring_bytes(K));
    uint64_t* hb = ha + units;
    uint2* spos = reinterpret_cast<uint2*>(hb + units);
    uint16_t* ch = reinterpret_cast<uint16_t*>(spos + units);
    C.kval = reinterpret_cast<double*>(ch + units);
    uint32_t* s_trail = reinterpret_cast<uint32_t*>(C.kval + kCacheSlots * kvs);   // [units * K] when trail_smem

    if (lane < 4) s_acc[lane] = 0;

    bool need_m1 = false;
    for (int f = 0; f < T.n_funcs; ++f) need_m1 |= (T.funcs[f].kind == LT_FUNC_MPREF);
    const int nf = PROG == 1 ? 2 : T.n_funcs;

    while (true) {
        unsigned int s = 0;
        if (lane == 0) s = atomicAdd(A.queue, 1u);
        s = __shfl_sync(kFull, s, 0);
        if (s >= (unsigned)A.n_sent) break;
        if (A.order) s = __ldg(A.order + s);
        const int s0 = __ldg(A.sent_off + s), s1 = __ldg(A.sent_off + s + 1);
        const int st = __ldg(A.status + s);
        // ---- stage syllables, prefix hashes and the sentence's CSR row ----
        int L = 0;
        const int raw_len = (st == LT_SENT_OK) ? (s1 - s0) : 0;
        for (int base = 0; base < raw_len; base += 32) {
            const int idx = s0 + base + lane;
            const bool valid = base + lane < raw_len;
            const uint32_t c = valid ? (uint32_t)__ldg(A.text + idx) : 0x20u;
            const bool keep = valid && (c != 0x20u);
            const unsigned km = __ballot_sync(kFull, keep);
            const int pos = L + __popc(km & lt_mask);
            if (keep) ch[pos] = (uint16_t)c;
            L += __popc(km);
        }
        __syncwarp();
        bool big_bucket = false;
        for (int i = lane; i < L; i += 32) {
            const uint2 row = __ldg(A.pos + s0 + i);
            spos[i] = row;
            big_bucket |= row.y > (uint32_t)kBucketCached;
        }
        prefix_hashes_inline(ch, L, lane, ha, hb);
        SentView v{ch, ha, hb, nullptr, KB ? A.imp : nullptr};

        if (L == 0 && lane == 0) { A.path_len[s] = 0; A.scores[s] = 0.0; }

        // beam[0] = [BOS] (beam.py:21-23)
        if (lane == 0) {
            e_score[0] = 0.0;
            e_p1[0] = h2_mul(T.bos, kM1a, kM1b);
            e_pp[0] = H2{0, 0};
            e_c1[0] = H2{0, 0};
            e_meta[0] = (uint32_t)LT_TAG_BOS;
            s_nbeam[0] = 1;
            s_nnon[0] = 1;
            s_nonunk[0] = 0;
        }
        __syncwarp();

        // the position loop, in the copy that fits the sentence (beam_positions.inc)
        bool lean = false;
        if constexpr (kLeanCopy) lean = !__any_sync(kFull, big_bucket);
        if (lean) {
            if constexpr (kLeanCopy) {
                constexpr bool kBig = false;
#include "beam_positions.inc"
            }
        } else {
            constexpr bool kBig = true;
#include "beam_positions.inc"
        }

        // ---- best path: matures[0] (tagger.py:78); with A.kbest every survivor (beam.py:59-61) ----
        // lane 0 follows the back-pointers (a dependent chain) and lists (end, edge reference); then the
        // lanes fetch the edge records side by side
        if constexpr (KB != 0) {
            const int nsurv = (L > 0) ? (int)s_nbeam[L % kRing] : 1;
            if (lane == 0) A.kb_count[s] = (st == LT_SENT_OK) ? nsurv : 0;
            for (int r = lane; r < K; r += 32) {
                A.kb_len[(size_t)s * K + r] = 0;
                A.kb_scores[(size_t)s * K + r] = 0.0;
            }
            __syncwarp();
        }
        if (L > 0) {
            uint64_t* s_path = ha;              // the prefix hashes are no longer needed
            const int nout = (KB != 0) ? (int)s_nbeam[L % kRing] : 1;
            for (int r0 = 0; r0 < nout; ++r0) {
                int W = 0;
                if (lane == 0) {
                    const double final_score = e_score[(L % kRing) * K + r0];
                    if (r0 == 0) A.scores[s] = final_score;
                    if constexpr (KB != 0) A.kb_scores[(size_t)s * K + r0] = final_score;
                    int e = L, r = r0;
                    while (e > 0) {
                        uint32_t eref, span;
                        if (trail_smem) {
                            const uint32_t t = s_trail[(e - 1) * K + r];
                            span = (uint32_t)LT_WINDOW - (t >> 27);
                            const uint32_t bidx = t & kPayUnk;
                            eref = (bidx == kPayUnk) ? kTrailUnk : spos[e - 1].x + bidx;
                            r = (int)((t >> 20) & 0x7Fu);
                        } else {
                            const uint64_t t = A.trail[(size_t)(s0 + e - 1) * K + r];
                            eref = (uint32_t)t;
                            span = (uint32_t)((t >> 32) & 0xFFu);
                            r = (int)((t >> 40) & 0xFFu);
                        }
                        s_path[W] = (uint64_t)eref | ((uint64_t)e << 32) | ((uint64_t)span << 48);
                        ++W;
                        e -= (int)span;
                    }
                    if (r0 == 0) {
                        A.path_len[s] = W;
                        s_acc[3] += (uint32_t)W;
                    }
                    if constexpr (KB != 0) A.kb_len[(size_t)s * K + r0] = W;
                }
                W = __shfl_sync(kFull, W, 0);
                __syncwarp();
                for (int w = lane; w < W; w += 32) {
                    const uint64_t t = s_path[w];
                    const uint32_t eref = (uint32_t)t;
                    lt_edge ed;
                    if (eref == kTrailUnk) {
                        const uint32_t e = (uint32_t)(t >> 32) & 0xFFFFu, span = (uint32_t)(t >> 48);
                        ed.b = (uint16_t)(e - span); ed.e = (uint16_t)e; ed.len = (uint16_t)span;
                        ed.tag0 = LT_TAG_UNK; ed.tag1 = LT_NO_TAG; ed.rule = LT_NO_RULE; ed.split = 0;
                        ed.flags = LT_EDGE_UNK; ed.reserved = 0;
                        if constexpr (CONS != 0) {
                            // at a forced constraint end the only unknown-word slot is the forced word's
                            const uint32_t d = __ldg(A.cdesc + s0 + e - 1);
                            if (d & kConsForced) {
                                ed.tag0 = (uint8_t)((d >> kConsTagShift) & 0xFFu);
                                ed.flags = (uint8_t)(LT_EDGE_FORCED | ((d & kConsIsL) ? LT_EDGE_IS_L : 0u));
                            }
                        }
                    } else {
                        ed = A.edges[eref];
                    }
                    if (r0 == 0) A.path_tmp[s0 + w] = ed;
                    if constexpr (KB != 0) A.kb_tmp[(size_t)s0 * K + (size_t)r0 * (s1 - s0) + w] = ed;
                }
                __syncwarp();
            }
        }
        __syncwarp();
    }
    // counters (per warp and launch each stays far below 2^32)
    __syncwarp();
    if (lane < 4) atomicAdd(A.counters + 3 + lane, (unsigned long long)s_acc[lane]);
}

}  // namespace lt
