// lattice.cuh — lattice construction kernel (dictionary lookup + lemmatizer + eojeol enumeration).
//
// Replaces, for a whole batch, sentence_lookup_as_begin_index -> sentence_lookup ->
// MorphemeLookup.lookup -> morpheme_lookup -> lr_lookup -> MorphemeDictionary.lookup ->
// analyze_morphology -> get_lemma_candidates of the reference
// (dictionary/lookup.py:344-369, :7-62, :99-132, :212-279, :171-210; dictionary/dictionary.py:304-315;
// dictionary/lemmatizer.py:5-112).
//
// One warp per sentence, sentences pulled from an atomic work queue, ONE launch per batch.
//   1. stage: space-stripped syllables, eojeol starts and two prefix-hash arrays (warp scan) in
//      shared memory; every string the reference would build is a hash composed from these.
//   2. rule lists of the 1/2/3-syllable keys starting at every syllable (3 probes per syllable).
//   3. SUBSTRING TABLE: the dictionary payload (tag set + lemmatizer bits) of every substring of
//      at most `max_str` syllables (no longer string is in the dictionary) — one wave of
//      independent probes.  All plain dictionary tests of the enumeration below (the large majority
//      of the reference's string probes) are then shared-memory reads.
//   4. per eojeol, lanes = (task, split position) items in a flat index space, so lanes stay busy:
//        stage 1 (lr_lookup): tasks {whole, left_i, right_i}, n items per pair -> n*n items
//        stage 2 (sub-word scan, only when stage 1 found nothing): (begin, span, split) items
//      an item tests its plain split in the table; where a conjugation key starts at its split it
//      QUEUES a descriptor, and drain_rules() applies the rules (prefix + stem, eomi + suffix: the
//      only dictionary probes of the enumeration) with one descriptor per lane.  Hits are staged in
//      shared memory with a sort key (end, begin, class, split, candidate order) that encodes the
//      reference's emission order.
//   5. the eojeol's hits are filtered (lr_lookup keeps a split only when both sides are non-empty,
//      lookup.py:205-209) and ranked by key (a counting loop, or an in-place bitonic sort for eojeols with many
//      hits); staged edges go to HBM in rank order with one atomic reservation per flush (normally one per
//      sentence).  An eojeol whose hits outgrow the staging area goes, alone, to a retry pass with a larger one
//      (the RP = 1 instantiation); the sentence's other eojeols are finished here.
// Output is CSR keyed by END position: pos[sent_off[s]+e-1] = (first edge, count) of the edges of
// sentence s ending at syllable e, ordered by begin and, within one (b, e) span, in the reference's
// emission order (the only order beam_search can observe, SURVEY App. A Q5).
#pragma once
#include "tables.cuh"

namespace lt {

constexpr int kLatWarps = 4;                 // preferred warps per CTA of the lattice kernel
constexpr int kLatMaxWarps = 8;              // largest CTA (128 registers per thread either way)
#ifndef LT_RULE_QUEUE
#define LT_RULE_QUEUE 256
#endif
constexpr int kRuleQueue = LT_RULE_QUEUE;    // rule-work descriptors per warp; a pass queues at most 3 per lane (96)
constexpr int kRuleDrainAt = kRuleQueue - 96;   // drained between two passes once more than this many wait
constexpr unsigned kFull = 0xFFFFFFFFu;

// flags[] written by the lattice kernel, read by the beam kernel and the host
constexpr int kFlagEdgeOverflow = 0;         // edge buffer too small (cursor holds the needed size)
constexpr int kFlagStageOverflow = 1;        // an eojeol's hits did not fit the staging buffer

struct LatticeArgs {
    const uint16_t* text;       // raw UTF-16 units, spaces included
    const int32_t* sent_off;    // n_sent + 1
    int32_t n_sent;
    int32_t units;              // shared-memory elements per sentence array (>= longest sentence + 8)
    int32_t hcap;               // staging capacity (hits) per warp
    int32_t max_str;            // longest dictionary string (syllables), >= 1
    uint2* pos;                 // [n_units] out: (first edge, count) per (sentence, end position)
    lt_edge* edges;             // out
    uint32_t edge_cap;
    int32_t max_units;          // sentences with more raw code units are skipped with LT_SENT_TOO_LONG
    unsigned long long* cursor; // edge allocation cursor (64 bits: the sum of all reservations cannot wrap)
    uint32_t* flags;
    int32_t* sent_len;          // [n_sent] syllables
    int32_t* sent_edges;        // [n_sent] dictionary edges
    int32_t* status;            // [n_sent]
    unsigned long long* counters;   // [0]=L [1]=P [2]=E
    unsigned int* queue;        // work-queue cursor
    const uint32_t* order;      // queue position -> sentence index (longest first), or nullptr
    // Two-pass staging: when `retry_list` is set, an EOJEOL that outgrows the staging area of the main pass is
    // appended to it as (sentence, eojeol index) instead of raising the overflow flag, and the main pass goes on
    // with the sentence's other eojeols; the retry pass (retry_pass = 1, a small launch with a larger staging
    // area) takes its eojeols from that list and adds their edges to the sentence's lattice.
    uint2* retry_list;
    unsigned int* retry_count;
    int32_t retry_pass;
    int32_t mode;               // LT_LOOKUP_*: which eojeol lookup is enumerated
    int32_t sort_min;           // eojeols with at least this many staged hits are ranked by sorting (rank_staged)
};

// Per-warp shared memory.  `units` = elements per sentence array (>= longest sentence + 8, a
// multiple of 8), `hcap` = staging capacity; the substring table (units * max_str words) comes last,
// so that with `units` and `hcap` known at compile time every array sits at a constant offset.
__host__ __device__ inline size_t lattice_fixed_smem(int units, int hcap) {
    size_t bytes = (size_t)kRuleQueue * 16;        // rule-work queue
    bytes += (size_t)hcap * (8 + 16 + 4);          // staged keys, edge records, task id / final rank
    bytes += (size_t)units * (8 * 2 + 8 * 3);      // ha, hb, rref
    bytes += (size_t)units * 4 * 4;                // pstart, pcnt, tcnt (2 tasks per syllable of an eojeol)
    bytes += (size_t)units * (2 * 2 + 1);          // chars, eojeol starts, nend
    bytes += 64;                                   // counters
    return (bytes + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t lattice_warp_smem(int units, int hcap, int max_str) {
    return lattice_fixed_smem(units, hcap) + (((size_t)units * 4 * (size_t)max_str + 15) & ~(size_t)15);
}
// sentence-array sizes with their own kernel instantiation (together with the default staging capacity)
constexpr int kLatDefaultHcap = 128;
__host__ __device__ inline int lattice_units_class(int lcap) {
    const int need = lcap + 8;
    return need <= 64 ? 64 : (need <= 128 ? 128 : 0);
}

struct SentView {
    const uint16_t* ch;
    const uint64_t* ha;
    const uint64_t* hb;
    const uint2* rref;      // rref[3 * p + (key_len - 1)] = (first rule, count | k3_first << 31)
    const H2* imp;          // beam kernel, imported lattices: (word, morph0, morph1) hashes of LT_EDGE_EXPLICIT edges
};

__device__ __forceinline__ H2 sub_hash(const DevTables& T, const SentView& v, int b, int e) {
    return h2_sub(H2{v.ha[b], v.hb[b]}, H2{v.ha[e], v.hb[e]}, pow_at(T, (uint32_t)(e - b)));
}

// q / d for the small flat item indices of the enumeration loops: exact through a float reciprocal while
// q < 2^20, an integer division otherwise.  `inv` = small_rcp(d), once per loop: the hardware's approximate
// reciprocal (one instruction; the IEEE-rounded 1.0f / d carries an out-of-line slow path, and a call inside
// these loops costs more than it looks, see beam_positions.inc).  Error budget: rcp.approx is within one ulp
// (2^-23 relative), the multiply rounds once more (2^-24): |(q + 0.5) * inv - (q + 0.5) / d| < (q + 0.5) / d *
// 1.5 * 2^-23, which stays below the 0.5 / d distance to the next integer boundary while q + 0.5 < 2^21.4.
__device__ __forceinline__ float small_rcp(int d) {
#if defined(LT_SIMT_EMU)
    return 1.0f / (float)d;
#else
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"((float)d));
    return r;
#endif
}
__device__ __forceinline__ int small_div(int q, int d, float inv) {
    return q < (1 << 20) ? __float2int_rz(((float)q + 0.5f) * inv) : q / d;
}
// sqrt for the triangular item decode (the caller corrects the result by one either way)
__device__ __forceinline__ float approx_sqrt(float x) {
#if defined(LT_SIMT_EMU)
    return sqrtf(x);
#else
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}

// A shared-memory word as ONE lane reads it between two warp barriers: warp-uniform by construction, whatever
// the lanes that leave the second barrier first go on to write.
__device__ __forceinline__ uint32_t warp_read(const uint32_t* p) {
    __syncwarp();
    return __shfl_sync(kFull, *p, 0);
}

__device__ __forceinline__ bool is_py_space(uint32_t c) {
    // str.split() separators in the BMP
    return (c >= 0x09 && c <= 0x0D) || (c >= 0x1C && c <= 0x20) || c == 0x85 || c == 0xA0 || c == 0x1680 ||
           (c >= 0x2000 && c <= 0x200A) || c == 0x2028 || c == 0x2029 || c == 0x202F || c == 0x205F ||
           c == 0x3000;
}

// Prefix hashes of the staged syllables by warp scan: H[0] = 0, H[i+1] = H[i] * B + (c_i + 1).
__device__ __forceinline__ void prefix_hashes_inline(const uint16_t* ch, int L, int lane, uint64_t* ha, uint64_t* hb) {
    H2 carry{0, 0};
    if (lane == 0) {
        ha[0] = 0;
        hb[0] = 0;
    }
    constexpr uint64_t A1 = kBaseA, A2 = A1 * A1, A4 = A2 * A2, A8 = A4 * A4, A16 = A8 * A8;
    constexpr uint64_t B1 = kBaseB, B2 = B1 * B1, B4 = B2 * B2, B8 = B4 * B4, B16 = B8 * B8;
    for (int base = 0; base < L; base += 32) {
        const int i = base + lane;
        const uint64_t v = (i < L) ? (uint64_t)ch[i] + 1u : 0u;
        uint64_t sa = v, sb = v, ta, tb;
        ta = __shfl_up_sync(kFull, sa, 1);  tb = __shfl_up_sync(kFull, sb, 1);
        if (lane >= 1)  { sa += ta * A1;  sb += tb * B1; }
        ta = __shfl_up_sync(kFull, sa, 2);  tb = __shfl_up_sync(kFull, sb, 2);
        if (lane >= 2)  { sa += ta * A2;  sb += tb * B2; }
        ta = __shfl_up_sync(kFull, sa, 4);  tb = __shfl_up_sync(kFull, sb, 4);
        if (lane >= 4)  { sa += ta * A4;  sb += tb * B4; }
        ta = __shfl_up_sync(kFull, sa, 8);  tb = __shfl_up_sync(kFull, sb, 8);
        if (lane >= 8)  { sa += ta * A8;  sb += tb * B8; }
        ta = __shfl_up_sync(kFull, sa, 16); tb = __shfl_up_sync(kFull, sb, 16);
        if (lane >= 16) { sa += ta * A16; sb += tb * B16; }
        // sa = sum_{j<=lane} v_j * B^(lane-j); prefix = carry * B^(lane+1) + sa
        uint64_t pa = 1, pb = 1;   // B^(lane+1)
        {
            uint64_t xa = A1, xb = B1;
            const int k = lane + 1;
            #pragma unroll
            for (int bit = 0; bit < 6; ++bit) {
                if (k & (1 << bit)) { pa *= xa; pb *= xb; }
                xa *= xa; xb *= xb;
            }
        }
        const uint64_t outa = carry.a * pa + sa, outb = carry.b * pb + sb;
        if (i < L) {
            ha[i + 1] = outa;
            hb[i + 1] = outb;
        }
        carry.a = __shfl_sync(kFull, outa, 31);
        carry.b = __shfl_sync(kFull, outb, 31);
    }
    __syncwarp();
}

// (out of line in the lattice kernel, whose instruction footprint is the tighter one; the beam kernel inlines it)
#ifndef LT_PH_ATTR
#define LT_PH_ATTR __forceinline__        // (r2y: 2.7 us per C2 batch faster than out of line)
#endif
__device__ LT_PH_ATTR void prefix_hashes(const uint16_t* ch, int L, int lane, uint64_t* ha, uint64_t* hb) {
    prefix_hashes_inline(ch, L, lane, ha, hb);
}

// Stage the sentence: compaction, eojeol starts, prefix hashes.  Returns syllable count; n_eoj and
// bad (non-U+0020 whitespace seen) by reference.  eoj[n_eoj] = L.
__device__ __forceinline__ int stage_sentence(const uint16_t* __restrict__ text, int s0, int s1, int lane,
                                              uint16_t* ch, uint16_t* eoj, uint64_t* ha, uint64_t* hb,
                                              int& n_eoj, bool& bad) {
    int L = 0;
    n_eoj = 0;
    bad = false;
    uint32_t prev_last = 0x20;
    for (int base = s0; base < s1; base += 32) {
        int idx = base + lane;
        bool valid = idx < s1;
        uint32_t c = valid ? (uint32_t)__ldg(text + idx) : 0x20u;
        bool space = (c == 0x20u);
        if (valid && !space && is_py_space(c)) bad = true;
        uint32_t prev = __shfl_up_sync(kFull, c, 1);
        if (lane == 0) prev = prev_last;
        bool keep = valid && !space;
        bool start = keep && (prev == 0x20u);
        unsigned km = __ballot_sync(kFull, keep);
        unsigned sm = __ballot_sync(kFull, start);
        unsigned lt_mask = (1u << lane) - 1u;
        int pos = L + __popc(km & lt_mask);
        if (keep) ch[pos] = (uint16_t)c;
        if (start) eoj[n_eoj + __popc(sm & lt_mask)] = (uint16_t)pos;
        L += __popc(km);
        n_eoj += __popc(sm);
        prev_last = __shfl_sync(kFull, c, 31);
    }
    bad = __any_sync(kFull, bad);
    if (lane == 0) eoj[n_eoj] = (uint16_t)L;
    __syncwarp();
    prefix_hashes(ch, L, lane, ha, hb);
    return L;
}


// ---- enumeration state ---------------------------------------------------------------------------

// substring payload: bits 0..28 tag set, bit 29 in .verbs, bit 30 in .adjectives, bit 31 in .eomis
constexpr uint32_t kSubTagMask = 0x1FFFFFFFu;
constexpr uint32_t kSubVerb = 1u << 29, kSubAdj = 1u << 30, kSubEomi = 1u << 31;

struct Enum {
    const uint32_t* sub;     // [L * max_str]
    int max_str;
    // staging
    uint64_t* hkey;
    lt_edge* hrec;
    uint32_t* htask;         // task id while an eojeol is enumerated; afterwards htask[r] = staging slot of the survivor with rank r
    uint32_t* tcnt;          // hits per task of the current eojeol
    uint32_t* nh;            // staged entries (shared counter)
    int hcap;
    uint4* rq;               // rule-work queue: (word, split, conjugation key) triples waiting for their rules to be applied
    uint32_t* rqn;           // queued descriptors (shared counter)
};

// The per-warp shared-memory arrays as views (layout: lattice_fixed_smem / lattice_warp_smem).
struct LatticeViews {
    SentView v;
    Enum E;
    uint32_t* pstart;
    uint32_t* pcnt;
    uint16_t* ch;
    uint16_t* eoj;
    uint8_t* nend;
    uint64_t* ha;
    uint64_t* hb;
    uint2* rref;
};
template <int UC, int HCT>
__device__ __forceinline__ LatticeViews lattice_views(unsigned char* base, int units_rt, int hcap_rt, int max_str) {
    const int units = UC ? UC : units_rt;
    const int HC = HCT ? HCT : hcap_rt;
    uint4* rq = reinterpret_cast<uint4*>(base);
    uint64_t* hkey = reinterpret_cast<uint64_t*>(rq + kRuleQueue);
    lt_edge* hrec = reinterpret_cast<lt_edge*>(hkey + HC);
    uint32_t* htask = reinterpret_cast<uint32_t*>(hrec + HC);
    uint64_t* ha = reinterpret_cast<uint64_t*>(htask + HC);          // (kRuleQueue * 16 + HC * 28 is a multiple of 8 for even HC)
    uint64_t* hb = ha + units;
    uint2* rref = reinterpret_cast<uint2*>(hb + units);
    uint32_t* pstart = reinterpret_cast<uint32_t*>(rref + 3 * units);
    uint32_t* pcnt = pstart + units;
    uint32_t* tcnt = pcnt + units;
    uint16_t* ch = reinterpret_cast<uint16_t*>(tcnt + 2 * units);
    uint16_t* eoj = ch + units;
    uint8_t* nend = reinterpret_cast<uint8_t*>(eoj + units);
    uint32_t* nh = reinterpret_cast<uint32_t*>(nend + units);          // units is a multiple of 8
    uint32_t* rqn = nh + 1;
    uint32_t* sub = reinterpret_cast<uint32_t*>(base + lattice_fixed_smem(units, HC));
    LatticeViews W;
    W.v = SentView{ch, ha, hb, rref, nullptr};
    W.E = Enum{sub, max_str, hkey, hrec, htask, tcnt, nh, HC, rq, rqn};
    W.pstart = pstart; W.pcnt = pcnt; W.ch = ch; W.eoj = eoj; W.nend = nend; W.ha = ha; W.hb = hb; W.rref = rref;
    return W;
}

__device__ __forceinline__ uint32_t sub_get(const Enum& E, int x, int y) {
    const int len = y - x;
    if (len <= 0 || len > E.max_str) return 0u;
    return E.sub[x * E.max_str + (len - 1)];
}

// sort key: end | begin | pass | class (0 tag hits, 1 lemma hits) | split | order within the split.
// `pass` = 1 for the hits of word_lookup's substring loop, which come after the hits of its initial
// whole-eojeol lookup (lookup.py:157-168); 0 everywhere else.  k < 2^18: at most 255 rules per key.
__device__ __forceinline__ uint64_t hit_key(int e, int b, uint32_t cls, uint32_t split, uint32_t k, uint32_t pass = 0) {
    return ((uint64_t)e << 48) | ((uint64_t)b << 32) | ((uint64_t)pass << 31) | ((uint64_t)cls << 30) |
           ((uint64_t)(split & 0xFFFu) << 18) | (uint64_t)(k & 0x3FFFFu);
}

#ifndef LT_STAGE_ATTR
#define LT_STAGE_ATTR __forceinline__
#endif
#ifndef LT_FLUSH_ATTR
#define LT_FLUSH_ATTR __forceinline__     // (r2y: 5 us per C2 batch faster than out of line; drain_rules is the opposite, +80 us inline)
#endif
__device__ LT_STAGE_ATTR void stage_hit(const Enum& E, const lt_edge& rec, uint64_t key, uint32_t task) {
    const uint32_t slot = atomicAdd(E.nh, 1u);
    if (slot < (uint32_t)E.hcap) {
        E.hrec[slot] = rec;
        E.hkey[slot] = key;
        E.htask[slot] = task;
    }
    E.tcnt[task] = 1u;              // (only ever tested against zero)
}

// One (stem, eomi) lemma candidate whose strings are COMPOSED (a rule applied): the eomi must be a
// known Eomi; an Adjective stem is reported before a Verb stem (lemmatizer.py:44-50).  With
// reps > 1 the same candidate recurs at candidate indices cand + rep * rep_stride.
__device__ __forceinline__ void rule_candidate(const DevTables& T, const Enum& E, H2 stem, uint32_t stem_len, H2 eomi,
                                               uint32_t eomi_len, lt_edge proto, uint32_t split, uint32_t cand,
                                               uint32_t reps, uint32_t rep_stride, uint32_t task, uint32_t pass) {
    if (eomi_len > (uint32_t)E.max_str || stem_len > (uint32_t)E.max_str) return;    // longer than any entry
    // both probes in flight together: the stem's is wasted when the eomi misses, but a lane never waits twice
    const uint64_t pe = dict_probe(T, eomi, eomi_len);
    if (!((uint32_t)(pe >> 32) & kLemEomi)) return;
    const uint32_t ps = (uint32_t)(dict_probe(T, stem, stem_len) >> 32);
    if (!(ps & (kLemAdj | kLemVerb))) return;
    for (uint32_t rep = 0; rep < reps; ++rep) {
        const uint32_t k = (cand + rep * rep_stride) * 2u;
        if (ps & kLemAdj) {
            proto.tag0 = LT_TAG_ADJECTIVE;
            stage_hit(E, proto, hit_key(proto.e, proto.b, 1, split, k, pass), task);
        }
        if (ps & kLemVerb) {
            proto.tag0 = LT_TAG_VERB;
            stage_hit(E, proto, hit_key(proto.e, proto.b, 1, split, k + 1, pass), task);
        }
    }
}

// Rule work is QUEUED, not done in place: the items of an eojeol that meet a conjugation key are a
// minority of the lanes, so applying the rules inside the item loop runs the most expensive code of
// the kernel (rule records, hash composition, two dictionary probes per rule) on a handful of lanes.
// emit_pass() queues one descriptor per (word, split, key); drain_rules() then gives every lane one.
//   x = b | p << 12 | suffix code << 24 (0: p+1, 1: p+2, 2: e) | reps_is_count << 26 | is_l << 27 | skip2 << 28 | pass << 29
//   y = e | task << 12        z = first candidate index | rule count << 19        w = first rule
// Rules of one key applied at split p of the word [b, e): stem = word[:p-b] + rule.stem,
// eomi = rule.eomi + word[suffix_from - b:]  (lemmatizer.py:100-102, :107-111).  `cand0` is the
// candidate index of the key's first rule inside this split; with reps > 1 the whole list repeats
// (the nested duplicate loop of lemmatizer.py:100-102) at stride `count`.
// (Out of line; its arguments are the warp's shared-memory base and sizes by value, from which it
// rebuilds the array views — passing the views by reference would force the caller's copies into
// local memory for the whole kernel.)
#ifndef LT_DRAIN_ATTR
#define LT_DRAIN_ATTR __noinline__
#endif
template <int UC, int HCT>
__device__ LT_DRAIN_ATTR void drain_rules(const DevTables& T, unsigned char* base, int units_rt, int hcap_rt, int max_str, int lane) {
    const LatticeViews W = lattice_views<UC, HCT>(base, units_rt, hcap_rt, max_str);
    const SentView v = W.v;
    const Enum E = W.E;
    __syncwarp();
    const uint32_t n = *E.rqn;
    for (uint32_t i = lane; i < n; i += 32) {
        const uint4 d = E.rq[i];
        const int b = (int)(d.x & 0xFFFu), p = (int)((d.x >> 12) & 0xFFFu), e = (int)(d.y & 0xFFFu);
        const uint32_t code = (d.x >> 24) & 3u;
        const int suffix_from = (code == 0) ? p + 1 : (code == 1 ? p + 2 : e);
        const uint32_t count = d.z >> 19, cand0 = d.z & 0x7FFFFu, task = d.y >> 12;
        const uint32_t reps = ((d.x >> 26) & 1u) ? count : 1u;
        lt_edge proto;
        proto.b = (uint16_t)b;
        proto.e = (uint16_t)e;
        proto.len = (uint16_t)(e - b);
        proto.tag0 = 0;
        proto.tag1 = LT_TAG_EOMI;
        proto.split = (uint16_t)(p - b);
        proto.flags = (uint8_t)(LT_EDGE_LEMMA | (((d.x >> 27) & 1u) ? LT_EDGE_IS_L : 0) | (((d.x >> 28) & 1u) ? LT_EDGE_SKIP2 : 0));
        proto.reserved = 0;
        H2 suf{0, 0};
        uint32_t suf_len = 0;
        if (suffix_from < e) {
            suf = sub_hash(T, v, suffix_from, e);
            suf_len = (uint32_t)(e - suffix_from);
        }
        const H2 pre = (p > b) ? sub_hash(T, v, b, p) : H2{0, 0};
        const H2 pw_suf = pow_at(T, suf_len);
        RuleRec next = rule_load(T, d.w);
        for (uint32_t r = 0; r < count; ++r) {
            const RuleRec rec = next;
            if (r + 1 < count) next = rule_load(T, d.w + r + 1);      // in flight while this rule is probed
            // no dictionary string is longer than max_str: most candidates die here, before any hashing
            if (rec.eomi_len + suf_len > (uint32_t)E.max_str || (uint32_t)(p - b) + rec.stem_len > (uint32_t)E.max_str) continue;
            const H2 stem = h2_concat(pre, rec.stem, pow_at(T, rec.stem_len));
            const H2 eomi = h2_concat(rec.eomi, suf, pw_suf);
            proto.rule = d.w + r;
            rule_candidate(T, E, stem, (uint32_t)(p - b) + rec.stem_len, eomi, rec.eomi_len + suf_len, proto,
                           (uint32_t)(p - b), cand0 + r, reps, count, task, (d.x >> 29) & 1u);
        }
    }
    __syncwarp();
    if (lane == 0) *E.rqn = 0;
    __syncwarp();
}

// One pass of an enumeration loop = 32 items, one per lane.  All lanes first decide what their item
// produces — single-morpheme hits (`tagbits`), the plain-split analyses and the conjugation keys that
// start at the split position (lemmatizer.py:90-112) — then the hits and the rule descriptors of
// the whole pass are written side by side at offsets from ONE warp scan: no atomics, and the warp
// stays converged (staging hit by hit under `if (found)` ran the staging code on 3-5 lanes at a time).
//   tagbits   bit t: emit the single-morpheme word with tag t (Word.len = tag_len, is_l = tag_is_l)
//   order4    position of tag t in the emission order of its span, 4 bits per tag id — or ~0: the
//             dictionary's tag order (T.tag_pos, get_tags, dictionary.py:238-242)
//   lemmas    also run the lemmatizer part for (word [b, e), split p)
// Returns the number of lemma candidates the reference generates for the item.
template <int UC, int HCT>
__device__ __forceinline__ uint32_t emit_pass(const DevTables& T, const SentView& v, const Enum& E, unsigned char* base, int units_rt,
                                              int lane, bool valid,
                                              int b, int e, int p, uint32_t task, bool is_l, uint32_t tagbits,
                                              uint32_t tag_len, bool tag_is_l, uint64_t order4, bool lemmas, uint32_t pass) {
    uint32_t ncand = 0;
    uint32_t hits = valid ? tagbits : 0u;
    uint2 r1 = make_uint2(0u, 0u), rf = r1, rs = r1;
    const bool last = (p == e - 1);
    if (valid && lemmas) {
        // plain split (not at the last syllable): both strings are sentence substrings -> table
        if (!last) {
            ncand = 1;
            if (sub_get(E, p + 1, e) & kSubEomi) {
                const uint32_t ps = sub_get(E, b, p + 1);
                hits |= ((ps & kSubAdj) ? 1u << 29 : 0u) | ((ps & kSubVerb) ? 1u << 30 : 0u);
            }
        }
        r1 = v.rref[3 * p + 0];
        const uint2 r2 = (p + 2 <= e) ? v.rref[3 * p + 1] : make_uint2(0u, 0u);
        const uint2 r3 = (p + 3 <= e) ? v.rref[3 * p + 2] : make_uint2(0u, 0u);
        // {word[i:i+2], word[i:i+3]} in set order; at the last syllable both slices are that syllable itself:
        // its rules once more, with an empty suffix
        const bool k3_first = (r3.y >> 31) != 0;
        rf = last ? r1 : (k3_first ? r3 : r2);
        rs = last ? make_uint2(0u, 0u) : (k3_first ? r2 : r3);
    }
    const uint32_t c1 = r1.y & 0xFFFFu, cf = rf.y & 0xFFFFu, cs = rs.y & 0xFFFFu;
    // one-syllable key: the whole rule list once per rule of the key (lemmatizer.py:100-102)
    const uint32_t after1 = 1u + c1 * c1;
    ncand += c1 * c1 + cf + cs;
    const uint32_t nh_mine = (uint32_t)__popc(hits);
    const uint32_t np_mine = (c1 ? 1u : 0u) + (cf ? 1u : 0u) + (cs ? 1u : 0u);
    uint32_t incl = nh_mine | (np_mine << 16);
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += t;
    }
    const uint32_t total = __shfl_sync(kFull, incl, 31);
    const uint32_t cur_h = *E.nh, cur_q = *E.rqn;
    __syncwarp();                                   // every lane has read the counters
    if (lane == 31) {
        *E.nh = cur_h + (total & 0xFFFFu);
        *E.rqn = cur_q + (total >> 16);
    }
    uint32_t slot = cur_h + (incl & 0xFFFFu) - nh_mine;
    if (hits) E.tcnt[task] = 1u;                    // (only ever tested against zero)
    #pragma unroll 1
    while (hits) {
        const uint32_t t = (uint32_t)__ffs(hits) - 1u;
        hits &= hits - 1u;
        if (slot < (uint32_t)E.hcap) {
            const bool lemma = t >= 29u;
            const uint32_t tag0 = lemma ? (t == 29u ? (uint32_t)LT_TAG_ADJECTIVE : (uint32_t)LT_TAG_VERB) : t;
            const uint32_t len = lemma ? (uint32_t)(e - b) : tag_len;
            const uint32_t flags = lemma ? ((is_l ? LT_EDGE_IS_L : 0u) | LT_EDGE_LEMMA) : (tag_is_l ? LT_EDGE_IS_L : 0u);
            const uint32_t split = lemma ? (uint32_t)(p - b) : 0u;
            const uint32_t k = lemma ? t - 29u
                                     : (order4 == ~0ull ? (uint32_t)T.tag_pos[t] : (uint32_t)((order4 >> (4u * (t & 15u))) & 0xFu));
            reinterpret_cast<uint4*>(E.hrec)[slot] =
                make_uint4((uint32_t)b | ((uint32_t)e << 16), len | (tag0 << 16) | ((lemma ? (uint32_t)LT_TAG_EOMI : (uint32_t)LT_NO_TAG) << 24),
                           LT_NO_RULE, split | (flags << 16));
            E.hkey[slot] = hit_key(e, b, lemma ? 1u : 0u, split, k, pass);
            E.htask[slot] = task;
        }
        ++slot;
    }
    const uint32_t common = (uint32_t)b | ((uint32_t)p << 12) | (is_l ? 1u << 27 : 0u) | (pass << 29);
    const uint32_t ytask = (uint32_t)e | (task << 12);
    uint32_t qs = cur_q + (incl >> 16) - np_mine;
    if (c1) E.rq[qs++] = make_uint4(common | (0u << 24) | (1u << 26), ytask, 1u | (c1 << 19), r1.x);
    if (cf) E.rq[qs++] = make_uint4(common | ((last ? 2u : 1u) << 24) | (1u << 28), ytask, after1 | (cf << 19), rf.x);
    if (cs) E.rq[qs++] = make_uint4(common | (1u << 24) | (1u << 28), ytask, (after1 + cf) | (cs << 19), rs.x);
    __syncwarp();
    return ncand;
}

// Write the staged survivors to HBM in rank order (ord[r] = staging slot of the record with rank r): consecutive
// lanes write consecutive edge records; CSR bookkeeping in shared memory.
__device__ LT_FLUSH_ATTR void flush_staged(const LatticeArgs& A, int lane, uint32_t alive, const uint32_t* ord, const lt_edge* hrec,
                                          uint32_t* pcnt, uint32_t* pstart, uint32_t* nh) {
    if (alive > 0) {
        unsigned long long gbase64 = 0;
        if (lane == 0) gbase64 = atomicAdd(A.cursor, (unsigned long long)alive);
        gbase64 = __shfl_sync(kFull, gbase64, 0);
        const bool fits = gbase64 + alive <= (unsigned long long)A.edge_cap;
        const uint32_t gbase = (uint32_t)gbase64;      // exact whenever it is used (edge_cap < 2^32)
        if (!fits && lane == 0) atomicOr(A.flags + kFlagEdgeOverflow, 1u);
        #pragma unroll 1
        for (uint32_t r = lane; r < alive; r += 32) {
            const lt_edge rec = hrec[ord[r]];
            if (fits) A.edges[gbase + r] = rec;
            atomicAdd(&pcnt[rec.e - 1], 1u);
            atomicMin(&pstart[rec.e - 1], gbase + r);
        }
    }
    __syncwarp();
    if (lane == 0) *nh = 0;
    __syncwarp();
}

// Rank of an eojeol's survivors by sort key.  Staged entries [first, first + H) hold keys (dead ones ~0) and records;
// afterwards ord[alive .. alive + n_alive) lists the staging slots of the survivors in key order (`ord` is the task-id
// array, whose contents are dead once the split filter has run; ord[0, alive) belongs to earlier eojeols).
//   small eojeols (in the kernel): every entry counts the keys below its own (H^2 / 32 shared-memory reads per lane);
//   larger ones (here): bitonic sort of (key, slot) pairs in place, padded to P = a power of two with dead keys — taken
//                  when the padding fits the staging area (a 1 000-hit eojeol ranks in ~14 k warp instructions instead
//                  of ~160 k; the counting loop was 12 % of C3's main pass and most of its retry pass).
constexpr int kSortMin = 160;               // entries from which the sort pays (C3 sample, r3i: 48 / 96 / 160 -> lattice 1.859 / 1.836 / 1.829 ms) (LatticeArgs::sort_min; LT_SORT_MIN overrides)
#ifndef LT_RANK_UNROLL
#define LT_RANK_UNROLL 4
#endif
constexpr int kRankUnroll = LT_RANK_UNROLL;
__device__ __noinline__ void rank_by_sort(uint64_t* hkey, uint32_t* ord, uint32_t first, uint32_t H, uint32_t P, uint32_t alive,
                                          uint32_t n_alive, int lane) {
    for (uint32_t i = lane; i < P; i += 32) {
        if (i >= H) hkey[first + i] = ~0ull;
        ord[first + i] = first + i;
    }
    __syncwarp();
    uint64_t* key = hkey + first;
    uint32_t* pay = ord + first;
    for (uint32_t k = 2; k <= P; k <<= 1) {
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            #pragma unroll 2
            for (uint32_t t = lane; t < P / 2; t += 32) {
                const uint32_t i = ((t & ~(j - 1u)) << 1) | (t & (j - 1u));      // bit j clear
                const uint32_t q = i | j;
                const uint64_t a = key[i], b = key[q];
                const bool ascending = (i & k) == 0;
                if ((a > b) == ascending) {
                    key[i] = b; key[q] = a;
                    const uint32_t pa = pay[i], pb = pay[q];
                    pay[i] = pb; pay[q] = pa;
                }
            }
            __syncwarp();
        }
    }
    // survivors first, in key order: their slots move down to ord[alive ..) (never above where they were read)
    for (uint32_t base = 0; base < n_alive; base += 32) {
        const uint32_t r = base + lane;
        const uint32_t src = (r < n_alive) ? pay[r] : 0u;
        __syncwarp();
        if (r < n_alive) ord[alive + r] = src;
        __syncwarp();
    }
}

// ---- the kernel -----------------------------------------------------------------------------------

#ifndef LT_LAT_MINB
#define LT_LAT_MINB 2
#endif
constexpr int lattice_max_threads(int, int, int) { return kLatMaxWarps * 32; }      // (register caps for more resident CTAs
constexpr int lattice_min_blocks(int, int, int) { return LT_LAT_MINB; }              // spill and lose: profiles/README.md, r2d)
// UC / HCT: sentence-array size and staging capacity when known at compile time (0 = A.units / A.hcap)
// LM: 0 = MorphemeLookup only (what Tagger.tag uses; the other lookups compile out of the throughput path),
//     1 = the lookup named by A.mode.
// RP: 1 = the retry pass (one eojeol per work item); the main-pass instantiations carry none of its code.
template <int UC, int HCT, int LM = 0, int RP = 0>
__global__ void __launch_bounds__(lattice_max_threads(UC, HCT, LM), lattice_min_blocks(UC, HCT, LM)) lattice_kernel(const __grid_constant__ DevTables T,
                                                                const __grid_constant__ LatticeArgs A) {
    LT_DYN_SMEM(smem_raw);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int units = UC ? UC : A.units;
    const int HC = HCT ? HCT : A.hcap;
    const int DM = A.max_str;
    unsigned char* base = smem_raw + (size_t)warp * lattice_warp_smem(units, HC, DM);
    const LatticeViews W = lattice_views<UC, HCT>(base, units, HC, DM);
    uint64_t* ha = W.ha;
    uint64_t* hb = W.hb;
    uint2* rref = W.rref;
    uint64_t* hkey = W.E.hkey;
    lt_edge* hrec = W.E.hrec;
    uint32_t* htask = W.E.htask;
    uint32_t* pstart = W.pstart;
    uint32_t* pcnt = W.pcnt;
    uint32_t* tcnt = W.E.tcnt;
    uint16_t* ch = W.ch;
    uint16_t* eoj = W.eoj;
    uint8_t* nend = W.nend;
    uint32_t* nh = W.E.nh;
    uint32_t* rqn = W.E.rqn;
    uint32_t* sub = const_cast<uint32_t*>(W.E.sub);

    unsigned long long acc_L = 0, acc_P = 0, acc_E = 0;

    while (true) {
        unsigned int s = 0;
        if (lane == 0) s = atomicAdd(A.queue, 1u);
        s = __shfl_sync(kFull, s, 0);
        int w_first = 0, w_count = 0x7FFFFFFF;       // eojeols of the sentence this warp enumerates
        if (RP != 0) {
            if (s >= *A.retry_count) break;
            const uint2 item = A.retry_list[s];
            s = item.x;
            w_first = (int)item.y;
            w_count = 1;
        } else {
            if (s >= (unsigned)A.n_sent) break;
            if (A.order) s = __ldg(A.order + s);
        }
        const int s0 = __ldg(A.sent_off + s), s1 = __ldg(A.sent_off + s + 1);
        if (s1 - s0 > A.max_units) {
            // longer than the per-warp arrays hold: the sentence gets a status of its own, the batch goes on
            #pragma unroll 1
            for (int p = lane; p < s1 - s0; p += 32) A.pos[s0 + p] = make_uint2(0u, 0u);
            if (lane == 0) {
                A.sent_len[s] = 0;
                A.sent_edges[s] = 0;
                A.status[s] = LT_SENT_TOO_LONG;
            }
            __syncwarp();
            continue;
        }
        int n_eoj;
        bool bad;
        const int L = stage_sentence(A.text, s0, s1, lane, ch, eoj, ha, hb, n_eoj, bad);
        const SentView v = W.v;
        const Enum E = W.E;

        // conjugation-rule lists of the keys starting at every syllable
        for (int p = lane; p < L; p += 32) {
            uint32_t c0 = ch[p], c1 = (p + 1 < L) ? ch[p + 1] : 0u, c2 = (p + 2 < L) ? ch[p + 2] : 0u;
            // (keys past the sentence end are probed too — c1 / c2 are 0 there — and discarded)
            const uint64_t k1 = rule_key(c0, 0, 0, 1), k2 = rule_key(c0, c1, 0, 2), k3 = rule_key(c0, c1, c2, 3);
            uint2 r1 = make_uint2(0u, 0u), r2 = r1, r3 = r1;
            if (T.has_rules) {
                const RuleProbe q1 = rule_first(T, k1), q2 = rule_first(T, k2), q3 = rule_first(T, k3);
                r1 = rule_resolve(q1, k1);
                if (p + 1 < L) r2 = rule_resolve(q2, k2);
                if (p + 2 < L) r3 = rule_resolve(q3, k3);
            }
            rref[3 * p + 0] = r1;
            rref[3 * p + 1] = r2;
            rref[3 * p + 2] = r3;
        }
        // substring table: every substring of at most max_str syllables, one wave of probes
        const float inv_dm = small_rcp(DM);
        for (int q = lane; q < L * DM; q += 32) {
            const int x = small_div(q, DM, inv_dm), len = q - x * DM + 1;
            uint32_t payload = 0;
            if (x + len <= L) {
                const uint64_t pl = dict_probe(T, sub_hash(T, v, x, x + len), (uint32_t)len);
                payload = ((uint32_t)pl & kSubTagMask) | (((uint32_t)(pl >> 32) & 7u) << 29);
            }
            sub[q] = payload;
        }
        #pragma unroll 1
        for (int p = lane; p < s1 - s0; p += 32) { pstart[p] = 0xFFFFFFFFu; pcnt[p] = 0; }
        if (lane == 0) { *nh = 0; *rqn = 0; }
        __syncwarp();

        uint32_t ncand = 0;      // lemma candidates the reference generates (lane-local)
        uint32_t nsub = 0;       // distinct substrings examined (lane 0 only)
        uint32_t slots = 0;      // staged entries, dead ones included (warp-uniform copy of *nh)
        uint32_t alive = 0;      // staged entries that survive = next free rank (warp-uniform)
        uint32_t sent_total = 0;
        bool overflow = false;

        auto flush = [&]() {
            flush_staged(A, lane, alive, htask, hrec, pcnt, pstart, nh);
            slots = 0;
            alive = 0;
        };

        const int mode = LM ? A.mode : LT_LOOKUP_MORPHEME;
        const bool word_mode = LM && mode >= LT_LOOKUP_WORD;
        const int w_end = (w_count < n_eoj - w_first) ? w_first + w_count : n_eoj;
        for (int w = w_first; w < w_end && !overflow; ++w) {
            const int o = eoj[w];
            const int n = eoj[w + 1] - o;
            const int oe = o + n;
            for (int attempt = 0; attempt < 2; ++attempt) {
                // ---------------- stage 1: whole eojeol + every left/right split ----------------
                #pragma unroll 1
                for (int u = lane; u < 2 * n; u += 32) tcnt[u] = 0;
                __syncwarp();
                uint32_t ncand_try = 0;
                const float inv_n = small_rcp(n);
                // (word_lookup starts with the whole-eojeol lookup alone: the items of task 0, lookup.py:157)
                const int n_items1 = word_mode ? n : n * n;
                // (the passes run in an inner loop without any call; it is left for drain_rules when the queue fills up
                // and when the items are done)
                for (int q0 = 0; q0 < n_items1;) {
                  for (bool room = true; room && q0 < n_items1; q0 += 32) {
                    const int q = q0 + lane;
                    {
                        const bool valid = q < n_items1;
                        const int qq = valid ? q : 0;
                        const int i = small_div(qq, n, inv_n), r = qq - i * n;
                        const int p = o + r;
                        // task: i == 0 whole; r < i: left_i = [o, o+i); else right_i = [o+i, oe)
                        const bool left = (i > 0) && (r < i);
                        const int b = (i > 0 && !left) ? o + i : o;
                        const int e = left ? o + i : oe;
                        const uint32_t task = (i == 0) ? 0u : (left ? 2u * i : 2u * i + 1u);
                        // Noun + Josa special case: both edges carry len = n and nothing else is looked up (lookup.py:200-203)
                        const bool special = (i > 0) && ((sub_get(E, o, o + i) >> LT_TAG_NOUN) & 1u) && ((sub_get(E, o + i, oe) >> LT_TAG_JOSA) & 1u);
                        // the task's first item also reports its tag hits: one per tag of the string, in the dictionary's
                        // tag order (get_tags, dictionary.py:238-242)
                        uint32_t tagbits = 0;
                        if (p == b) tagbits = special ? (left ? 1u << LT_TAG_NOUN : 1u << LT_TAG_JOSA) : (sub_get(E, b, e) & kSubTagMask & T.order_mask);
                        ncand_try += emit_pass<UC, HCT>(T, v, E, base, units, lane, valid, b, e, p, task, b == o, tagbits, special ? (uint32_t)n : (uint32_t)(e - b),
                                               special ? left : (b == o), special ? 0ull : ~0ull, !special, 0u);
                    }
                    // (read by one lane between two barriers: a lane that ran ahead into the next pass must not be able
                    // to change what the others see here)
                    room = warp_read(rqn) <= (uint32_t)kRuleDrainAt;      // a pass queues at most 3 per lane
                  }
                  drain_rules<UC, HCT>(T, base, units, HC, DM, lane);
                }
                // ---- a split survives only when both sides found something (lookup.py:205-209) ----
                uint32_t nstaged = *nh;
                bool too_many = nstaged > (uint32_t)HC;
                uint32_t alive_here = 0;
                if (!too_many) {
                    // LRLookup(prefer_exact_match=True) returns the whole-eojeol analyses alone when there are any (lookup.py:192-193)
                    const bool exact_only = (mode == LT_LOOKUP_LR) && (tcnt[0] > 0);
                    for (uint32_t h = slots + lane; h < nstaged; h += 32) {
                        const uint32_t task = htask[h];
                        bool ok = true;
                        if (task >= 2) ok = (tcnt[task] > 0) && (tcnt[task ^ 1u] > 0) && !exact_only;
                        if (!ok) hkey[h] = ~0ull;
                        alive_here += ok ? 1u : 0u;
                    }
                    #pragma unroll
                    for (int d = 16; d; d >>= 1) alive_here += __shfl_xor_sync(kFull, alive_here, d);
                }
                uint32_t nsub_try = (uint32_t)(2 * n - 1);
                // second stage of the lookup:
                //   MorphemeLookup: sub-word scan when the first stage found nothing, begins from 1 (lookup.py:259-277)
                //   WordLookup: every substring's full lookup, begins from 0 (lookup.py:161-168) — when the whole
                //               eojeol is unknown, or always without prefer_exact_match (the whole-eojeol hits stay)
                //   LRLookup: none
                const bool scan = !too_many && mode != LT_LOOKUP_EXACT &&
                                  (word_mode ? (mode == LT_LOOKUP_WORD_ALL || alive_here == 0)
                                                          : (mode == LT_LOOKUP_MORPHEME && alive_here == 0 && n >= 2));
                if (scan) {
                    __syncwarp();
                    const uint32_t pass = word_mode ? 1u : 0u;
                    if (lane == 0 && !word_mode) *nh = slots;          // forget the dead stage-1 hits
                    const int M = word_mode ? n : ((T.max_len > 0) ? T.max_len : n);
                    const int bl0 = word_mode ? 0 : 1;
                    // which positions end a stand-alone Noun found by this scan
                    if (!word_mode) {
                        #pragma unroll 1
                        for (int el = 1 + lane; el <= n; el += 32) {
                            bool any_noun = false;
                            int b_lo = el - M; if (b_lo < 1) b_lo = 1;
                            #pragma unroll 1
                            for (int bl = b_lo; bl < el; ++bl) any_noun |= ((sub_get(E, o + bl, o + el) >> LT_TAG_NOUN) & 1u) != 0;
                            nend[o + el] = any_noun ? 1 : 0;
                        }
                    }
                    if (lane == 0) tcnt[0] = 0;
                    __syncwarp();
                    const int tri = M * (M + 1) / 2;
                    const int items = (n - bl0) * tri;
                    const float inv_tri = small_rcp(tri);
                    // stand-alone tags in list order (lookup.py:104-105), then Josa after a Noun
                    constexpr uint32_t standalone_tags = (1u << LT_TAG_NOUN) | (1u << LT_TAG_ADVERB) | (1u << LT_TAG_EXCLAMATION) |
                                                         (1u << LT_TAG_DETERMINER) | (1u << LT_TAG_NUMBER);
                    constexpr uint64_t standalone_order = (0ull << (4 * LT_TAG_NOUN)) | (1ull << (4 * LT_TAG_ADVERB)) |
                                                          (2ull << (4 * LT_TAG_EXCLAMATION)) | (3ull << (4 * LT_TAG_DETERMINER)) |
                                                          (4ull << (4 * LT_TAG_NUMBER)) | (5ull << (4 * LT_TAG_JOSA));
                    for (int q0 = 0; q0 < items;) {
                      for (bool room = true; room && q0 < items; q0 += 32) {
                        const int q = q0 + lane;
                        {
                            const bool in_range = q < items;
                            const int qq = in_range ? q : 0;
                            const int blq = small_div(qq, tri, inv_tri);
                            const int bl = bl0 + blq;
                            int t = qq - blq * tri;
                            // t -> (span, split offset inside the span): span (span - 1) / 2 <= t < span (span + 1) / 2
                            int span = (int)((1.0f + approx_sqrt(8.0f * (float)t + 1.0f)) * 0.5f);
                            span -= (span * (span - 1) / 2 > t) ? 1 : 0;
                            span += (span * (span + 1) / 2 <= t) ? 1 : 0;
                            t -= span * (span - 1) / 2;
                            const bool valid = in_range && (bl + span <= n);
                            const int b = o + bl, e = valid ? b + span : b + 1, p = valid ? b + t : b;
                            uint32_t tagbits = 0;
                            if (valid && t == 0) {
                                const uint32_t m = sub_get(E, b, e);
                                // WordLookup: MorphemeDictionary.lookup of the substring, one hit per tag in dictionary order;
                                // MorphemeLookup: the stand-alone tags, and Josa right after a Noun found by this scan
                                tagbits = word_mode ? (m & kSubTagMask & T.order_mask)
                                                    : ((m & standalone_tags) | ((nend[b] && ((m >> LT_TAG_JOSA) & 1u)) ? 1u << LT_TAG_JOSA : 0u));
                            }
                            const bool first = word_mode && bl == 0;
                            ncand_try += emit_pass<UC, HCT>(T, v, E, base, units, lane, valid, b, e, p, 0u, first, tagbits, (uint32_t)span, first,
                                                   word_mode ? ~0ull : standalone_order, true, pass);
                        }
                        room = warp_read(rqn) <= (uint32_t)kRuleDrainAt;
                      }
                      drain_rules<UC, HCT>(T, base, units, HC, DM, lane);
                    }
                    nstaged = *nh;
                    too_many = nstaged > (uint32_t)HC;
                    alive_here = nstaged - slots;             // every stage-2 hit survives
                    // pairs (b, e), 1 <= b < e <= min(b+M, n), minus the (b, n) already examined by stage 1
                    // sum_{bl=1}^{n-1} min(M, n - bl) in closed form
                    const int m1 = min(M, n - 1);
                    const uint32_t pairs = (uint32_t)(m1 * (m1 + 1) / 2 + (n - 1 - m1) * M);
                    nsub_try += pairs - (uint32_t)m1;
                }
                if (too_many) {
                    // the eojeol alone may fit once the staged edges of earlier eojeols are written out
                    __syncwarp();
                    if (lane == 0) *nh = slots;
                    __syncwarp();
                    if (attempt == 0 && slots > 0) { flush(); continue; }
                    if (RP == 0 && A.retry_list != nullptr) {
                        // this eojeol alone goes to the retry pass; the sentence's other eojeols are done here
                        if (lane == 0) A.retry_list[atomicAdd(A.retry_count, 1u)] = make_uint2(s, (uint32_t)w);
                        __syncwarp();
                        break;
                    }
                    overflow = true;
                    break;
                }
                ncand += ncand_try;
                if (lane == 0) nsub += nsub_try;
                // ---- final position of every survivor: rank of its key among the eojeol's survivors ----
                __syncwarp();
                {
                    const uint32_t H = nstaged - slots;
                    uint32_t P = 0;                      // padded size when the eojeol is ranked by sorting
                    // (the instantiation for short sentences with the small staging area goes without: the call alone costs
                    // it 1.5 % and its eojeols hardly ever reach the threshold; LT_SORT_MIN does not apply there)
                    constexpr bool kCanSort = !(UC == 64 && HCT == kLatDefaultHcap);
                    if (kCanSort && H >= (uint32_t)A.sort_min) {
                        P = 32;
                        while (P < H) P <<= 1;
                        if (slots + P > (uint32_t)HC) P = 0;
                    }
                    if (kCanSort && P) {
                        rank_by_sort(hkey, htask, slots, H, P, alive, alive_here, lane);
                    } else {
                        for (uint32_t h = slots + lane; h < nstaged; h += 32) {
                            const uint64_t key = hkey[h];
                            if (key != ~0ull) {
                                uint32_t rank = alive;
                                #pragma unroll kRankUnroll
                                for (uint32_t g = slots; g < nstaged; ++g) rank += (hkey[g] < key) ? 1u : 0u;
                                htask[rank] = h;        // (task ids are dead by now: a rank slot may be any entry of this eojeol)
                            }
                        }
                    }
                }
                slots = nstaged;
                alive += alive_here;
                sent_total += alive_here;
                __syncwarp();
                break;
            }
        }
        if (overflow) {
            if (lane == 0) atomicOr(A.flags + kFlagStageOverflow, 1u);
        } else {
            flush();
        }
        __syncwarp();
        #pragma unroll
        for (int d = 16; d; d >>= 1) ncand += __shfl_xor_sync(kFull, ncand, d);
        if constexpr (RP != 0) {
            // one eojeol of a sentence the main pass has otherwise finished: its positions, its edges, its share of
            // the work counters; a sentence that had no edge without it gets its status back
            const int o = (w_first < n_eoj) ? eoj[w_first] : 0, oe = (w_first < n_eoj) ? eoj[w_first + 1] : 0;
            #pragma unroll 1
            for (int p = o + lane; p < oe; p += 32) {
                const uint32_t c = pcnt[p];
                A.pos[s0 + p] = make_uint2(c ? pstart[p] : 0u, c);
            }
            if (lane == 0) {
                if (sent_total > 0) {
                    atomicAdd(A.sent_edges + s, (int32_t)sent_total);
                    atomicCAS(A.status + s, (int32_t)LT_SENT_NO_EDGES, (int32_t)LT_SENT_OK);
                }
                acc_P += (unsigned long long)nsub + 2ull * ncand;
                acc_E += sent_total;
            }
            __syncwarp();
        } else {
            #pragma unroll 1
            for (int p = lane; p < s1 - s0; p += 32) {
                const uint32_t c = pcnt[p];
                A.pos[s0 + p] = make_uint2(c ? pstart[p] : 0u, c);
            }
            if (lane == 0) {
                A.sent_len[s] = L;
                A.sent_edges[s] = (int32_t)sent_total;
                int st = LT_SENT_OK;
                if (bad) st = LT_SENT_BAD_SPACE;
                else if (L > 0 && sent_total == 0) st = LT_SENT_NO_EDGES;
                A.status[s] = st;
                acc_L += (unsigned long long)L;
                acc_P += (unsigned long long)nsub + 2ull * ncand;
                acc_E += sent_total;
            }
            __syncwarp();
        }
    }
    if (lane == 0) {
        atomicAdd(A.counters + 0, acc_L);
        atomicAdd(A.counters + 1, acc_P);
        atomicAdd(A.counters + 2, acc_E);
    }
}

}  // namespace lt
