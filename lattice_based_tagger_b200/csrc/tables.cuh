// tables.cuh — layout of the device-resident tables and the probe routines the kernels use.
//
// HBM layout (all built once by lt_tables_create, read-only afterwards):
//   dict   cuckoo table (two slots per key), 16 B slots {fp, tagmask, lemma bits}; key = (string, length)
//   rules  cuckoo table, 16 B slots {exact 1..3-syllable key, first rule, count|k3_first}
//   rrec   one 48 B record per (stem, eomi) rule: hashes and lengths of both strings
//   feat   cuckoo table (two slots per key), 16 B slots {fp, fp64 weight}; key = feature tuple / preference
//   dense  per trigram scorer: tag x tag matrix (template 3), length vectors (templates 4, 6)
//          with presence masks — staged into shared memory by the beam kernel
//   pows   base^n pairs for composing polynomial hashes
#pragma once
#include "cuda_compat.cuh"
#include <stdint.h>

#include "../../include/lt_b200.h"
#include "hash.cuh"

namespace lt {

struct DictSlot {
    uint64_t fp;        // 0 = empty
    uint32_t tagmask;   // bit t: string is in tag t's set
    uint32_t lemma;     // bit0 verbs, bit1 adjectives, bit2 eomis
};
static_assert(sizeof(DictSlot) == 16, "DictSlot");

constexpr uint32_t kLemVerb = 1u, kLemAdj = 2u, kLemEomi = 4u;

struct RuleSlot {
    uint64_t key;       // rule_key(); 0 = empty (len field is never 0 for a real key)
    uint32_t first;     // index of the key's first rule record
    uint32_t count;     // low 16 bits: number of rules; bit 31: k3_first
};
static_assert(sizeof(RuleSlot) == 16, "RuleSlot");

struct alignas(16) RuleRec {
    H2 stem, eomi;
    uint32_t stem_len, eomi_len;
    uint64_t pad;
};
static_assert(sizeof(RuleRec) == 48, "RuleRec");

struct FeatSlot {
    uint64_t fp;        // 0 = empty
    double w;
};
static_assert(sizeof(FeatSlot) == 16, "FeatSlot");

constexpr int kT4Dense = 64;   // template-4 lengths below this are looked up densely

// Dense block of one trigram scorer, in doubles, for n_tags = NT:
//   [0, NT*NT)            template 3 weights, row = tj, col = tk
//   [NT*NT, +kT4Dense)    template 4 weights by len
//   [.., +16)             template 6 weights by min(8, len) (0..8 used)
// followed (as raw 32-bit words, 2 per double slot) by presence masks:
//   NT words   template 3 row masks (bit tk)
//   2 words    template 4 presence (bits 0..63)
//   1 word     template 6 presence (bits 0..8)
__host__ __device__ inline int dense_doubles(int nt) { return nt * nt + kT4Dense + 16; }
__host__ __device__ inline int dense_mask_words(int nt) { return nt + 3; }
__host__ __device__ inline int dense_block_bytes(int nt) {
    return (dense_doubles(nt) * 8 + dense_mask_words(nt) * 4 + 7) & ~7;
}

struct DevTables {
    const DictSlot* dict;
    uint64_t dict_mask;
    uint32_t dict_bits;           // log2(slots)
    uint32_t reserved3;
    const RuleSlot* rules;
    uint32_t rule_bits;           // log2(slots)
    uint32_t reserved4;
    const RuleRec* rrec;
    const FeatSlot* feat;
    uint64_t feat_mask;
    uint32_t feat_bits;           // log2(slots)
    uint32_t reserved2;
    const unsigned char* dense;   // n_tri blocks of dense_block_bytes(n_tags)
    const H2* pows;
    int32_t n_pows;
    int32_t n_tags;
    int32_t n_tag_order;
    int32_t max_len;
    int32_t n_funcs;
    int32_t n_tri;                // number of LT_FUNC_TRIGRAM scorers
    int32_t has_rules;
    int32_t max_str;              // longest dictionary string (syllables)
    uint8_t tag_order[LT_MAX_TAGS];
    uint8_t tag_pos[32];           // position of a tag id in tag_order (the emission order of a string's tags)
    uint32_t order_mask;           // tag ids that appear in tag_order
    lt_func funcs[LT_MAX_FUNCS];
    int8_t  func_dense[LT_MAX_FUNCS];   // dense block index of a trigram scorer, -1 otherwise
    H2 bos;                        // hash of the literal 'BOS' (beam.py:21)
    H2 seeds[LT_MAX_FUNCS][10];    // feature_seed(template 0..8, f); [9] = the scorer's preference kind
};

#if defined(LT_DEVICE_CODE)

__device__ __forceinline__ uint4 ldg16(const void* p) {
    return __ldg(reinterpret_cast<const uint4*>(p));
}

// dictionary probe, split so that callers can put several probes in flight: both slots of the key
// are loaded at once; the payload is (tagmask | lemma << 32), 0 when absent
struct DictProbe {
    uint4 s, t;
};
__device__ __forceinline__ DictProbe dict_first(const DevTables& T, H2 h, uint32_t len) {
    const uint64_t x = dict_slot_hash(h, len);
    DictProbe p;
    p.s = ldg16(T.dict + cuckoo_slot1(x, T.dict_bits));
    p.t = ldg16(T.dict + cuckoo_slot2(x, T.dict_bits));
    return p;
}
__device__ __forceinline__ uint64_t dict_resolve(const DictProbe& p, H2 h, uint32_t len) {
    const uint64_t fp = dict_fp(h, len);
    const uint32_t flo = (uint32_t)fp, fhi = (uint32_t)(fp >> 32);
    if (p.s.x == flo && p.s.y == fhi) return (uint64_t)p.s.z | ((uint64_t)p.s.w << 32);
    if (p.t.x == flo && p.t.y == fhi) return (uint64_t)p.t.z | ((uint64_t)p.t.w << 32);
    return 0;
}
__device__ __forceinline__ uint64_t dict_probe(const DevTables& T, H2 h, uint32_t len) {
    return dict_resolve(dict_first(T, h, len), h, len);
}

// rule probe: (first, count|flag) of an exact 1..3 syllable key; count = 0 when absent (cuckoo table)
struct RuleProbe {
    uint4 s, t;
};
__device__ __forceinline__ RuleProbe rule_first(const DevTables& T, uint64_t key) {
    const uint64_t x = fmix64(key);
    RuleProbe p;
    p.s = ldg16(T.rules + cuckoo_slot1(x, T.rule_bits));
    p.t = ldg16(T.rules + cuckoo_slot2(x, T.rule_bits));
    return p;
}
__device__ __forceinline__ uint2 rule_resolve(const RuleProbe& p, uint64_t key) {
    const uint32_t klo = (uint32_t)key, khi = (uint32_t)(key >> 32);
    if (p.s.x == klo && p.s.y == khi) return make_uint2(p.s.z, p.s.w);
    if (p.t.x == klo && p.t.y == khi) return make_uint2(p.t.z, p.t.w);
    return make_uint2(0u, 0u);
}

__device__ __forceinline__ RuleRec rule_load(const DevTables& T, uint32_t idx) {
    const uint4* p = reinterpret_cast<const uint4*>(T.rrec + idx);
    const uint4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
    RuleRec r;
    r.stem.a = (uint64_t)a.x | ((uint64_t)a.y << 32);
    r.stem.b = (uint64_t)a.z | ((uint64_t)a.w << 32);
    r.eomi.a = (uint64_t)b.x | ((uint64_t)b.y << 32);
    r.eomi.b = (uint64_t)b.z | ((uint64_t)b.w << 32);
    r.stem_len = c.x;
    r.eomi_len = c.y;
    r.pad = 0;
    return r;
}

// feature probe, split in two so that callers can put the loads of several probes in flight
struct FeatProbe {
    uint4 s, t;     // the key's two slots
};
__device__ __forceinline__ FeatProbe feat_first(const DevTables& T, FKey k) {
    FeatProbe p;
    const uint64_t x = feature_slot_hash(k.k1);
    p.s = ldg16(T.feat + cuckoo_slot1(x, T.feat_bits));
    p.t = ldg16(T.feat + cuckoo_slot2(x, T.feat_bits));
    return p;
}
__device__ __forceinline__ bool feat_resolve(const DevTables& T, FKey k, FeatProbe p, double& w) {
    const uint32_t flo = (uint32_t)k.k2, fhi = (uint32_t)(k.k2 >> 32);
    const bool in_s = (p.s.x == flo) && (p.s.y == fhi);
    const bool in_t = (p.t.x == flo) && (p.t.y == fhi);
    if (in_s || in_t) w = __hiloint2double((int)(in_s ? p.s.w : p.t.w), (int)(in_s ? p.s.z : p.t.z));   // a miss leaves w alone
    return in_s || in_t;
}
// the slot that holds key k, for a probe feat_resolve found (the slot whose weight it took)
__device__ __forceinline__ uint32_t feat_hit_slot(const DevTables& T, FKey k, const FeatProbe& p) {
    const uint64_t x = feature_slot_hash(k.k1);
    const bool in_s = (p.s.x == (uint32_t)k.k2) && (p.s.y == (uint32_t)(k.k2 >> 32));
    return (uint32_t)(in_s ? cuckoo_slot1(x, T.feat_bits) : cuckoo_slot2(x, T.feat_bits));
}

__device__ __forceinline__ H2 pow_at(const DevTables& T, uint32_t n) {
    const uint64_t* p = reinterpret_cast<const uint64_t*>(T.pows + n);
    return H2{__ldg(p), __ldg(p + 1)};
}

#endif  // __CUDACC__

}  // namespace lt
