// lt_b200.cu — C ABI (include/lt_b200.h): host-side table compiler, batch workspace, launches.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -shared
//        -Xcompiler -fPIC  (see __graft_entry__.build()).  -fmad=false keeps every fp64
// multiply and add of the score arithmetic separately rounded, as in the reference's Python.
#include "cuda_compat.cuh"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/lt_b200.h"
#include "beam.cuh"
#include "constraints.cuh"
#include "evaluate.cuh"
#include "hash.cuh"
#include "lattice.cuh"
#include "paths.cuh"
#include "scan.cuh"
#include "tables.cuh"
#include "train.cuh"
#include "violation.cuh"

using namespace lt;

static constexpr uint32_t kDstNone = 0xFFFFFFFFu, kDstDense = 0x80000000u;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_error;

static int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

#define CU(call)                                                                                  \
    do {                                                                                          \
        cudaError_t _e = (call);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return fail(LT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

extern "C" const char* lt_last_error(void) { return g_error.c_str(); }
extern "C" int lt_abi_version(void) { return LT_ABI_VERSION; }

// ------------------------------------------------------------------------------------------------
// tables
// ------------------------------------------------------------------------------------------------
// Every entry point runs on the tables' device and puts the caller's current device back on return.
struct DeviceGuard {
    int prev = -1, dev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device) : dev(device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
};
#define ON_DEVICE(device)                                                                         \
    DeviceGuard _guard(device);                                                                   \
    if (_guard.err != cudaSuccess) return fail(LT_ERR_CUDA, "cudaSetDevice(%d) failed: %s", (int)(device), cudaGetErrorString(_guard.err))

// A device buffer that frees itself; grown by ensure().
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
};

static int ensure(DevBuf& b, size_t bytes) {
    if (bytes <= b.cap) return LT_OK;
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        e = cudaMalloc(&b.p, bytes);
        want = bytes;
    }
    if (e != cudaSuccess) return fail(LT_ERR_CUDA, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    b.cap = want;
    return LT_OK;
}

// Data uploaded once: a buffer of exactly `bytes` (at least 16, so that it is never null) and no slack behind it.
static int upload_once(DevBuf& b, const void* src, size_t bytes) {
    CU(cudaMalloc(&b.p, std::max<size_t>(bytes, 16)));
    b.cap = std::max<size_t>(bytes, 16);
    if (bytes) CU(cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice));
    return LT_OK;
}

struct lt_tables {
    int device = 0;
    DevTables dev{};
    std::vector<void*> allocations;
    int64_t bytes = 0;
    int sm_count = 0;
    // where the weight of input feature i lives (lt_tables_update_weights): a slot of the hashed table, an offset into
    // the dense blocks (kDstDense | byte offset / 8), or kDstNone for a feature no tuple can equal
    std::vector<uint32_t> feat_dst;
    std::vector<uint8_t> feat_func;                    // owning scorer of input feature i (lt_trainer_create's check)
    std::vector<unsigned char> dense_host;
    DevBuf d_feat_dst, d_weights;
    // path sets (paths.cuh): a feature hit is a slot of the hashed table or feat_slots + a dense offset; per hit the
    // desc index of its feature, and the perceptron's count per hit — both made on first use
    DevBuf d_hit_feat, d_counts;
};

static H2 hash_units(const uint16_t* p, int64_t n) {
    H2 h{0, 0};
    for (int64_t i = 0; i < n; ++i) h = h2_push(h, p[i]);
    return h;
}

static uint64_t next_pow2(uint64_t x) {
    uint64_t p = 16;
    while (p < x) p <<= 1;
    return p;
}

// Cuckoo table builder (two slots per key, one entry per slot).  An item is identified by its slot
// hash x and its fingerprint; two items equal in both are a 128-bit collision (or a repeated key).
// Placement is the usual random walk: take a free slot of the two, else evict the occupant of the
// slot the walk did not just come from and re-place that one; a walk that does not end doubles the table.
struct CuckooItem {
    uint64_t x, fp, payload;
};
struct CuckooSlot {
    uint64_t fp, payload;
};
static int build_cuckoo(const std::vector<CuckooItem>& items, uint64_t min_slots, std::vector<CuckooSlot>* table,
                        uint32_t* bits_out, const char* what, std::vector<uint32_t>* slot_of = nullptr) {
    uint32_t bits = 4;
    while ((1ull << bits) < min_slots) ++bits;
    for (const CuckooItem& it : items)
        if (it.fp == 0) return fail(LT_ERR_COLLISION, "one of the %s hashes to the reserved fingerprint 0", what);
    for (; bits <= 32; ++bits) {
        const uint64_t slots = 1ull << bits;
        std::vector<int64_t> owner(slots, -1);
        bool placed_all = true;
        for (int64_t idx = 0; idx < (int64_t)items.size() && placed_all; ++idx) {
            const uint64_t a0 = cuckoo_slot1(items[idx].x, bits), b0 = cuckoo_slot2(items[idx].x, bits);
            for (uint64_t sl : {a0, b0}) {
                const int64_t o = owner[sl];
                if (o >= 0 && items[o].x == items[idx].x && items[o].fp == items[idx].fp)
                    return fail(LT_ERR_COLLISION, "two %s share the 128-bit hash (or one was given twice)", what);
            }
            int64_t cur = idx;
            uint64_t from = ~0ull;
            bool placed = false;
            for (int kick = 0; kick < 2000; ++kick) {
                const uint64_t a = cuckoo_slot1(items[cur].x, bits), b = cuckoo_slot2(items[cur].x, bits);
                if (owner[a] < 0) { owner[a] = cur; placed = true; break; }
                if (owner[b] < 0) { owner[b] = cur; placed = true; break; }
                const uint64_t v = (a == from) ? b : a;
                std::swap(cur, owner[v]);
                from = v;
            }
            placed_all = placed;
        }
        if (!placed_all) continue;
        table->assign(slots, CuckooSlot{0, 0});
        if (slot_of) slot_of->assign(items.size(), 0xFFFFFFFFu);
        for (uint64_t sl = 0; sl < slots; ++sl)
            if (owner[sl] >= 0) {
                (*table)[sl] = CuckooSlot{items[owner[sl]].fp, items[owner[sl]].payload};
                if (slot_of) (*slot_of)[(size_t)owner[sl]] = (uint32_t)sl;
            }
        *bits_out = bits;
        return LT_OK;
    }
    return fail(LT_ERR_CAPACITY, "could not place the %s in a cuckoo table", what);
}

template <typename T>
static int upload(lt_tables* t, const std::vector<T>& host, const T** out) {
    void* d = nullptr;
    size_t bytes = std::max<size_t>(host.size(), 1) * sizeof(T);
    CU(cudaMalloc(&d, bytes));
    t->allocations.push_back(d);
    t->bytes += (int64_t)bytes;
    if (!host.empty()) CU(cudaMemcpy(d, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = reinterpret_cast<const T*>(d);
    return LT_OK;
}

extern "C" void lt_tables_destroy(lt_tables* t) {
    if (!t) return;
    DeviceGuard guard(t->device);
    for (void* p : t->allocations) cudaFree(p);
    delete t;
}

extern "C" int64_t lt_tables_device_bytes(const lt_tables* t) { return t ? t->bytes : 0; }

static int build_tables(const lt_tables_desc* d, lt_tables* t) {
    DevTables& D = t->dev;
    if (d->abi_version != LT_ABI_VERSION) return fail(LT_ERR_INVALID, "abi_version %d != %d", d->abi_version, LT_ABI_VERSION);
    if (d->n_tags < LT_TAG_UNK + 1 || d->n_tags > LT_MAX_TAGS) return fail(LT_ERR_INVALID, "n_tags %d out of range", d->n_tags);
    if (d->n_tag_order < 0 || d->n_tag_order > LT_MAX_TAGS) return fail(LT_ERR_INVALID, "n_tag_order out of range");
    if (d->n_funcs < 0 || d->n_funcs > LT_MAX_FUNCS) return fail(LT_ERR_INVALID, "at most %d score functions", LT_MAX_FUNCS);
    D.n_tags = d->n_tags;
    D.n_tag_order = d->n_tag_order;
    D.max_len = d->max_len;
    D.order_mask = 0;
    for (int i = 0; i < 32; ++i) D.tag_pos[i] = 0xFF;
    for (int i = 0; i < d->n_tag_order; ++i) {
        const uint8_t t = d->tag_order[i];
        if (t >= LT_MAX_TAGS) return fail(LT_ERR_INVALID, "tag_order[%d] = %d out of range", i, (int)t);
        D.tag_order[i] = t;
        if (!((D.order_mask >> t) & 1u)) D.tag_pos[t] = (uint8_t)i;      // a repeated tag keeps its first position
        D.order_mask |= 1u << t;
    }

    // ---- powers of the hash bases ----
    int64_t max_str = 1;
    for (int64_t i = 0; i < d->n_dict; ++i) max_str = std::max(max_str, d->dict_off[i + 1] - d->dict_off[i]);
    D.max_str = (int32_t)std::min<int64_t>(max_str, 65535);
    const int n_pows = 65536 + 64;
    std::vector<H2> pows(n_pows);
    pows[0] = H2{1, 1};
    for (int i = 1; i < n_pows; ++i) pows[i] = H2{pows[i - 1].a * kBaseA, pows[i - 1].b * kBaseB};
    D.n_pows = n_pows;
    if (int rc = upload(t, pows, &D.pows)) return rc;

    // ---- dictionary ----
    {
        std::vector<CuckooItem> items((size_t)d->n_dict);
        for (int64_t i = 0; i < d->n_dict; ++i) {
            const int64_t len = d->dict_off[i + 1] - d->dict_off[i];
            if (len < 0 || len > 65535) return fail(LT_ERR_INVALID, "dictionary entry %lld has length %lld", (long long)i, (long long)len);
            const H2 h = hash_units(d->dict_chars + d->dict_off[i], len);
            items[i] = CuckooItem{dict_slot_hash(h, (uint32_t)len), dict_fp(h, (uint32_t)len),
                                  (uint64_t)d->dict_tagmask[i] | ((uint64_t)d->dict_lemma[i] << 32)};
        }
        std::vector<CuckooSlot> slots;
        if (int rc = build_cuckoo(items, next_pow2((uint64_t)d->n_dict * (d->n_dict < (1 << 22) ? 4 : 2)), &slots, &D.dict_bits,
                                  "dictionary entries"))
            return rc;
        static_assert(sizeof(CuckooSlot) == sizeof(DictSlot), "slot layout");
        std::vector<DictSlot> table(slots.size());
        for (size_t i = 0; i < slots.size(); ++i)
            table[i] = DictSlot{slots[i].fp, (uint32_t)slots[i].payload, (uint32_t)(slots[i].payload >> 32)};
        D.dict_mask = table.size() - 1;
        if (int rc = upload(t, table, &D.dict)) return rc;
    }

    // ---- rules ----
    {
        std::vector<RuleRec> recs((size_t)d->n_rules);
        for (int64_t r = 0; r < d->n_rules; ++r) {
            const int64_t s0 = d->rule_stem_off[r], e0 = d->rule_eomi_off[r], s1 = d->rule_stem_off[r + 1];
            if (!(s0 <= e0 && e0 <= s1)) return fail(LT_ERR_INVALID, "rule %lld has inconsistent offsets", (long long)r);
            recs[r].stem = hash_units(d->rule_chars + s0, e0 - s0);
            recs[r].eomi = hash_units(d->rule_chars + e0, s1 - e0);
            recs[r].stem_len = (uint32_t)(e0 - s0);
            recs[r].eomi_len = (uint32_t)(s1 - e0);
            recs[r].pad = 0;
        }
        if (int rc = upload(t, recs, &D.rrec)) return rc;
        std::vector<CuckooItem> items((size_t)d->n_rule_keys);
        for (int64_t k = 0; k < d->n_rule_keys; ++k) {
            const uint32_t len = d->rule_key_len[k];
            if (len < 1 || len > 3) return fail(LT_ERR_INVALID, "rule key %lld has length %u (1..3 expected)", (long long)k, len);
            const uint16_t* c = d->rule_key_chars + 3 * k;
            const uint64_t key = rule_key(c[0], len > 1 ? c[1] : 0, len > 2 ? c[2] : 0, len);
            const int64_t first = d->rule_first[k], count = d->rule_first[k + 1] - first;
            if (count < 0 || count > 255) return fail(LT_ERR_INVALID, "rule key %lld has %lld rules (at most 255)", (long long)k, (long long)count);
            items[k] = CuckooItem{fmix64(key), key, (uint64_t)(uint32_t)first |
                                  ((uint64_t)((uint32_t)count | (d->rule_k3_first[k] ? 0x80000000u : 0u)) << 32)};
        }
        std::vector<CuckooSlot> slots;
        if (int rc = build_cuckoo(items, next_pow2((uint64_t)d->n_rule_keys * 4), &slots, &D.rule_bits, "rule keys")) return rc;
        static_assert(sizeof(CuckooSlot) == sizeof(RuleSlot), "slot layout");
        std::vector<RuleSlot> table(slots.size());
        for (size_t i = 0; i < slots.size(); ++i)
            table[i] = RuleSlot{slots[i].fp, (uint32_t)slots[i].payload, (uint32_t)(slots[i].payload >> 32)};
        D.has_rules = d->n_rule_keys > 0;
        if (int rc = upload(t, table, &D.rules)) return rc;
    }

    // ---- score program ----
    D.n_funcs = d->n_funcs;
    D.n_tri = 0;
    for (int f = 0; f < d->n_funcs; ++f) {
        D.funcs[f] = d->funcs[f];
        D.func_dense[f] = -1;
        switch (d->funcs[f].kind) {
            case LT_FUNC_REG: case LT_FUNC_MPREF: case LT_FUNC_WPREF: break;
            case LT_FUNC_TRIGRAM: D.func_dense[f] = (int8_t)D.n_tri++; break;
            default: return fail(LT_ERR_INVALID, "score function %d has unknown kind %d", f, d->funcs[f].kind);
        }
    }

    for (int f = 0; f < LT_MAX_FUNCS; ++f) {
        for (int tmpl = 0; tmpl < 9; ++tmpl) D.seeds[f][tmpl] = feature_seed((uint32_t)tmpl, (uint32_t)f);
        const int kind = f < d->n_funcs ? d->funcs[f].kind : 0;
        D.seeds[f][9] = feature_seed(kind == LT_FUNC_WPREF ? kKindWPref : kKindMPref, (uint32_t)f);
    }

    // ---- feature strings ----
    std::vector<H2> fstr((size_t)d->n_fstr);
    for (int64_t i = 0; i < d->n_fstr; ++i)
        fstr[i] = hash_units(d->fstr_chars + d->fstr_off[i], d->fstr_off[i + 1] - d->fstr_off[i]);
    auto str_hash = [&](int32_t id, H2* out) -> bool {
        if (id < 0) { *out = H2{0, 0}; return true; }
        if (id >= d->n_fstr) return false;
        *out = fstr[id];
        return true;
    };

    // ---- dense blocks + hashed feature table ----
    const int NT = d->n_tags;
    const size_t blk = (size_t)dense_block_bytes(NT);
    std::vector<unsigned char> dense(std::max<size_t>(1, (size_t)D.n_tri * blk), 0);
    struct Pending { FKey key; double w; };
    std::vector<Pending> pending;
    std::vector<int64_t> pending_src;                    // input feature of a hashed entry (-1: a preference)
    pending.reserve((size_t)(d->n_feat + d->n_pref));
    t->feat_dst.assign((size_t)d->n_feat, kDstNone);
    t->feat_func.assign(d->feat_func, d->feat_func + d->n_feat);
    for (int64_t i = 0; i < d->n_feat; ++i) {
        const int f = d->feat_func[i];
        if (f >= d->n_funcs || D.func_dense[f] < 0) return fail(LT_ERR_INVALID, "feature %lld belongs to scorer %d which is not a trigram scorer", (long long)i, f);
        const int tmpl = d->feat_template[i];
        const int32_t* s = d->feat_s + 3 * i;
        const int32_t* a = d->feat_a + 2 * i;
        const double w = d->feat_weight[i];
        unsigned char* base = dense.data() + (size_t)D.func_dense[f] * blk;
        double* t3 = reinterpret_cast<double*>(base);
        double* t4 = t3 + NT * NT;
        double* t6 = t4 + kT4Dense;
        uint32_t* m3 = reinterpret_cast<uint32_t*>(t6 + 16);
        uint32_t* m4 = m3 + NT;
        uint32_t* m6 = m4 + 2;
        if (tmpl == 3) {
            if (a[0] < 0 || a[0] >= NT || a[1] < 0 || a[1] >= NT) return fail(LT_ERR_INVALID, "feature %lld: tag id out of range", (long long)i);
            t3[a[0] * NT + a[1]] = w;
            m3[a[0]] |= 1u << a[1];
            t->feat_dst[i] = kDstDense | (uint32_t)(&t3[a[0] * NT + a[1]] - reinterpret_cast<double*>(dense.data()));
            continue;
        }
        if (tmpl == 4 && a[0] >= 0 && a[0] < kT4Dense) {
            t4[a[0]] = w;
            m4[a[0] >> 5] |= 1u << (a[0] & 31);
            t->feat_dst[i] = kDstDense | (uint32_t)(&t4[a[0]] - reinterpret_cast<double*>(dense.data()));
            continue;
        }
        if (tmpl == 6) {
            if (a[0] < 0 || a[0] > 8) continue;          // min(8, len) never exceeds 8
            t6[a[0]] = w;
            m6[0] |= 1u << a[0];
            t->feat_dst[i] = kDstDense | (uint32_t)(&t6[a[0]] - reinterpret_cast<double*>(dense.data()));
            continue;
        }
        if (tmpl < 0 || tmpl > 8) return fail(LT_ERR_INVALID, "feature %lld: template %d", (long long)i, tmpl);
        if (a[0] < 0 || a[1] < 0 || a[0] >= (1 << 24) || a[1] >= (1 << 24)) continue;   // cannot equal a generated tuple
        H2 h0, h1, h2;
        if (!str_hash(s[0], &h0) || !str_hash(s[1], &h1) || !str_hash(s[2], &h2))
            return fail(LT_ERR_INVALID, "feature %lld: string id out of range", (long long)i);
        // Component slots are by ROLE so that the beam kernel can keep per-word hash products:
        // slot 0 = current word k (or its morpheme), slot 1 = previous word j (or the contextual
        // morpheme), slot 2 = word i.  The description lists them in template order.
        H2 r0 = h0, r1{0, 0}, r2{0, 0};
        switch (tmpl) {
            case 0: r0 = h1; r1 = h0; break;                 // (wj, wk, tk)
            case 1: r0 = H2{0, 0}; r1 = h0; break;           // (wj, tk)
            case 7: r0 = h2; r1 = h1; r2 = h0; break;        // (wi, wj, wk)
            case 8: r0 = h1; r1 = h0; break;                 // (m?, mk)
            default: break;                                  // 2, 4, 5: (wk) in slot 0
        }
        pending.push_back(Pending{feature_key((uint32_t)tmpl, (uint32_t)f, r0, r1, r2, (uint32_t)a[0], (uint32_t)a[1]), w});
        pending_src.push_back(i);
    }
    for (int64_t i = 0; i < d->n_pref; ++i) {
        const int f = d->pref_func[i];
        if (f >= d->n_funcs) return fail(LT_ERR_INVALID, "preference %lld: scorer index", (long long)i);
        const int kind = d->funcs[f].kind;
        if (kind != LT_FUNC_MPREF && kind != LT_FUNC_WPREF) return fail(LT_ERR_INVALID, "preference %lld belongs to a non-preference scorer", (long long)i);
        H2 h0;
        if (!str_hash(d->pref_s[i], &h0)) return fail(LT_ERR_INVALID, "preference %lld: string id out of range", (long long)i);
        pending.push_back(Pending{feature_key(kind == LT_FUNC_MPREF ? kKindMPref : kKindWPref, (uint32_t)f, h0, H2{0, 0}, H2{0, 0},
                                              d->pref_tag[i], 0), d->pref_value[i]});
        pending_src.push_back(-1);
    }
    {
        const uint64_t n = pending.size();
        std::vector<CuckooItem> items((size_t)n);
        for (uint64_t i = 0; i < n; ++i) {
            uint64_t wbits;
            memcpy(&wbits, &pending[i].w, 8);
            items[i] = CuckooItem{feature_slot_hash(pending[i].key.k1), pending[i].key.k2, wbits};
        }
        std::vector<CuckooSlot> slots;
        std::vector<uint32_t> slot_of;
        if (int rc = build_cuckoo(items, next_pow2(n * (n < (1u << 22) ? 4 : 2)), &slots, &D.feat_bits, "feature keys", &slot_of)) return rc;
        for (uint64_t i = 0; i < n; ++i)
            if (pending_src[i] >= 0) t->feat_dst[(size_t)pending_src[i]] = slot_of[i];
        static_assert(sizeof(CuckooSlot) == sizeof(FeatSlot), "slot layout");
        std::vector<FeatSlot> table(slots.size());
        for (size_t i = 0; i < slots.size(); ++i) {
            table[i].fp = slots[i].fp;
            memcpy(&table[i].w, &slots[i].payload, 8);
        }
        D.feat_mask = table.size() - 1;
        if (int rc = upload(t, table, &D.feat)) return rc;
    }
    if (int rc = upload(t, dense, &D.dense)) return rc;
    t->dense_host = dense;

    const uint16_t bos[3] = {'B', 'O', 'S'};
    D.bos = hash_units(bos, 3);
    return LT_OK;
}

extern "C" int lt_tables_create(const lt_tables_desc* desc, int device, lt_tables** out) {
    if (!desc || !out) return fail(LT_ERR_INVALID, "null argument");
    *out = nullptr;
    ON_DEVICE(device);
    lt_tables* t = new lt_tables();
    t->device = device;
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { delete t; return fail(LT_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e)); }
    t->sm_count = prop.multiProcessorCount;
    int rc = build_tables(desc, t);
    if (rc != LT_OK) { lt_tables_destroy(t); return rc; }
    *out = t;
    return LT_OK;
}

// ------------------------------------------------------------------------------------------------
// batch workspace
// ------------------------------------------------------------------------------------------------
// control words on the device: work-queue cursors, the 64-bit edge cursor, overflow flags, retry list length
enum { kCtlLatticeQueue = 0, kCtlBeamQueue = 1, kCtlCursor = 2 /* 2 words */, kCtlFlags = 4 /* 2 words */, kCtlRetryQueue = 6,
       kCtlRetryCount = 7, kCtlWords = 8 };

static const size_t kSmemBudget = 200 * 1024;
static const size_t kBeamCtaSmemMax = 226 * 1024;    // one large beam CTA may take (nearly) all the shared memory an SM has

// Launch shapes are decided once per (array size, capacity) and kept: kernel instantiation, CTA shape,
// shared memory, resident CTAs per SM.  Nothing of this is recomputed (or asked of the driver) per batch.
struct LatticePlan {
    int units = 0, hcap = 0;                  // key
    bool generic = false, any_lookup = false, retry = false;
    void (*fn)(const DevTables, const LatticeArgs) = nullptr;
    int warps = 0, per_sm = 1;
    size_t smem = 0, warp_smem = 0;
};
struct BeamPlan {
    int units = 0, beam = 0;                  // key
    bool kbest = false, hbm_trail = false, constrained = false;
    void (*fn)(const DevTables, const BeamArgs) = nullptr;
    int warps = 0, per_sm = 1;
    size_t smem = 0, warp_smem = 0;
    bool trail_smem = false;
};

// events of a timed batch (lt_batch_timings): host text in, lattice kernels, beam kernel, path packing, results out
enum { kEvHostIn, kEvLatticeStart, kEvLatticeEnd, kEvBeamStart, kEvBeamEnd, kEvPackEnd, kEvHostOut, kStageEvents };

struct lt_constraints {
    lt_tables* tables = nullptr;
    int device = 0;
    int32_t n_sent = 0;
    DevBuf cons, off;               // [n_cons] constraints, [n_sent + 1] offsets
};

struct lt_batch {
    lt_tables* tables = nullptr;
    cudaStream_t own_stream = nullptr;
    unsigned int* h_ctl = nullptr;   // pinned: the control words come back with the results without stalling the copies queued behind them
    cudaStream_t last_stream = nullptr;
    // inputs (host entry point) and per-unit / per-sentence arrays
    DevBuf text, sent_off, pos, scan_tmp;
    DevBuf sent_len, sent_edges, status, path_len, path_off, scores;
    DevBuf edges, trail, path_tmp, path_out, counters, ctl, order, retry;
    DevBuf kb_tmp, kb_out, kb_len, kb_off, kb_scores, kb_count;      // all survivors (lt_beam_kbest)
    DevBuf imp;                    // string hashes of an imported lattice (lt_lattice_import)
    DevBuf pth_ch, pth_ha, pth_hb;               // lt_perceptron_delta: syllables and prefix hashes of the batch's sentences
    DevBuf pth_scores, pth_feat, pth_nfeat;      // lt_pathset_eval results
    DevBuf pc_delta, pc_differs, pc_count;       // lt_perceptron_delta results
    DevBuf ev_image, ev_class, ev_counts, ev_scores, ev_reason;   // lt_evaluate: gold images (scratch), results
    DevBuf cons_status, cons_desc;               // constrained search: its per-sentence status, position descriptors
    const lt_constraints* cons = nullptr;        // bound by lt_batch_set_constraints for the searches to come
    const lt_constraints* search_cons = nullptr; // the set the last search ran with (its reruns run with it too)
    bool imported = false;
    const uint16_t* d_text = nullptr;
    const int32_t* d_sent_off = nullptr;
    int32_t n_sent = 0;
    int64_t n_units = 0;
    int32_t max_sent_units = 0;
    int32_t lcap = 0;
    int32_t beam = 0;
    int32_t lookup_mode = LT_LOOKUP_MORPHEME;
    int32_t hcap = 128;            // lattice staging capacity per warp of the main pass
    bool use_retry = false;        // a batch outgrew `hcap`: such sentences go to a retry pass from now on (sticky)
    int32_t retry_hcap = 0;        // staging capacity of the retry pass (grows on overflow, sticky)
    bool sort_by_length = true;    // persistent warps pull the longest sentences first (LT_SORT_BY_LENGTH=0 disables)
    uint32_t edge_cap = 0;         // edge buffer capacity (grows on overflow, sticky)
    bool edge_cap_fixed = false;   // LT_EDGE_CAP given: start there instead of the size guess (tests)
    bool debug = false;            // LT_DEBUG: print launch shapes
    bool trail_smem_ok = true;     // LT_TRAIL_SMEM=0 keeps the back-pointers in HBM
    bool hbm_trail = false;        // a trainer step that reads the back-pointers: HBM, 0xFF before every search of the step
    int adapt_div = 32;            // LT_ADAPT_DIV: the main pass's staging area doubles when more than n_sent / this many eojeols
                                   // needed the retry pass (0 = never; measured on C3: the default is right)
    int sort_min = kSortMin;       // LT_SORT_MIN: staged hits per eojeol from which the lattice kernel ranks by sorting (tests: 1)
    int prologue_ctas = kPrologueMaxCtas;   // LT_PROLOGUE_CTAS: CTAs of the work-order prologue (1 = exact order)
    int64_t n_edges = 0;
    bool have_lattice = false, have_paths = false, have_kbest = false, resolved = false;
    bool beam_state_clean = false;   // beam queue cursor / counters still zero from the batch prologue
    cudaEvent_t ev[kStageEvents]{};
    bool timed = false;
    int reruns = 0;                // grow-and-rerun rounds so far (cumulative)
    int64_t launches = 0;          // kernels launched so far (cumulative)
    int64_t words_hint = -1;       // path records of the previous batch: the speculative part of the result copy
    uint32_t last_retried = 0;
    std::vector<LatticePlan> lattice_plans;
    std::vector<BeamPlan> beam_plans;
    const LatticePlan* last_lattice_plan = nullptr;
    const BeamPlan* last_beam_plan = nullptr;
};

// Longest sentence (raw UTF-16 code units, spaces included) both kernels can hold in shared memory with
// these tables: the lattice kernel's per-warp arrays grow with the longest dictionary string (substring
// table), the beam kernel's with the beam size.  Longer sentences get LT_SENT_TOO_LONG.
static int32_t unit_limit(const lt_tables* t) {
    const int max_str = std::max(1, t->dev.max_str);
    const size_t dense_bytes = ((size_t)t->dev.n_tri * dense_block_bytes(t->dev.n_tags) + 15) & ~(size_t)15;
    int32_t lo = 8, hi = 4088;
    auto fits = [&](int32_t lcap) {
        return lattice_warp_smem(lcap + 8, kLatDefaultHcap, max_str) <= kSmemBudget &&
               dense_bytes + beam_warp_smem(lcap + 8, LT_MAX_BEAM, beam_kval_doubles(t->dev.n_funcs, false), false) <= kSmemBudget;
    };
    if (fits(hi)) return hi;
    while (hi - lo > 8) {
        const int32_t mid = ((lo + hi) / 2) & ~7;
        if (fits(mid)) lo = mid; else hi = mid;
    }
    return lo;
}

extern "C" int32_t lt_tables_max_sentence_units(const lt_tables* t) { return t ? unit_limit(t) : 0; }

// where each input feature's weight lives (feat_dst) on the device, uploaded on first use
static int upload_feat_dst(lt_tables* t) {
    if (t->d_feat_dst.p || t->feat_dst.empty()) return LT_OK;
    return upload_once(t->d_feat_dst, t->feat_dst.data(), t->feat_dst.size() * 4);
}

// New weights for the features the tables were built with (the trainer's epoch: same features, new
// coefficients) — written in place: a scatter into the hashed table's weight fields and a rewrite of the small
// dense blocks.  No table is rebuilt.  The caller must not have a batch in flight on these tables.
extern "C" int lt_tables_update_weights(lt_tables* t, const double* weights, int64_t n_weights) {
    if (!t || (n_weights > 0 && !weights)) return fail(LT_ERR_INVALID, "null argument");
    if ((size_t)n_weights != t->feat_dst.size())
        return fail(LT_ERR_INVALID, "the tables were built with %zu features, %lld weights given", t->feat_dst.size(), (long long)n_weights);
    ON_DEVICE(t->device);
    if (n_weights == 0) return LT_OK;
    if (int rc = upload_feat_dst(t)) return rc;
    if (int rc = ensure(t->d_weights, (size_t)n_weights * 8)) return rc;
    CU(cudaMemcpy(t->d_weights.p, weights, (size_t)n_weights * 8, cudaMemcpyHostToDevice));
    const unsigned grid = (unsigned)std::min<int64_t>((n_weights + 255) / 256, (int64_t)t->sm_count * 16);
    LT_LAUNCH(scatter_weights, grid, 256, 0, (cudaStream_t) nullptr, const_cast<FeatSlot*>(t->dev.feat),
              static_cast<const uint32_t*>(t->d_feat_dst.p), static_cast<const double*>(t->d_weights.p), n_weights);
    CU(cudaGetLastError());
    double* dense = reinterpret_cast<double*>(t->dense_host.data());
    bool any_dense = false;
    for (int64_t i = 0; i < n_weights; ++i)
        if (t->feat_dst[(size_t)i] != kDstNone && (t->feat_dst[(size_t)i] & kDstDense)) {
            dense[t->feat_dst[(size_t)i] & ~kDstDense] = weights[i];
            any_dense = true;
        }
    if (any_dense)
        CU(cudaMemcpy(const_cast<unsigned char*>(t->dev.dense), t->dense_host.data(), t->dense_host.size(), cudaMemcpyHostToDevice));
    CU(cudaDeviceSynchronize());
    return LT_OK;
}

extern "C" int lt_batch_create(lt_tables* tables, lt_batch** out) {
    if (!tables || !out) return fail(LT_ERR_INVALID, "null argument");
    ON_DEVICE(tables->device);
    lt_batch* b = new lt_batch();
    b->tables = tables;
    CU(cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking));
    CU(cudaMallocHost(reinterpret_cast<void**>(&b->h_ctl), kCtlWords * sizeof(unsigned int)));
    for (auto& e : b->ev) CU(cudaEventCreate(&e));
    // debugging / test knobs, read once here: tiny initial capacities exercise the grow-and-rerun path
    if (const char* env = getenv("LT_HIT_CAP")) b->hcap = std::max(8, atoi(env));
    if (const char* env = getenv("LT_SORT_BY_LENGTH")) b->sort_by_length = atoi(env) != 0;
    if (const char* env = getenv("LT_EDGE_CAP")) { b->edge_cap = (uint32_t)std::max(16, atoi(env)); b->edge_cap_fixed = true; }
    if (const char* env = getenv("LT_TRAIL_SMEM")) b->trail_smem_ok = atoi(env) != 0;
    if (const char* env = getenv("LT_ADAPT_DIV")) b->adapt_div = std::max(0, atoi(env));
    if (const char* env = getenv("LT_SORT_MIN")) b->sort_min = std::max(1, atoi(env));
    if (const char* env = getenv("LT_PROLOGUE_CTAS")) b->prologue_ctas = std::min(32, std::max(1, atoi(env)));
    b->debug = getenv("LT_DEBUG") != nullptr;
    *out = b;
    return LT_OK;
}

extern "C" void lt_batch_destroy(lt_batch* b) {
    if (!b) return;
    DeviceGuard guard(b->tables->device);
    for (auto& e : b->ev)
        if (e) cudaEventDestroy(e);
    if (b->h_ctl) cudaFreeHost(b->h_ctl);
    if (b->own_stream) cudaStreamDestroy(b->own_stream);
    delete b;
}

extern "C" int lt_batch_set_lookup(lt_batch* b, int32_t mode) {
    if (!b) return fail(LT_ERR_INVALID, "null argument");
    if (mode < LT_LOOKUP_MORPHEME || mode > LT_LOOKUP_EXACT) return fail(LT_ERR_INVALID, "unknown lookup mode %d", mode);
    b->lookup_mode = mode;
    return LT_OK;
}

static int scan_u32(lt_batch* b, const uint32_t* in, uint32_t* out, int64_t n, cudaStream_t st) {
    if (n <= kScanSmallMax) {
        LT_LAUNCH(scan_small, 1, kScanSmallThreads, 0, st, in, out, n);
        CU(cudaGetLastError());
        b->launches += 1;
        return LT_OK;
    }
    const int64_t tiles = (n + kScanTile - 1) / kScanTile;
    if (int rc = ensure(b->scan_tmp, (size_t)tiles * 4)) return rc;
    uint32_t* sums = static_cast<uint32_t*>(b->scan_tmp.p);
    LT_LAUNCH(scan_tile_sums, (unsigned)tiles, kScanThreads, 0, st, in, n, sums);
    LT_LAUNCH(scan_sums, 1, kScanThreads, 0, st, sums, tiles);
    LT_LAUNCH(scan_apply, (unsigned)tiles, kScanThreads, 0, st, in, out, n, sums);
    CU(cudaGetLastError());
    b->launches += 3;
    return LT_OK;
}

// raise a kernel's dynamic shared-memory limit once per device (and again only when more is needed).  The limit
// belongs to the function on the device, not to the tables: the cache is keyed by (device, function) and shared by all
// tables, or a second tables' smaller request would lower the limit below what the first one's plans were sized for.
// (One cache per kernel signature Fn; the function pointer in the key tells the instantiations apart.)
template <typename Fn>
static int smem_limit(lt_tables* t, Fn fn, size_t bytes) {
    static std::mutex mu;
    static std::vector<std::pair<std::pair<int, const void*>, size_t>> limits;
    std::lock_guard<std::mutex> lock(mu);
    const std::pair<int, const void*> key(t->device, reinterpret_cast<const void*>(fn));
    for (auto& kv : limits)
        if (kv.first == key) {
            if (kv.second >= bytes) return LT_OK;
            CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            kv.second = bytes;
            return LT_OK;
        }
    CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    limits.emplace_back(key, bytes);
    return LT_OK;
}

// ---- launch plans --------------------------------------------------------------------------------
static int lattice_plan(lt_batch* b, int lcap, int hcap, bool retry_pass, const LatticePlan** out) {
    lt_tables* t = b->tables;
    const int max_str = std::max(1, t->dev.max_str);
    if (hcap & 1) ++hcap;                               // keeps the arrays behind the staging area 8-byte aligned
    // common sentence-array sizes (with the default staging capacity) have their own instantiation
    const bool any_lookup = b->lookup_mode != LT_LOOKUP_MORPHEME;      // the other lookups run in the generic instantiation
    const int uclass = (!any_lookup && !retry_pass && (hcap == kLatDefaultHcap || hcap == 2 * kLatDefaultHcap)) ? lattice_units_class(lcap) : 0;
    const int units = uclass ? uclass : lcap + 8;
    for (const LatticePlan& p : b->lattice_plans)
        if (p.units == units && p.hcap == hcap && p.generic == (uclass == 0) && p.any_lookup == any_lookup && p.retry == retry_pass) { *out = &p; return LT_OK; }
    LatticePlan P;
    P.units = units;
    P.hcap = hcap;
    P.generic = uclass == 0;
    P.any_lookup = any_lookup;
    P.retry = retry_pass;
    P.warp_smem = lattice_warp_smem(units, hcap, max_str);
    if (retry_pass) {
        if (P.warp_smem > kSmemBudget)
            return fail(LT_ERR_CAPACITY, "one eojeol yields more than %d lattice candidates; the staging buffer cannot grow further", hcap / 2);
        P.warps = (int)std::max<size_t>(1, std::min<size_t>(2, kSmemBudget / P.warp_smem));
    } else {
        // CTA shape: the warps per CTA (1..8) that keep the most warps resident on an SM (128 registers per
        // thread allow 16); ties go to 4-warp CTAs
        int best_res = 0;
        const int reg_warps = 16;
        for (int w : {kLatWarps, 8, 6, 5, 3, 2, 1}) {
            const size_t cta = P.warp_smem * w;
            if (cta > kSmemBudget) continue;
            const int res = w * (int)std::min<size_t>(reg_warps / w, (size_t)228 * 1024 / (cta + 1024));
            if (res > best_res) { best_res = res; P.warps = w; }
        }
        if (P.warps < 1)
            return fail(LT_ERR_INVALID, "a sentence of %d code units (dictionary strings up to %d) does not fit the lattice "
                                        "kernel's shared memory", lcap, max_str);
    }
    P.smem = P.warp_smem * P.warps;
    P.fn = (uclass == 64 && hcap == kLatDefaultHcap) ? lt::lattice_kernel<64, kLatDefaultHcap>
         : (uclass == 128 && hcap == kLatDefaultHcap) ? lt::lattice_kernel<128, kLatDefaultHcap>
         : (uclass == 64 && hcap == 2 * kLatDefaultHcap) ? lt::lattice_kernel<64, 2 * kLatDefaultHcap>
         : (uclass == 128 && hcap == 2 * kLatDefaultHcap) ? lt::lattice_kernel<128, 2 * kLatDefaultHcap>
         : retry_pass ? (any_lookup ? lt::lattice_kernel<0, 0, 1, 1> : lt::lattice_kernel<0, 0, 0, 1>)
         : any_lookup ? lt::lattice_kernel<0, 0, 1> : lt::lattice_kernel<0, 0, 0>;
    if (int rc = smem_limit(t, P.fn, P.smem)) return rc;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&P.per_sm, P.fn, P.warps * 32, P.smem));
    P.per_sm = std::max(1, P.per_sm);
    if (b->debug)
        fprintf(stderr, "[lt] lattice kernel%s: units %d%s hcap %d%s max_str %d, %zu B/warp, %d warps/CTA, %zu B/CTA, %d CTAs/SM\n",
                retry_pass ? " (retry pass)" : "", units, uclass ? " (sized instantiation)" : "", hcap, any_lookup ? " any lookup" : "",
                max_str, P.warp_smem, P.warps, P.smem, P.per_sm);
    b->lattice_plans.push_back(P);
    *out = &b->lattice_plans.back();
    return LT_OK;
}

static int beam_plan(lt_batch* b, int lcap, int beam_size, bool kbest, bool constrained, const BeamPlan** out) {
    lt_tables* t = b->tables;
    // sentence arrays: common sizes are template parameters of the kernel (for beams 5 and 10); the all-survivors
    // variant (lt_beam_kbest) and the constrained search exist in the generic instantiations only
    const int uclass = (!kbest && !constrained && (beam_size == 5 || beam_size == 10)) ? beam_units_class(lcap) : 0;
    const int units = uclass ? uclass : lcap + 8;
    for (const BeamPlan& p : b->beam_plans)
        if (p.units == units && p.beam == beam_size && p.kbest == kbest && p.hbm_trail == b->hbm_trail && p.constrained == constrained) {
            *out = &p;
            return LT_OK;
        }
    const size_t dense_bytes = ((size_t)t->dev.n_tri * dense_block_bytes(t->dev.n_tags) + 15) & ~(size_t)15;
    const bool reg_tri = !constrained && t->dev.n_funcs == 2 && t->dev.funcs[0].kind == LT_FUNC_REG && t->dev.funcs[1].kind == LT_FUNC_TRIGRAM;
    const bool prog1 = reg_tri && !kbest;                      // the instantiation specialised for that score program
    const int kvd = beam_kval_doubles(t->dev.n_funcs, prog1);
    // CTA shape: the warps per CTA (1..8) that keep the most warps resident on an SM under the kernel's
    // 128 registers per thread (16 warps) and the per-warp shared memory; ties go to 4-warp CTAs
    auto resident_warps = [&](size_t warp_smem, int w) -> int {
        const size_t cta = dense_bytes + warp_smem * w;
        if (cta > (w > 8 ? kBeamCtaSmemMax : kSmemBudget)) return 0;
        return w * (int)std::min<size_t>(LT_BEAM_REG_WARPS / w, (size_t)228 * 1024 / (cta + 1024));
    };
    auto best_warps = [&](size_t warp_smem) -> int {
        int best = 0, best_res = 0;
        // (ties go to the earlier entry: 4-warp CTAs first, then the larger shapes)
        for (int w : {kBeamWarps, 8, 6, 5, 3, 2, 1, 7, 9, 10, 11, 12, 13, 14, 15, 16}) {
            if (w > kBeamMaxWarps) continue;
            const int r = resident_warps(warp_smem, w);
            if (r > best_res) { best_res = r; best = w; }
        }
        return best;
    };
    // back-pointers live in shared memory when that does not lower the residency
    const size_t smem_hbm_trail = beam_warp_smem(units, beam_size, kvd, false);
    const size_t smem_own_trail = beam_warp_smem(units, beam_size, kvd, true);
    const int w_hbm = best_warps(smem_hbm_trail), w_own = best_warps(smem_own_trail);
    if (w_hbm == 0)
        return fail(LT_ERR_INVALID, "sentence length %d with beam %d does not fit the beam kernel's shared memory", lcap, beam_size);
    BeamPlan P;
    P.units = units;
    P.beam = beam_size;
    P.kbest = kbest;
    P.hbm_trail = b->hbm_trail;
    P.constrained = constrained;
    P.trail_smem = !b->hbm_trail && b->trail_smem_ok && w_own > 0 && resident_warps(smem_own_trail, w_own) >= resident_warps(smem_hbm_trail, w_hbm);
    P.warp_smem = P.trail_smem ? smem_own_trail : smem_hbm_trail;
    P.warps = P.trail_smem ? w_own : w_hbm;
    P.smem = dense_bytes + P.warp_smem * P.warps;
    // common beam sizes, sentence-array sizes and the (RegularizationScore, SimpleTrigramFeatureScore)
    // score program get their own instantiation (compile-time array offsets, unrolled scorer loop)
    if (constrained && kbest)
        P.fn = beam_size <= kRankMaxBeam ? beam_kernel<2, 0, 0, 0, 1, -1, 1> : (beam_size <= 32 ? beam_kernel<1, 0, 0, 0, 1, -1, 1> : beam_kernel<0, 0, 0, 0, 1, -1, 1>);
    else if (constrained)
        P.fn = beam_size <= kRankMaxBeam ? beam_kernel<2, 0, 0, 0, 0, -1, 1> : (beam_size <= 32 ? beam_kernel<1, 0, 0, 0, 0, -1, 1> : beam_kernel<0, 0, 0, 0, 0, -1, 1>);
    else if (kbest) P.fn = beam_size <= kRankMaxBeam ? beam_kernel<2, 0, 0, 0, 1> : (beam_size <= 32 ? beam_kernel<1, 0, 0, 0, 1> : beam_kernel<0, 0, 0, 0, 1>);
    // (the specialised kernels also know at compile time where the back-pointers live)
    else if (beam_size == 5 && uclass == 64) P.fn = reg_tri ? (P.trail_smem ? beam_kernel<2, 5, 64, 1, 0, 1> : beam_kernel<2, 5, 64, 1, 0, 0>) : beam_kernel<2, 5, 64, 0>;
    else if (beam_size == 5 && uclass == 128) P.fn = reg_tri ? (P.trail_smem ? beam_kernel<2, 5, 128, 1, 0, 1> : beam_kernel<2, 5, 128, 1, 0, 0>) : beam_kernel<2, 5, 128, 0>;
    else if (beam_size == 5) P.fn = reg_tri ? beam_kernel<2, 5, 0, 1> : beam_kernel<2, 5, 0, 0>;
    else if (beam_size == 10 && uclass == 64) P.fn = reg_tri ? (P.trail_smem ? beam_kernel<2, 10, 64, 1, 0, 1> : beam_kernel<2, 10, 64, 1, 0, 0>) : beam_kernel<2, 10, 64, 0>;
    else if (beam_size == 10 && uclass == 128) P.fn = reg_tri ? (P.trail_smem ? beam_kernel<2, 10, 128, 1, 0, 1> : beam_kernel<2, 10, 128, 1, 0, 0>) : beam_kernel<2, 10, 128, 0>;
    else if (beam_size == 10) P.fn = reg_tri ? beam_kernel<2, 10, 0, 1> : beam_kernel<2, 10, 0, 0>;
    else if (beam_size <= kRankMaxBeam) P.fn = reg_tri ? beam_kernel<2, 0, 0, 1> : beam_kernel<2, 0, 0, 0>;
    else if (beam_size == 32) P.fn = reg_tri ? beam_kernel<1, 32, 0, 1> : beam_kernel<1, 32, 0, 0>;
    else if (beam_size <= 32) P.fn = reg_tri ? beam_kernel<1, 0, 0, 1> : beam_kernel<1, 0, 0, 0>;
    else P.fn = reg_tri ? beam_kernel<0, 0, 0, 1> : beam_kernel<0, 0, 0, 0>;
    if (int rc = smem_limit(t, P.fn, P.smem)) return rc;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&P.per_sm, P.fn, P.warps * 32, P.smem));
    P.per_sm = std::max(1, P.per_sm);
    if (b->debug)
        fprintf(stderr, "[lt] beam kernel: beam %d units %d%s, %zu B/warp, %d warps/CTA, %zu B/CTA, %d CTAs/SM, trail in %s%s%s%s\n", beam_size,
                units, uclass ? " (sized instantiation)" : "", P.warp_smem, P.warps, P.smem, P.per_sm, P.trail_smem ? "shared memory" : "HBM",
                prog1 ? ", reg+trigram program" : "", kbest ? ", k-best" : "", constrained ? ", constrained" : "");
    b->beam_plans.push_back(P);
    *out = &b->beam_plans.back();
    return LT_OK;
}

// ---- launches ----------------------------------------------------------------------------------
// The inputs of the next lattice: text and sentence offsets in device memory, read on stream st.  The per-warp
// arrays are sized for the longest sentence the caller reports, capped at what fits shared memory; the kernels
// skip any sentence beyond that size (LT_SENT_TOO_LONG) instead of trusting the number.
static void bind_batch(lt_batch* b, const uint16_t* d_text, const int32_t* d_sent_off, int32_t n_sent, int64_t n_units,
                       int32_t max_sent_units, cudaStream_t st) {
    b->last_stream = st;
    b->d_text = d_text;
    b->d_sent_off = d_sent_off;
    b->n_sent = n_sent;
    b->n_units = n_units;
    b->max_sent_units = max_sent_units;
    b->beam = 0;
    b->lcap = std::max(8, (std::min(max_sent_units, unit_limit(b->tables)) + 7) & ~7);
    b->have_lattice = b->have_paths = b->have_kbest = false;
    b->imported = b->resolved = false;
}

// per-sentence statuses of the last search: the lattice's, or a constrained search's own (LT_SENT_BAD_CONSTRAINT)
static const void* search_status(const lt_batch* b) { return b->search_cons ? b->cons_status.p : b->status.p; }

// the order in which persistent warps take sentences (longest first), or nullptr: in input order
static uint32_t* work_order(const lt_batch* b) {
    return (b->sort_by_length && b->n_sent > 1) ? static_cast<uint32_t*>(b->order.p) : nullptr;
}

// Per-sentence buffers and control words of the bound batch; the batch prologue zeroes the control words and
// counters and computes the work order.
static int start_batch(lt_batch* b, cudaStream_t st) {
    const int n_sent = b->n_sent;
    if (int rc = ensure(b->pos, ((size_t)b->n_units + 1) * sizeof(uint2))) return rc;
    if (int rc = ensure(b->sent_len, (size_t)std::max(1, n_sent) * 4)) return rc;
    if (int rc = ensure(b->sent_edges, (size_t)std::max(1, n_sent) * 4)) return rc;
    if (int rc = ensure(b->status, (size_t)std::max(1, n_sent) * 4)) return rc;
    if (int rc = ensure(b->counters, 8 * sizeof(unsigned long long))) return rc;
    if (int rc = ensure(b->ctl, kCtlWords * sizeof(unsigned int))) return rc;
    if (b->sort_by_length && n_sent > 1)
        if (int rc = ensure(b->order, (size_t)n_sent * 4)) return rc;
    uint32_t* order = work_order(b);
    LT_LAUNCH(batch_prologue, (unsigned)(order ? std::min(b->prologue_ctas, prologue_ctas(n_sent)) : 1), 1024, 0, st, b->d_sent_off, n_sent,
              order, static_cast<unsigned int*>(b->ctl.p), kCtlWords, static_cast<unsigned long long*>(b->counters.p), 8);
    CU(cudaGetLastError());
    b->launches += 1;
    b->beam_state_clean = true;
    return LT_OK;
}

static int launch_lattice(lt_batch* b, cudaStream_t st) {
    lt_tables* t = b->tables;
    const int n_sent = b->n_sent;
    const int64_t n_units = b->n_units;
    const int lcap = b->lcap;
    const LatticePlan* P = nullptr;
    if (int rc = lattice_plan(b, lcap, b->hcap, false, &P)) return rc;
    b->last_lattice_plan = P;
    if (!b->edge_cap_fixed) {
        const uint64_t guess = (uint64_t)n_units * 3 + 4096;
        if (b->edge_cap < guess) b->edge_cap = (uint32_t)std::min<uint64_t>(guess, 0xFFFFFFF0ull);
    }
    if (int rc = ensure(b->edges, (size_t)b->edge_cap * sizeof(lt_edge))) return rc;
    if (int rc = start_batch(b, st)) return rc;

    LatticeArgs A{};
    A.text = b->d_text;
    A.sent_off = b->d_sent_off;
    A.n_sent = n_sent;
    A.units = P->units;
    A.hcap = P->hcap;
    A.max_str = std::max(1, t->dev.max_str);
    A.pos = static_cast<uint2*>(b->pos.p);
    A.edges = static_cast<lt_edge*>(b->edges.p);
    A.edge_cap = b->edge_cap;
    A.max_units = lcap;
    A.mode = b->lookup_mode;
    A.sort_min = b->sort_min;
    unsigned int* ctl = static_cast<unsigned int*>(b->ctl.p);
    A.cursor = reinterpret_cast<unsigned long long*>(ctl + kCtlCursor);
    A.flags = ctl + kCtlFlags;
    A.sent_len = static_cast<int32_t*>(b->sent_len.p);
    A.sent_edges = static_cast<int32_t*>(b->sent_edges.p);
    A.status = static_cast<int32_t*>(b->status.p);
    A.counters = static_cast<unsigned long long*>(b->counters.p);
    A.queue = ctl + kCtlLatticeQueue;
    A.order = work_order(b);

    const int64_t want_blocks = ((int64_t)n_sent + P->warps - 1) / P->warps;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want_blocks, (int64_t)t->sm_count * P->per_sm));
    if (b->use_retry) {
        // (sentence, eojeol) pairs: an eojeol takes at least one code unit and a separator
        if (int rc = ensure(b->retry, ((size_t)n_units / 2 + (size_t)n_sent + 16) * sizeof(uint2))) return rc;
        A.retry_list = static_cast<uint2*>(b->retry.p);
        A.retry_count = ctl + kCtlRetryCount;
    }
    if (b->timed) CU(cudaEventRecord(b->ev[kEvLatticeStart], st));
    if (n_sent > 0) {
        LT_LAUNCH(P->fn, grid, P->warps * 32, P->smem, st, t->dev, A);
        b->launches += 1;
    }
    CU(cudaGetLastError());
    if (b->use_retry && n_sent > 0) {
        // retry pass: the few sentences with an eojeol beyond `hcap` hits, with a staging area of their own size
        const LatticePlan* Rp = nullptr;
        if (int rc = lattice_plan(b, lcap, b->retry_hcap, true, &Rp)) return rc;
        LatticeArgs R = A;
        R.units = Rp->units;
        R.hcap = Rp->hcap;
        R.queue = ctl + kCtlRetryQueue;
        R.retry_pass = 1;
        LT_LAUNCH(Rp->fn, (unsigned)(t->sm_count * Rp->per_sm), Rp->warps * 32, Rp->smem, st, t->dev, R);
        CU(cudaGetLastError());
        b->launches += 1;
    }
    if (b->timed) CU(cudaEventRecord(b->ev[kEvLatticeEnd], st));
    b->have_lattice = true;
    b->have_paths = false;
    b->have_kbest = false;
    b->resolved = false;
    return LT_OK;
}

static int launch_beam(lt_batch* b, cudaStream_t st, bool kbest) {
    lt_tables* t = b->tables;
    // (an imported lattice names its strings: only the all-survivors instantiations read those, see edge_hashes)
    kbest = kbest || b->imported;
    const int beam_size = b->beam;
    const int n_sent = b->n_sent;
    const size_t nu = (size_t)b->n_units + 1;

    if (int rc = ensure(b->path_tmp, nu * sizeof(lt_edge))) return rc;
    if (int rc = ensure(b->path_out, nu * sizeof(lt_edge))) return rc;
    if (int rc = ensure(b->path_len, (size_t)(n_sent + 1) * 4)) return rc;
    if (int rc = ensure(b->path_off, (size_t)(n_sent + 1) * 4)) return rc;
    if (int rc = ensure(b->scores, (size_t)std::max(1, n_sent) * 8)) return rc;
    const size_t nk = (size_t)n_sent * beam_size;
    if (kbest) {
        if (nk + 1 > 0x7FFFFFFFull || nu * beam_size > 0x7FFFFFFFull)
            return fail(LT_ERR_CAPACITY, "k-best output of %d sentences x beam %d is too large for one batch; split it", n_sent, beam_size);
        if (int rc = ensure(b->kb_tmp, nu * beam_size * sizeof(lt_edge))) return rc;
        if (int rc = ensure(b->kb_out, nu * beam_size * sizeof(lt_edge))) return rc;
        if (int rc = ensure(b->kb_len, (nk + 1) * 4)) return rc;
        if (int rc = ensure(b->kb_off, (nk + 1) * 4)) return rc;
        if (int rc = ensure(b->kb_scores, std::max<size_t>(1, nk) * 8)) return rc;
        if (int rc = ensure(b->kb_count, (size_t)std::max(1, n_sent) * 4)) return rc;
    }

    const lt_constraints* cons = b->search_cons;
    const BeamPlan* P = nullptr;
    if (int rc = beam_plan(b, b->lcap, beam_size, kbest, cons != nullptr, &P)) return rc;
    b->last_beam_plan = P;
    if (!P->trail_smem)
        if (int rc = ensure(b->trail, nu * (size_t)beam_size * 8)) return rc;
    // span byte 0xFF (> LT_WINDOW) marks the ranks this search leaves unfilled (violation.cuh)
    if (b->hbm_trail) CU(cudaMemsetAsync(b->trail.p, 0xFF, nu * (size_t)beam_size * 8, st));

    unsigned int* ctl = static_cast<unsigned int*>(b->ctl.p);
    BeamArgs A{};
    A.text = b->d_text;
    A.sent_off = b->d_sent_off;
    A.n_sent = n_sent;
    A.units = P->units;
    A.beam = beam_size;
    A.warps = P->warps;
    A.pos = static_cast<const uint2*>(b->pos.p);
    A.edges = static_cast<const lt_edge*>(b->edges.p);
    A.status = static_cast<const int32_t*>(b->status.p);
    A.flags = ctl + kCtlFlags;
    A.trail = static_cast<uint64_t*>(b->trail.p);
    A.path_tmp = static_cast<lt_edge*>(b->path_tmp.p);
    A.path_len = static_cast<int32_t*>(b->path_len.p);
    A.scores = static_cast<double*>(b->scores.p);
    A.counters = static_cast<unsigned long long*>(b->counters.p);
    A.queue = ctl + kCtlBeamQueue;
    A.order = work_order(b);
    A.trail_smem = P->trail_smem ? 1 : 0;
    A.imp = b->imported ? static_cast<const H2*>(b->imp.p) : nullptr;
    A.kbest = kbest ? 1 : 0;
    A.kb_tmp = static_cast<lt_edge*>(b->kb_tmp.p);
    A.kb_len = static_cast<int32_t*>(b->kb_len.p);
    A.kb_scores = static_cast<double*>(b->kb_scores.p);
    A.kb_count = static_cast<int32_t*>(b->kb_count.p);
    if (cons) {
        // the search's statuses and the position descriptors of its constraints (constraints.cuh), from the lattice
        // as it stands: a rerun after a grown lattice prepares them again
        if (int rc = ensure(b->cons_status, (size_t)std::max(1, n_sent) * 4)) return rc;
        if (int rc = ensure(b->cons_desc, nu * 4)) return rc;
        ConstraintArgs C{};
        C.text = b->d_text;
        C.sent_off = b->d_sent_off;
        C.n_sent = n_sent;
        C.status = static_cast<const int32_t*>(b->status.p);
        C.flags = ctl + kCtlFlags;
        C.pos = static_cast<const uint2*>(b->pos.p);
        C.edges = static_cast<const lt_edge*>(b->edges.p);
        C.cons = static_cast<const lt_constraint*>(cons->cons.p);
        C.cons_off = static_cast<const int64_t*>(cons->off.p);
        C.search_status = static_cast<int32_t*>(b->cons_status.p);
        C.desc = static_cast<uint32_t*>(b->cons_desc.p);
        if (n_sent > 0) {
            const unsigned cgrid = (unsigned)std::min<int64_t>(((int64_t)n_sent + kConsWarps - 1) / kConsWarps, (int64_t)t->sm_count * 8);
            LT_LAUNCH(constraint_prep_kernel, cgrid, kConsWarps * 32, 0, st, C);
            CU(cudaGetLastError());
            b->launches += 1;
        }
        A.status = C.search_status;
        A.cdesc = C.desc;
    }

    const int64_t want_blocks = ((int64_t)n_sent + P->warps - 1) / P->warps;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want_blocks, (int64_t)t->sm_count * P->per_sm));

    // queue cursor and counters of this stage are zero after the batch prologue; a second search of the
    // same lattice resets them (path_len needs no clearing: the kernel writes every entry)
    if (!b->beam_state_clean) {
        LT_LAUNCH(beam_reset, 1, 32, 0, st, ctl + kCtlBeamQueue, static_cast<unsigned long long*>(b->counters.p) + 3, 4);
        CU(cudaGetLastError());
        b->launches += 1;
    }
    b->beam_state_clean = false;
    if (b->timed) CU(cudaEventRecord(b->ev[kEvBeamStart], st));
    if (n_sent > 0) {
        LT_LAUNCH(P->fn, grid, P->warps * 32, P->smem, st, t->dev, A);
        b->launches += 1;
    }
    CU(cudaGetLastError());
    if (b->timed) CU(cudaEventRecord(b->ev[kEvBeamEnd], st));
    if (n_sent > 0 && n_sent <= kPackScanMax) {
        // offsets and packing in one launch (scan.cuh: pack_paths_scan)
        const int ctas = (int)std::min<int64_t>(((int64_t)n_sent + 31) / 32, (int64_t)t->sm_count);
        const int per = (n_sent + ctas - 1) / ctas;
        LT_LAUNCH(pack_paths_scan, (unsigned)((n_sent + per - 1) / per), kPackScanThreads, 0, st, static_cast<const lt_edge*>(b->path_tmp.p),
                  b->d_sent_off, static_cast<const int32_t*>(b->path_len.p), static_cast<uint32_t*>(b->path_off.p), n_sent, per,
                  static_cast<lt_edge*>(b->path_out.p));
        CU(cudaGetLastError());
        b->launches += 1;
    } else {
    if (int rc = scan_u32(b, reinterpret_cast<const uint32_t*>(b->path_len.p), static_cast<uint32_t*>(b->path_off.p),
                          (int64_t)n_sent + 1, st))
        return rc;
    if (n_sent > 0) {
        const unsigned pgrid = (unsigned)std::min<int64_t>(((int64_t)n_sent + 7) / 8, (int64_t)t->sm_count * 8);
        LT_LAUNCH(pack_paths, pgrid, 256, 0, st, static_cast<const lt_edge*>(b->path_tmp.p), b->d_sent_off,
                  static_cast<const uint32_t*>(b->path_off.p), n_sent, static_cast<lt_edge*>(b->path_out.p));
        CU(cudaGetLastError());
        b->launches += 1;
    }
    }
    if (kbest) {
        // (kb_len[n_sent * beam] is the scan's sentinel entry; the kernel cannot know it is the last one)
        CU(cudaMemsetAsync(static_cast<int32_t*>(b->kb_len.p) + nk, 0, 4, st));
        if (int rc = scan_u32(b, reinterpret_cast<const uint32_t*>(b->kb_len.p), static_cast<uint32_t*>(b->kb_off.p), (int64_t)nk + 1, st))
            return rc;
        if (n_sent > 0) {
            const unsigned pgrid = (unsigned)std::min<int64_t>(((int64_t)nk + 7) / 8, (int64_t)t->sm_count * 8);
            LT_LAUNCH(pack_paths_k, pgrid, 256, 0, st, static_cast<const lt_edge*>(b->kb_tmp.p), b->d_sent_off,
                      static_cast<const uint32_t*>(b->kb_off.p), n_sent, beam_size, static_cast<lt_edge*>(b->kb_out.p));
            CU(cudaGetLastError());
            b->launches += 1;
        }
    }
    if (b->timed) CU(cudaEventRecord(b->ev[kEvPackEnd], st));
    b->have_paths = true;
    b->have_kbest = kbest;
    b->resolved = false;
    return LT_OK;
}

// The retry pass is meant for outliers: when more than 1 / 32 of a batch's sentences needed it, the main
// pass's staging area doubles for the batches to come (as long as the retry pass's is larger).
static void adapt_staging(lt_batch* b, unsigned int retried) {
    b->last_retried = retried;
    if (!b->use_retry || b->n_sent < 64) return;
    if (b->adapt_div > 0 && (uint64_t)retried * (uint64_t)b->adapt_div > (uint64_t)b->n_sent && b->hcap * 2 < b->retry_hcap) b->hcap *= 2;
}

static uint64_t cursor_of(const unsigned int* ctl) { return (uint64_t)ctl[kCtlCursor] | ((uint64_t)ctl[kCtlCursor + 1] << 32); }

// The control words say whether the lattice outgrew a buffer (edge array or per-warp staging); if so,
// enlarge it and run the stages again — still on the device; capacities are sticky for later batches.
// Returns 1 when a rerun was launched, 0 when the batch is complete, < 0 (negated code) on failure.
static int check_and_rerun(lt_batch* b, const unsigned int* ctl, cudaStream_t st) {
    const bool edge_over = ctl[kCtlFlags + kFlagEdgeOverflow] != 0;
    const bool stage_over = ctl[kCtlFlags + kFlagStageOverflow] != 0;
    if (!edge_over && !stage_over) {
        b->n_edges = (int64_t)cursor_of(ctl);
        b->resolved = true;
        adapt_staging(b, ctl[kCtlRetryCount]);
        return 0;
    }
    if (edge_over) {
        const uint64_t cur = cursor_of(ctl);
        const uint64_t need = cur + cur / 4 + 4096;
        if (need > 0xFFFFFFF0ull) return -fail(LT_ERR_CAPACITY, "the batch produces more than 2^32 lattice edges; split it");
        b->edge_cap = (uint32_t)need;
    }
    if (stage_over) {
        // first time: switch the two-pass scheme on (the main pass keeps its small staging area and its
        // residency); afterwards the retry pass's staging area doubles
        const int max_str = std::max(1, b->tables->dev.max_str);
        const int next = b->use_retry ? b->retry_hcap * 2 : std::max(512, b->hcap * 4);
        if (lattice_warp_smem(b->lcap + 8, next, max_str) > kSmemBudget)
            return -fail(LT_ERR_CAPACITY, "one eojeol yields more than %d lattice candidates; the staging buffer cannot grow further",
                         b->use_retry ? b->retry_hcap : b->hcap);
        b->use_retry = true;
        b->retry_hcap = next;
    }
    ++b->reruns;
    const bool want_paths = b->have_paths, want_kbest = b->have_kbest;
    if (int rc = launch_lattice(b, st)) return -rc;
    if (want_paths)
        if (int rc = launch_beam(b, st, want_kbest)) return -rc;
    return 1;
}

// Wait for the batch and settle its buffers (see check_and_rerun).
static int resolve(lt_batch* b) {
    if (!b->have_lattice || b->resolved) return LT_OK;
    cudaStream_t st = b->last_stream;
    for (int round = 0; round < 12; ++round) {
        unsigned int* ctl = b->h_ctl;
        CU(cudaMemcpyAsync(ctl, b->ctl.p, kCtlWords * sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        const int r = check_and_rerun(b, ctl, st);
        if (r < 0) return -r;
        if (r == 0) return LT_OK;
    }
    return fail(LT_ERR_CAPACITY, "lattice buffers did not converge");
}

extern "C" int lt_lattice(lt_batch* b, const uint16_t* d_text, const int32_t* d_sent_off, int32_t n_sent,
                          int64_t n_units, int32_t max_sent_units, void* stream) {
    if (!b || n_sent < 0 || n_units < 0 || max_sent_units < 0) return fail(LT_ERR_INVALID, "bad argument");
    if (n_sent > 0 && (!d_text || !d_sent_off)) return fail(LT_ERR_INVALID, "null input pointer");
    ON_DEVICE(b->tables->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    bind_batch(b, d_text, d_sent_off, n_sent, n_units, max_sent_units, st);
    return launch_lattice(b, st);
}

// a search of n_sent sentences against the bound constraint set (checked before anything is launched)
static int check_constraints(const lt_batch* b, int32_t n_sent) {
    if (b->cons && b->cons->n_sent != n_sent)
        return fail(LT_ERR_INVALID, "the bound constraint set has %d sentences, the search %d", b->cons->n_sent, n_sent);
    return LT_OK;
}

static int beam_entry(lt_batch* b, int32_t beam_size, void* stream, bool kbest) {
    if (!b || !b->have_lattice) return fail(LT_ERR_INVALID, "lt_beam needs a lattice: call lt_lattice first");
    if (beam_size < 1 || beam_size > LT_MAX_BEAM) return fail(LT_ERR_INVALID, "beam_size must be in 1..%d", LT_MAX_BEAM);
    if (int rc = check_constraints(b, b->n_sent)) return rc;
    ON_DEVICE(b->tables->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    b->last_stream = st;
    b->beam = beam_size;
    b->search_cons = b->cons;
    return launch_beam(b, st, kbest);
}

extern "C" int lt_beam(lt_batch* b, int32_t beam_size, void* stream) { return beam_entry(b, beam_size, stream, false); }
extern "C" int lt_beam_kbest(lt_batch* b, int32_t beam_size, void* stream) { return beam_entry(b, beam_size, stream, true); }

extern "C" int lt_tag_batch_device(lt_batch* b, const uint16_t* d_text, const int32_t* d_sent_off, int32_t n_sent,
                                   int64_t n_units, int32_t max_sent_units, int32_t beam_size, void* stream) {
    if (b)
        if (int rc = check_constraints(b, n_sent)) return rc;
    if (int rc = lt_lattice(b, d_text, d_sent_off, n_sent, n_units, max_sent_units, stream)) return rc;
    return lt_beam(b, beam_size, stream);
}

extern "C" int lt_lattice_size(lt_batch* b, int64_t* n_edges) {
    if (!b || !b->have_lattice || !n_edges) return fail(LT_ERR_INVALID, "no lattice");
    ON_DEVICE(b->tables->device);
    if (int rc = resolve(b)) return rc;
    *n_edges = b->n_edges;
    return LT_OK;
}

extern "C" int lt_lattice_fetch(lt_batch* b, lt_edge* edges, int64_t edge_cap, int64_t* end_off) {
    if (!b || !b->have_lattice) return fail(LT_ERR_INVALID, "no lattice");
    ON_DEVICE(b->tables->device);
    if (int rc = resolve(b)) return rc;
    if (edge_cap < b->n_edges) return fail(LT_ERR_CAPACITY, "edge buffer holds %lld, need %lld", (long long)edge_cap, (long long)b->n_edges);
    if (b->n_edges > 0 && !edges) return fail(LT_ERR_INVALID, "null output pointer");
    // the device keeps each sentence's edges wherever its reservation landed; hand them out in
    // sentence order (CSR by end position)
    std::vector<lt_edge> raw((size_t)b->n_edges);
    std::vector<uint2> pos((size_t)b->n_units + 1);
    if (b->n_edges) CU(cudaMemcpy(raw.data(), b->edges.p, raw.size() * sizeof(lt_edge), cudaMemcpyDeviceToHost));
    if (b->n_units) CU(cudaMemcpy(pos.data(), b->pos.p, (size_t)b->n_units * sizeof(uint2), cudaMemcpyDeviceToHost));
    int64_t out = 0;
    for (int64_t i = 0; i < b->n_units; ++i) {
        if (end_off) end_off[i] = out;
        const uint2 pc = pos[i];
        if ((int64_t)pc.x + pc.y > b->n_edges || out + pc.y > b->n_edges) return fail(LT_ERR_INVALID, "corrupt lattice index");
        for (uint32_t k = 0; k < pc.y; ++k) edges[out++] = raw[pc.x + k];
    }
    if (end_off) end_off[b->n_units] = out;
    return LT_OK;
}

extern "C" int lt_lattice_status(lt_batch* b, int32_t* status, int32_t* sent_len) {
    if (!b || !b->have_lattice) return fail(LT_ERR_INVALID, "no lattice");
    ON_DEVICE(b->tables->device);
    if (int rc = resolve(b)) return rc;
    if (b->n_sent == 0) return LT_OK;
    if (status) CU(cudaMemcpy(status, b->status.p, (size_t)b->n_sent * 4, cudaMemcpyDeviceToHost));
    if (sent_len) CU(cudaMemcpy(sent_len, b->sent_len.p, (size_t)b->n_sent * 4, cudaMemcpyDeviceToHost));
    return LT_OK;
}

extern "C" int lt_paths_size(lt_batch* b, int64_t* n_words) {
    if (!b || !b->have_paths || !n_words) return fail(LT_ERR_INVALID, "no paths");
    ON_DEVICE(b->tables->device);
    if (int rc = resolve(b)) return rc;
    uint32_t total = 0;
    CU(cudaMemcpyAsync(&total, static_cast<uint32_t*>(b->path_off.p) + b->n_sent, 4, cudaMemcpyDeviceToHost, b->last_stream));
    CU(cudaStreamSynchronize(b->last_stream));
    *n_words = total;
    return LT_OK;
}

// Results to the host in (normally) ONE round trip: the control words (overflow flags), the small
// per-sentence arrays and a speculative prefix of the path records — as many as the previous batch
// produced plus a margin — travel together; only when the batch holds more records than that (or
// needed a rerun) does a second copy follow.
static int fetch_paths(lt_batch* b, int32_t* path_off, lt_edge* path_edges, int64_t path_cap, double* scores,
                       int32_t* status, cudaStream_t st) {
    const int n = b->n_sent;
    if (!path_off || (n > 0 && (!scores || !status))) return fail(LT_ERR_INVALID, "null output pointer");
    if (n == 0) {
        path_off[0] = 0;
        return LT_OK;
    }
    unsigned int* ctl = b->h_ctl;
    int64_t copied = 0;
    for (int round = 0; round < 12; ++round) {
        int64_t guess = b->words_hint < 0 ? b->n_units / 2 + 64 : b->words_hint + b->words_hint / 8 + 64;
        guess = std::min<int64_t>(std::min<int64_t>(guess, path_cap), b->n_units);
        if (!path_edges) guess = 0;
        CU(cudaMemcpyAsync(ctl, b->ctl.p, kCtlWords * sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(path_off, b->path_off.p, (size_t)(n + 1) * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(scores, b->scores.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(status, search_status(b), (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        if (guess > 0) CU(cudaMemcpyAsync(path_edges, b->path_out.p, (size_t)guess * sizeof(lt_edge), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        copied = guess;
        const int r = check_and_rerun(b, ctl, st);
        if (r < 0) return -r;
        if (r == 0) break;
        if (round == 11) return fail(LT_ERR_CAPACITY, "lattice buffers did not converge");
    }
    const int64_t total = path_off[n];
    b->words_hint = total;
    if (total > path_cap) return fail(LT_ERR_CAPACITY, "path buffer holds %lld records, need %lld", (long long)path_cap, (long long)total);
    if (total > 0 && !path_edges) return fail(LT_ERR_INVALID, "null output pointer");
    if (total > copied) {
        CU(cudaMemcpyAsync(path_edges + copied, static_cast<const lt_edge*>(b->path_out.p) + copied, (size_t)(total - copied) * sizeof(lt_edge),
                           cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return LT_OK;
}

extern "C" int lt_paths_fetch(lt_batch* b, int32_t* path_off, lt_edge* path_edges, int64_t path_cap, double* scores,
                              int32_t* status) {
    if (!b || !b->have_paths) return fail(LT_ERR_INVALID, "no paths");
    ON_DEVICE(b->tables->device);
    return fetch_paths(b, path_off, path_edges, path_cap, scores, status, b->last_stream);
}

// All survivors of the last lt_beam_kbest (beam_search's return value, beam/beam.py:59-61).
extern "C" int lt_kbest_size(lt_batch* b, int64_t* n_words) {
    if (!b || !b->have_kbest || !n_words) return fail(LT_ERR_INVALID, "no k-best paths: call lt_beam_kbest first");
    ON_DEVICE(b->tables->device);
    if (int rc = resolve(b)) return rc;
    uint32_t total = 0;
    CU(cudaMemcpyAsync(&total, static_cast<uint32_t*>(b->kb_off.p) + (size_t)b->n_sent * b->beam, 4, cudaMemcpyDeviceToHost, b->last_stream));
    CU(cudaStreamSynchronize(b->last_stream));
    *n_words = total;
    return LT_OK;
}

extern "C" int lt_kbest_fetch(lt_batch* b, int32_t* n_best, int32_t* path_off, lt_edge* path_edges, int64_t path_cap,
                              double* scores, int32_t* status) {
    if (!b || !b->have_kbest) return fail(LT_ERR_INVALID, "no k-best paths: call lt_beam_kbest first");
    if (!path_off) return fail(LT_ERR_INVALID, "null output pointer");
    ON_DEVICE(b->tables->device);
    if (int rc = resolve(b)) return rc;
    const size_t n = (size_t)b->n_sent, nk = n * (size_t)b->beam;
    cudaStream_t st = b->last_stream;
    if (n == 0) {
        path_off[0] = 0;
        return LT_OK;
    }
    if (!n_best || !scores || !status) return fail(LT_ERR_INVALID, "null output pointer");
    CU(cudaMemcpyAsync(path_off, b->kb_off.p, (nk + 1) * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(n_best, b->kb_count.p, n * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(scores, b->kb_scores.p, nk * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(status, search_status(b), n * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const int64_t total = path_off[nk];
    if (total > path_cap) return fail(LT_ERR_CAPACITY, "path buffer holds %lld records, need %lld", (long long)path_cap, (long long)total);
    if (total > 0 && !path_edges) return fail(LT_ERR_INVALID, "null output pointer");
    if (total) CU(cudaMemcpyAsync(path_edges, b->kb_out.p, (size_t)total * sizeof(lt_edge), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return LT_OK;
}

// host text -> the batch's own buffers, bound as the input of the next lattice on the batch's own stream
static int bind_host_text(lt_batch* b, const uint16_t* text, const int32_t* sent_off, int32_t n_sent) {
    if (!sent_off || n_sent < 0) return fail(LT_ERR_INVALID, "bad argument");
    const int64_t n_units = sent_off[n_sent];
    if (n_units > 0 && !text) return fail(LT_ERR_INVALID, "null text pointer");
    int32_t max_units = 0;
    for (int32_t i = 0; i < n_sent; ++i) {
        const int32_t len = sent_off[i + 1] - sent_off[i];
        if (len < 0) return fail(LT_ERR_INVALID, "sent_off is not monotone at %d", i);
        max_units = std::max(max_units, len);
    }
    if (sent_off[0] != 0) return fail(LT_ERR_INVALID, "sent_off[0] must be 0");
    cudaStream_t st = b->own_stream;
    if (int rc = ensure(b->text, (size_t)std::max<int64_t>(1, n_units) * 2)) return rc;
    if (int rc = ensure(b->sent_off, (size_t)(n_sent + 1) * 4)) return rc;
    if (n_units) CU(cudaMemcpyAsync(b->text.p, text, (size_t)n_units * 2, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(b->sent_off.p, sent_off, (size_t)(n_sent + 1) * 4, cudaMemcpyHostToDevice, st));
    bind_batch(b, static_cast<const uint16_t*>(b->text.p), static_cast<const int32_t*>(b->sent_off.p), n_sent, n_units, max_units, st);
    return LT_OK;
}

// ... and its lattice
static int host_lattice(lt_batch* b, const uint16_t* text, const int32_t* sent_off, int32_t n_sent) {
    if (int rc = bind_host_text(b, text, sent_off, n_sent)) return rc;
    return launch_lattice(b, b->own_stream);
}

extern "C" int lt_tag_batch_host(lt_batch* b, const uint16_t* text, const int32_t* sent_off, int32_t n_sent,
                                 int32_t beam_size, int32_t* path_off, lt_edge* path_edges, int64_t path_cap,
                                 double* scores, int32_t* status) {
    if (!b) return fail(LT_ERR_INVALID, "bad argument");
    if (int rc = check_constraints(b, n_sent)) return rc;
    ON_DEVICE(b->tables->device);
    cudaStream_t st = b->own_stream;
    const bool timed = b->timed;
    if (timed) CU(cudaEventRecord(b->ev[kEvHostIn], st));
    if (int rc = host_lattice(b, text, sent_off, n_sent)) return rc;
    if (int rc = lt_beam(b, beam_size, st)) return rc;
    if (int rc = fetch_paths(b, path_off, path_edges, path_cap, scores, status, st)) return rc;
    if (timed) {
        CU(cudaEventRecord(b->ev[kEvHostOut], st));
        CU(cudaEventSynchronize(b->ev[kEvHostOut]));
    }
    return LT_OK;
}

// beam_search over a batch in HOST memory, all survivors kept on the device for lt_kbest_fetch
extern "C" int lt_tag_batch_host_kbest(lt_batch* b, const uint16_t* text, const int32_t* sent_off, int32_t n_sent,
                                       int32_t beam_size) {
    if (!b) return fail(LT_ERR_INVALID, "bad argument");
    if (int rc = check_constraints(b, n_sent)) return rc;
    ON_DEVICE(b->tables->device);
    if (int rc = host_lattice(b, text, sent_off, n_sent)) return rc;
    return lt_beam_kbest(b, beam_size, b->own_stream);
}

// sentence_lookup_as_begin_index for a batch in HOST memory: copies the text in and builds the lattices
// (results with lt_lattice_size / lt_lattice_fetch)
extern "C" int lt_lattice_host(lt_batch* b, const uint16_t* text, const int32_t* sent_off, int32_t n_sent) {
    if (!b) return fail(LT_ERR_INVALID, "bad argument");
    ON_DEVICE(b->tables->device);
    return host_lattice(b, text, sent_off, n_sent);
}

// The (word, morph0, morph1) strings that LT_EDGE_EXPLICIT records name (lt_lattice_import, lt_pathset_create),
// validated, then hashed.
static int hash_strings(const uint16_t* str_chars, const int64_t* str_off, int64_t n_strings, std::vector<H2>* out) {
    if (n_strings % 3 != 0 || (n_strings > 0 && (!str_chars || !str_off))) return fail(LT_ERR_INVALID, "strings come in (word, morph0, morph1) triples");
    if (n_strings > 0 && str_off[0] < 0) return fail(LT_ERR_INVALID, "str_off[0] is negative");
    out->resize((size_t)n_strings);
    for (int64_t i = 0; i < n_strings; ++i) {
        if (str_off[i + 1] < str_off[i]) return fail(LT_ERR_INVALID, "str_off is not monotone at %lld", (long long)i);
        (*out)[(size_t)i] = hash_units(str_chars + str_off[i], str_off[i + 1] - str_off[i]);
    }
    return LT_OK;
}

// What is wrong with a given word record (nullptr: nothing): its tags, and the strings 3 * rule .. 3 * rule + 2
// of an LT_EDGE_EXPLICIT record.
static const char* check_explicit(const lt_edge& ed, int64_t n_strings, int n_tags) {
    if (ed.tag0 >= n_tags || (ed.tag1 != LT_NO_TAG && ed.tag1 >= n_tags)) return "tag id out of range";
    if ((ed.flags & LT_EDGE_EXPLICIT) && (int64_t)ed.rule * 3 + 2 >= n_strings) return "string index out of range";
    return nullptr;
}

// beam_search's `bindex` argument: a lattice built by the caller (see include/lt_b200.h)
extern "C" int lt_lattice_import(lt_batch* b, const uint16_t* text, const int32_t* sent_off, int32_t n_sent,
                                 const lt_edge* edges, const int64_t* end_off, const uint16_t* str_chars,
                                 const int64_t* str_off, int64_t n_strings) {
    if (!b || !end_off || n_strings < 0) return fail(LT_ERR_INVALID, "bad argument");
    ON_DEVICE(b->tables->device);
    if (int rc = bind_host_text(b, text, sent_off, n_sent)) return rc;
    cudaStream_t st = b->own_stream;
    const int64_t n_units = b->n_units;
    const int64_t n_edges = end_off[n_units];
    if (n_edges < 0 || n_edges > 0xFFFFFFF0ll) return fail(LT_ERR_INVALID, "edge count out of range");
    if (end_off[0] < 0) return fail(LT_ERR_INVALID, "end_off[0] is negative");
    if (n_edges > 0 && !edges) return fail(LT_ERR_INVALID, "null edge pointer");
    std::vector<H2> hashes;
    if (int rc = hash_strings(str_chars, str_off, n_strings, &hashes)) return rc;

    // CSR rows, per-sentence status and syllable counts, validated on the host
    std::vector<uint2> pos((size_t)n_units + 1, make_uint2(0u, 0u));
    std::vector<int32_t> status((size_t)std::max(1, n_sent), LT_SENT_OK), slen((size_t)std::max(1, n_sent), 0), sedges((size_t)std::max(1, n_sent), 0);
    const int n_tags = b->tables->dev.n_tags;
    for (int32_t s = 0; s < n_sent; ++s) {
        const int32_t s0 = sent_off[s], s1 = sent_off[s + 1];
        int32_t L = 0;
        bool bad = false;
        for (int32_t i = s0; i < s1; ++i) {
            const uint32_t c = text[i];
            if (c == 0x20u) continue;
            ++L;
            bad |= (c >= 0x09 && c <= 0x0D) || (c >= 0x1C && c <= 0x1F) || c == 0x85 || c == 0xA0 || c == 0x1680 ||
                   (c >= 0x2000 && c <= 0x200A) || c == 0x2028 || c == 0x2029 || c == 0x202F || c == 0x205F || c == 0x3000;
        }
        slen[s] = L;
        int64_t total = 0;
        for (int32_t p = 0; p < s1 - s0; ++p) {
            const int64_t lo = end_off[s0 + p], hi = end_off[s0 + p + 1];
            if (lo > hi || hi > n_edges) return fail(LT_ERR_INVALID, "end_off is not monotone at unit %d", s0 + p);
            if (hi > lo && p >= L) return fail(LT_ERR_INVALID, "sentence %d has edges ending beyond its %d syllables", s, L);
            pos[(size_t)s0 + p] = make_uint2((uint32_t)lo, (uint32_t)(hi - lo));
            uint32_t prev_b = 0;
            for (int64_t k = lo; k < hi; ++k) {
                const lt_edge& ed = edges[k];
                if (ed.e != p + 1 || ed.b >= ed.e) return fail(LT_ERR_INVALID, "edge %lld: span [%d, %d) does not end at syllable %d", (long long)k, ed.b, ed.e, p + 1);
                if (k > lo && ed.b < prev_b) return fail(LT_ERR_INVALID, "edge %lld: edges of one end position must be sorted by begin", (long long)k);
                prev_b = ed.b;
                if (const char* why = check_explicit(ed, n_strings, n_tags)) return fail(LT_ERR_INVALID, "edge %lld: %s", (long long)k, why);
                if (!(ed.flags & LT_EDGE_EXPLICIT) && (ed.flags & LT_EDGE_LEMMA) && ed.rule != LT_NO_RULE)
                    return fail(LT_ERR_INVALID, "edge %lld: imported lemma edges name their morphemes (LT_EDGE_EXPLICIT)", (long long)k);
            }
            total += hi - lo;
        }
        sedges[s] = (int32_t)std::min<int64_t>(total, 0x7FFFFFFF);
        if (s1 - s0 > b->lcap) status[s] = LT_SENT_TOO_LONG;
        else if (bad) status[s] = LT_SENT_BAD_SPACE;
        else if (L > 0 && total == 0) status[s] = LT_SENT_NO_EDGES;
    }

    // control words / counters zeroed and the work order computed, exactly as before a device-built lattice
    if (b->edge_cap < (uint64_t)n_edges + 16) b->edge_cap = (uint32_t)(n_edges + 16);
    if (int rc = ensure(b->edges, (size_t)b->edge_cap * sizeof(lt_edge))) return rc;
    if (int rc = ensure(b->imp, std::max<size_t>(1, hashes.size()) * sizeof(H2))) return rc;
    if (int rc = start_batch(b, st)) return rc;
    CU(cudaMemcpyAsync(b->pos.p, pos.data(), pos.size() * sizeof(uint2), cudaMemcpyHostToDevice, st));
    if (n_edges) CU(cudaMemcpyAsync(b->edges.p, edges, (size_t)n_edges * sizeof(lt_edge), cudaMemcpyHostToDevice, st));
    if (n_sent) {
        CU(cudaMemcpyAsync(b->status.p, status.data(), (size_t)n_sent * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(b->sent_len.p, slen.data(), (size_t)n_sent * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(b->sent_edges.p, sedges.data(), (size_t)n_sent * 4, cudaMemcpyHostToDevice, st));
    }
    if (!hashes.empty()) CU(cudaMemcpyAsync(b->imp.p, hashes.data(), hashes.size() * sizeof(H2), cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));          // the staging vectors above go out of scope
    b->have_lattice = true;
    b->imported = true;
    b->resolved = true;
    b->n_edges = n_edges;
    return LT_OK;
}

extern "C" int lt_batch_counters(lt_batch* b, lt_counters* out) {
    if (!b || !out) return fail(LT_ERR_INVALID, "null argument");
    ON_DEVICE(b->tables->device);
    unsigned long long c[8] = {0};
    if (b->counters.p && b->have_lattice) {
        if (int rc = resolve(b)) return rc;
        CU(cudaMemcpy(c, b->counters.p, sizeof c, cudaMemcpyDeviceToHost));
    }
    out->sentences = (uint64_t)b->n_sent;
    out->L = c[0]; out->P = c[1]; out->E = c[2]; out->T = c[3]; out->F = c[4]; out->Bk = c[5]; out->W = c[6];
    return LT_OK;
}

// State of the workspace: buffer capacities, rerun and launch counts, the launch shapes of the last batch.
extern "C" int lt_batch_info(lt_batch* b, lt_info* out) {
    if (!b || !out) return fail(LT_ERR_INVALID, "null argument");
    ON_DEVICE(b->tables->device);
    memset(out, 0, sizeof *out);
    if (b->have_lattice)
        if (int rc = resolve(b)) return rc;
    out->launches = b->launches;
    out->reruns = b->reruns;
    out->hcap = b->hcap;
    out->retry_hcap = b->use_retry ? b->retry_hcap : 0;
    out->retried = (int32_t)b->last_retried;
    out->edge_cap = (int64_t)b->edge_cap;
    out->n_edges = b->n_edges;
    out->unit_limit = unit_limit(b->tables);
    if (const LatticePlan* p = b->last_lattice_plan) {
        out->lattice_warps = p->warps;
        out->lattice_ctas_per_sm = p->per_sm;
        out->lattice_smem = (int32_t)p->smem;
    }
    if (const BeamPlan* p = b->last_beam_plan) {
        out->beam_warps = p->warps;
        out->beam_ctas_per_sm = p->per_sm;
        out->beam_smem = (int32_t)p->smem;
        out->beam_trail_smem = p->trail_smem ? 1 : 0;
    }
    out->sm_count = b->tables->sm_count;
    return LT_OK;
}

extern "C" int lt_batch_set_stage_timing(lt_batch* b, int32_t on) {
    if (!b) return fail(LT_ERR_INVALID, "null argument");
    b->timed = on != 0;
    return LT_OK;
}

// timings: enabled by the first call (so that un-timed batches record no events)
extern "C" int lt_batch_timings(lt_batch* b, lt_timings* out) {
    if (!b || !out) return fail(LT_ERR_INVALID, "null argument");
    ON_DEVICE(b->tables->device);
    memset(out, 0, sizeof *out);
    if (!b->timed) {
        b->timed = true;      // subsequent batches are timed
        return LT_OK;
    }
    if (!b->have_paths) return LT_OK;
    if (int rc = resolve(b)) return rc;
    auto ms = [&](int a, int c, float* dst) {
        float v = 0.f;
        if (cudaEventElapsedTime(&v, b->ev[a], b->ev[c]) == cudaSuccess) *dst = v;
        else cudaGetLastError();
    };
    ms(kEvLatticeStart, kEvLatticeEnd, &out->ms_lattice);
    ms(kEvBeamStart, kEvBeamEnd, &out->ms_beam);
    ms(kEvBeamEnd, kEvPackEnd, &out->ms_pack);
    ms(kEvHostIn, kEvLatticeStart, &out->ms_h2d);
    ms(kEvPackEnd, kEvHostOut, &out->ms_d2h);
    ms(kEvHostIn, kEvHostOut, &out->ms_total);
    return LT_OK;
}

// ------------------------------------------------------------------------------------------------
// constraint sets (constraints.cuh): spans the search must keep as words
// ------------------------------------------------------------------------------------------------
extern "C" void lt_constraints_destroy(lt_constraints* c) {
    if (!c) return;
    DeviceGuard guard(c->device);      // (the tables may be gone already)
    delete c;
}

extern "C" int lt_constraints_create(lt_tables* t, int32_t n_sent, const lt_constraint* cons, const int64_t* cons_off,
                                     lt_constraints** out) {
    if (!t || !out || !cons_off || n_sent < 0) return fail(LT_ERR_INVALID, "bad argument");
    *out = nullptr;
    if (cons_off[0] != 0) return fail(LT_ERR_INVALID, "cons_off[0] must be 0");
    for (int32_t s = 0; s < n_sent; ++s)
        if (cons_off[s + 1] < cons_off[s]) return fail(LT_ERR_INVALID, "cons_off is not monotone at sentence %d", s);
    const int64_t n_cons = cons_off[n_sent];
    if (n_cons > 0 && !cons) return fail(LT_ERR_INVALID, "null constraint pointer");
    const int n_tags = t->dev.n_tags;
    for (int32_t s = 0; s < n_sent; ++s)
        for (int64_t i = cons_off[s]; i < cons_off[s + 1]; ++i) {
            const lt_constraint& c = cons[i];
            const int64_t k = i - cons_off[s];
            if (c.e <= c.b || c.e - c.b > LT_WINDOW)
                return fail(LT_ERR_INVALID, "sentence %d, constraint %lld: span [%d, %d) is not 1..%d syllables", s, (long long)k, c.b, c.e,
                            LT_WINDOW);
            if (c.tag != LT_NO_TAG && (c.tag >= n_tags || c.tag == LT_TAG_BOS || c.tag == LT_TAG_EOS || c.tag == LT_TAG_UNK))
                return fail(LT_ERR_INVALID, "sentence %d, constraint %lld: tag %d is not a word tag of the tables (nor LT_NO_TAG)", s,
                            (long long)k, c.tag);
            if (k > 0 && cons[i - 1].e > c.b)
                return fail(LT_ERR_INVALID, "sentence %d, constraint %lld: begins at %d, before the previous one ends (%d); constraints are "
                                            "sorted by b and do not overlap", s, (long long)k, c.b, cons[i - 1].e);
        }
    ON_DEVICE(t->device);
    lt_constraints* c = new lt_constraints();
    c->tables = t;
    c->device = t->device;
    c->n_sent = n_sent;
    int rc = upload_once(c->cons, cons, (size_t)n_cons * sizeof(lt_constraint));
    if (rc == LT_OK) rc = upload_once(c->off, cons_off, (size_t)(n_sent + 1) * 8);
    if (rc != LT_OK) {
        delete c;
        return rc;
    }
    *out = c;
    return LT_OK;
}

extern "C" int lt_batch_set_constraints(lt_batch* b, const lt_constraints* c) {
    if (!b) return fail(LT_ERR_INVALID, "null argument");
    if (c && c->tables != b->tables) return fail(LT_ERR_INVALID, "the constraint set belongs to other tables");
    b->cons = c;
    return LT_OK;
}

// ------------------------------------------------------------------------------------------------
// path sets: scoring / featurizing given paths, the perceptron step (paths.cuh)
// ------------------------------------------------------------------------------------------------
struct lt_pathset {
    lt_tables* tables = nullptr;
    int device = 0;
    int32_t n_paths = 0;
    int64_t n_words = 0;
    bool ordered = true;            // every path: b < e, b strictly increasing (lt_evaluate needs it)
    DevBuf off, edges, hashes;      // [n_paths + 1] offsets, [n_words] records, [n_strings] string hashes
};

extern "C" void lt_pathset_destroy(lt_pathset* p) {
    if (!p) return;
    DeviceGuard guard(p->device);      // (the tables may be gone already)
    delete p;
}

extern "C" int lt_pathset_create(lt_tables* t, int32_t n_paths, const lt_edge* edges, const int64_t* path_off,
                                 const uint16_t* str_chars, const int64_t* str_off, int64_t n_strings, lt_pathset** out) {
    if (!t || !out || !path_off || n_paths < 0 || n_strings < 0) return fail(LT_ERR_INVALID, "bad argument");
    *out = nullptr;
    if (path_off[0] != 0) return fail(LT_ERR_INVALID, "path_off[0] must be 0");
    for (int32_t p = 0; p < n_paths; ++p)
        if (path_off[p + 1] < path_off[p]) return fail(LT_ERR_INVALID, "path_off is not monotone at %d", p);
    const int64_t n_words = path_off[n_paths];
    if (n_words > 0 && !edges) return fail(LT_ERR_INVALID, "null edge pointer");
    std::vector<H2> hashes;
    if (int rc = hash_strings(str_chars, str_off, n_strings, &hashes)) return rc;
    for (int64_t w = 0; w < n_words; ++w) {
        const lt_edge& ed = edges[w];
        if (!(ed.flags & LT_EDGE_EXPLICIT)) return fail(LT_ERR_INVALID, "word %lld is not LT_EDGE_EXPLICIT", (long long)w);
        if (const char* why = check_explicit(ed, n_strings, t->dev.n_tags)) return fail(LT_ERR_INVALID, "word %lld: %s", (long long)w, why);
    }
    bool ordered = true;
    for (int32_t q = 0; q < n_paths && ordered; ++q)
        for (int64_t w = path_off[q]; w < path_off[q + 1] && ordered; ++w)
            ordered = edges[w].b < edges[w].e && (w == path_off[q] || edges[w - 1].b < edges[w].b);
    ON_DEVICE(t->device);
    lt_pathset* p = new lt_pathset();
    p->tables = t;
    p->device = t->device;
    p->n_paths = n_paths;
    p->n_words = n_words;
    p->ordered = ordered;
    int rc = upload_once(p->off, path_off, (size_t)(n_paths + 1) * 8);
    if (rc == LT_OK) rc = upload_once(p->edges, edges, (size_t)n_words * sizeof(lt_edge));
    if (rc == LT_OK) rc = upload_once(p->hashes, hashes.data(), hashes.size() * sizeof(H2));
    if (rc != LT_OK) {
        delete p;
        return rc;
    }
    *out = p;
    return LT_OK;
}

static int check_trigram_func(const lt_tables* t, int32_t func) {
    if (func < 0 || func >= t->dev.n_funcs || t->dev.funcs[func].kind != LT_FUNC_TRIGRAM)
        return fail(LT_ERR_INVALID, "func %d is not an LT_FUNC_TRIGRAM scorer", func);
    return LT_OK;
}

// hits: slots of the hashed table, then the dense blocks' doubles
static uint32_t feat_slots(const lt_tables* t) { return (uint32_t)(t->dev.feat_mask + 1); }
static size_t n_hits(const lt_tables* t) {
    return (size_t)feat_slots(t) + (size_t)t->dev.n_tri * (size_t)dense_block_bytes(t->dev.n_tags) / 8;
}

static unsigned warp_grid(const lt_tables* t, int64_t n_warps) {
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n_warps + 7) / 8, (int64_t)t->sm_count * 8));
}

extern "C" int lt_pathset_eval(lt_batch* b, const lt_pathset* paths, int32_t func, double* scores, int64_t* feat_off,
                               int32_t* feat_idx, int64_t feat_cap) {
    if (!b || !paths) return fail(LT_ERR_INVALID, "null argument");
    if (paths->tables != b->tables) return fail(LT_ERR_INVALID, "the path set belongs to other tables");
    if (paths->n_paths > 0 && !scores) return fail(LT_ERR_INVALID, "null output pointer");
    lt_tables* t = b->tables;
    const bool want_feat = feat_off != nullptr;
    if (want_feat) {
        if (int rc = check_trigram_func(t, func)) return rc;
        if (feat_cap < 0 || (feat_cap > 0 && !feat_idx)) return fail(LT_ERR_INVALID, "bad feature buffer");
    }
    ON_DEVICE(t->device);
    cudaStream_t st = b->own_stream;
    const int64_t nw = paths->n_words;
    if (int rc = ensure(b->pth_scores, (size_t)std::max(1, paths->n_paths) * 8)) return rc;
    if (want_feat) {
        if (!t->d_hit_feat.p) {
            std::vector<int32_t> inv(n_hits(t), -1);
            for (size_t i = 0; i < t->feat_dst.size(); ++i) {
                const uint32_t d = t->feat_dst[i];
                if (d != kDstNone) inv[(d & kDstDense) ? feat_slots(t) + (d & ~kDstDense) : d] = (int32_t)i;
            }
            if (int rc = upload_once(t->d_hit_feat, inv.data(), inv.size() * 4)) return rc;
        }
        if (int rc = ensure(b->pth_feat, (size_t)std::max<int64_t>(1, nw) * 9 * 4)) return rc;
        if (int rc = ensure(b->pth_nfeat, (size_t)std::max<int64_t>(1, nw))) return rc;
    }
    PathEvalArgs A{};
    A.edges = static_cast<const lt_edge*>(paths->edges.p);
    A.off = static_cast<const int64_t*>(paths->off.p);
    A.hashes = static_cast<const H2*>(paths->hashes.p);
    A.n_paths = paths->n_paths;
    A.func = want_feat ? func : -1;
    A.scores = static_cast<double*>(b->pth_scores.p);
    A.feat = want_feat ? static_cast<int32_t*>(b->pth_feat.p) : nullptr;
    A.nfeat = static_cast<uint8_t*>(b->pth_nfeat.p);
    A.hit_feat = static_cast<const int32_t*>(t->d_hit_feat.p);
    if (paths->n_paths > 0) {
        LT_LAUNCH(path_eval_kernel, warp_grid(t, paths->n_paths), 256, 0, st, t->dev, A);
        CU(cudaGetLastError());
        b->launches += 1;
        CU(cudaMemcpyAsync(scores, A.scores, (size_t)paths->n_paths * 8, cudaMemcpyDeviceToHost, st));
    }
    std::vector<int32_t> feat;
    std::vector<uint8_t> nfeat;
    if (want_feat && nw > 0) {
        feat.resize((size_t)nw * 9);
        nfeat.resize((size_t)nw);
        CU(cudaMemcpyAsync(feat.data(), A.feat, feat.size() * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(nfeat.data(), A.nfeat, nfeat.size(), cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    if (want_feat) {
        int64_t total = 0;
        for (int64_t w = 0; w < nw; ++w) total += nfeat[(size_t)w];
        if (total > feat_cap) return fail(LT_ERR_CAPACITY, "feature buffer holds %lld, need %lld", (long long)feat_cap, (long long)total);
        int64_t o = 0;
        for (int64_t w = 0; w < nw; ++w) {
            feat_off[w] = o;
            for (int i = 0; i < nfeat[(size_t)w]; ++i) feat_idx[o++] = feat[(size_t)w * 9 + i];
        }
        feat_off[nw] = o;
    }
    return LT_OK;
}

// lt_perceptron_delta / lt_evaluate: the best paths of the last search next to one gold path per sentence
static int check_gold(const lt_batch* b, const lt_pathset* gold) {
    if (!b->have_paths) return fail(LT_ERR_INVALID, "no paths: run a search (lt_tag_batch_host, lt_beam, ...) first");
    if (b->search_cons)
        return fail(LT_ERR_INVALID, "the last search was constrained: its paths are not the ones this compares against gold paths");
    if (gold->tables != b->tables) return fail(LT_ERR_INVALID, "the gold path set belongs to other tables");
    if (gold->n_paths != b->n_sent) return fail(LT_ERR_INVALID, "%d gold paths for %d sentences", gold->n_paths, b->n_sent);
    return LT_OK;
}

// ... and what their kernels read of both, with the sentence scratch sized for the batch
static int search_and_gold(lt_batch* b, const lt_pathset* gold, SearchAndGold* g) {
    const size_t nu = (size_t)b->n_units, n_sent = (size_t)b->n_sent;
    if (int rc = ensure(b->pth_ch, std::max<size_t>(1, nu) * 2)) return rc;
    if (int rc = ensure(b->pth_ha, (nu + n_sent + 1) * 8)) return rc;
    if (int rc = ensure(b->pth_hb, (nu + n_sent + 1) * 8)) return rc;
    g->text = b->d_text;
    g->sent_off = b->d_sent_off;
    g->n_sent = b->n_sent;
    g->status = static_cast<const int32_t*>(b->status.p);
    g->path_off = static_cast<const uint32_t*>(b->path_off.p);
    g->path_edges = static_cast<const lt_edge*>(b->path_out.p);
    g->imp = b->imported ? static_cast<const H2*>(b->imp.p) : nullptr;
    g->gold_edges = static_cast<const lt_edge*>(gold->edges.p);
    g->gold_off = static_cast<const int64_t*>(gold->off.p);
    g->gold_hashes = static_cast<const H2*>(gold->hashes.p);
    g->ch = static_cast<uint16_t*>(b->pth_ch.p);
    g->ha = static_cast<uint64_t*>(b->pth_ha.p);
    g->hb = static_cast<uint64_t*>(b->pth_hb.p);
    return LT_OK;
}

extern "C" int lt_perceptron_delta(lt_batch* b, const lt_pathset* gold, int32_t func, int64_t* delta, int64_t n_delta,
                                   uint8_t* differs, int64_t* n_differ) {
    if (!b || !gold || !n_differ) return fail(LT_ERR_INVALID, "null argument");
    if (int rc = check_gold(b, gold)) return rc;
    lt_tables* t = b->tables;
    if (int rc = check_trigram_func(t, func)) return rc;
    if ((size_t)n_delta != t->feat_dst.size())
        return fail(LT_ERR_INVALID, "the tables were built with %zu features, delta has %lld", t->feat_dst.size(), (long long)n_delta);
    if ((n_delta > 0 && !delta) || (b->n_sent > 0 && !differs)) return fail(LT_ERR_INVALID, "null output pointer");
    ON_DEVICE(t->device);
    if (int rc = resolve(b)) return rc;
    cudaStream_t st = b->last_stream;
    const int n_sent = b->n_sent;
    PerceptronArgs A{};
    if (int rc = search_and_gold(b, gold, &A.sg)) return rc;
    if (int rc = ensure(t->d_counts, n_hits(t) * 8)) return rc;
    if (int rc = upload_feat_dst(t)) return rc;
    if (int rc = ensure(b->pc_delta, (size_t)std::max<int64_t>(1, n_delta) * 8)) return rc;
    if (int rc = ensure(b->pc_differs, (size_t)std::max(1, n_sent))) return rc;
    if (int rc = ensure(b->pc_count, 8)) return rc;
    CU(cudaMemsetAsync(t->d_counts.p, 0, n_hits(t) * 8, st));
    CU(cudaMemsetAsync(b->pc_count.p, 0, 8, st));
    A.func = func;
    A.counts = static_cast<unsigned long long*>(t->d_counts.p);
    A.differs = static_cast<uint8_t*>(b->pc_differs.p);
    A.n_differ = static_cast<unsigned long long*>(b->pc_count.p);
    if (n_sent > 0) {
        LT_LAUNCH(perceptron_kernel, warp_grid(t, n_sent), 256, 0, st, t->dev, A);
        CU(cudaGetLastError());
        b->launches += 1;
    }
    if (n_delta > 0) {
        const unsigned grid = (unsigned)std::min<int64_t>((n_delta + 255) / 256, (int64_t)t->sm_count * 16);
        LT_LAUNCH(gather_counts, grid, 256, 0, st, A.counts, static_cast<const uint32_t*>(t->d_feat_dst.p), n_delta, feat_slots(t),
                  static_cast<long long*>(b->pc_delta.p));
        CU(cudaGetLastError());
        b->launches += 1;
        CU(cudaMemcpyAsync(delta, b->pc_delta.p, (size_t)n_delta * 8, cudaMemcpyDeviceToHost, st));
    }
    unsigned long long nd = 0;
    if (n_sent > 0) CU(cudaMemcpyAsync(differs, b->pc_differs.p, (size_t)n_sent, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&nd, b->pc_count.p, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *n_differ = (int64_t)nd;
    return LT_OK;
}

// The best paths of the last search against gold paths (evaluate.cuh): class, counts, image scores and reason
// codes per sentence / gold word.
extern "C" int lt_evaluate(lt_batch* b, const lt_pathset* gold, uint8_t* sent_class, int32_t* counts, double* gold_scores,
                           uint8_t* word_reason) {
    if (!b || !gold) return fail(LT_ERR_INVALID, "null argument");
    if (int rc = check_gold(b, gold)) return rc;
    if (!gold->ordered) return fail(LT_ERR_INVALID, "a gold path has a word with b >= e or a b that does not increase");
    if (b->n_sent > 0 && !sent_class) return fail(LT_ERR_INVALID, "null output pointer");
    lt_tables* t = b->tables;
    ON_DEVICE(t->device);
    if (int rc = resolve(b)) return rc;
    cudaStream_t st = b->last_stream;
    const int n_sent = b->n_sent;
    const size_t nw = (size_t)gold->n_words;
    EvaluateArgs A{};
    if (int rc = search_and_gold(b, gold, &A.sg)) return rc;
    if (int rc = ensure(b->ev_image, std::max<size_t>(1, nw) * sizeof(lt_edge))) return rc;
    if (int rc = ensure(b->ev_class, (size_t)std::max(1, n_sent))) return rc;
    if (counts)
        if (int rc = ensure(b->ev_counts, (size_t)std::max(1, n_sent) * LT_EVAL_N_COUNTS * 4)) return rc;
    if (gold_scores)
        if (int rc = ensure(b->ev_scores, (size_t)std::max(1, n_sent) * 8)) return rc;
    if (word_reason)
        if (int rc = ensure(b->ev_reason, std::max<size_t>(1, nw))) return rc;
    A.scores = static_cast<const double*>(b->scores.p);
    A.pos = static_cast<const uint2*>(b->pos.p);
    A.edges = static_cast<const lt_edge*>(b->edges.p);
    A.image = static_cast<lt_edge*>(b->ev_image.p);
    A.sent_class = static_cast<uint8_t*>(b->ev_class.p);
    A.counts = counts ? static_cast<int32_t*>(b->ev_counts.p) : nullptr;
    A.gold_scores = gold_scores ? static_cast<double*>(b->ev_scores.p) : nullptr;
    A.word_reason = word_reason ? static_cast<uint8_t*>(b->ev_reason.p) : nullptr;
    if (n_sent > 0) {
        LT_LAUNCH(evaluate_kernel, warp_grid(t, n_sent), 256, 0, st, t->dev, A);
        CU(cudaGetLastError());
        b->launches += 1;
        CU(cudaMemcpyAsync(sent_class, A.sent_class, (size_t)n_sent, cudaMemcpyDeviceToHost, st));
        if (counts) CU(cudaMemcpyAsync(counts, A.counts, (size_t)n_sent * LT_EVAL_N_COUNTS * 4, cudaMemcpyDeviceToHost, st));
        if (gold_scores) CU(cudaMemcpyAsync(gold_scores, A.gold_scores, (size_t)n_sent * 8, cudaMemcpyDeviceToHost, st));
        if (word_reason && nw > 0) CU(cudaMemcpyAsync(word_reason, A.word_reason, nw, cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    return LT_OK;
}

// ------------------------------------------------------------------------------------------------
// mini-batch perceptron (train.cuh): weights and their running average in device memory
// ------------------------------------------------------------------------------------------------
struct lt_trainer {
    lt_tables* tables = nullptr;
    int device = 0;
    const lt_pathset* gold = nullptr;
    int32_t func = 0;
    int32_t n_sent = 0;
    int64_t n_coef = 0;
    int64_t steps = 0;
    std::vector<int32_t> sent_off;          // host copy: the size and longest sentence of a step's slice
    DevBuf text, off;                       // the corpus
    DevBuf feat_coef, w, u, acc;            // [n_feat] coefficient of each desc feature; [n_coef] w, u, step counts
    DevBuf differs, mistakes;               // [n_sent] flags of each sentence's last step; running count of mistakes
    int32_t mode = LT_UPDATE_FULL;          // lt_trainer_set_update
    std::vector<int64_t> gold_off;          // host copy: W of each sentence
    std::vector<uint8_t> full_last;         // [n_sent] the last step that covered the sentence was LT_UPDATE_FULL
    DevBuf prefix_words, violation;         // [n_sent] of the last EARLY / MAX_VIOLATION step that covered the sentence
    DevBuf gscore, chain;                   // violation_kernel scratch: [gold n_words] G_m, [step units] a rank-0 hypothesis
    cudaEvent_t done = nullptr;             // recorded after the last kernel of every step
};

extern "C" void lt_trainer_destroy(lt_trainer* tr) {
    if (!tr) return;
    DeviceGuard guard(tr->device);      // (the tables may be gone already)
    if (tr->done) cudaEventDestroy(tr->done);
    delete tr;
}

static int zeroed(DevBuf& b, size_t bytes) {
    if (int rc = ensure(b, std::max<size_t>(bytes, 16))) return rc;
    CU(cudaMemsetAsync(b.p, 0, std::max<size_t>(bytes, 16), nullptr));
    return LT_OK;
}

// the tables' weight of every trained feature := w[feat_coef[i]], on stream st
static int scatter_trainer_weights(lt_trainer* tr, cudaStream_t st) {
    lt_tables* t = tr->tables;
    const int64_t n_feat = (int64_t)t->feat_dst.size();
    if (n_feat == 0) return LT_OK;
    const unsigned grid = (unsigned)std::min<int64_t>((n_feat + 255) / 256, (int64_t)t->sm_count * 16);
    LT_LAUNCH(scatter_coef, grid, 256, 0, st, const_cast<FeatSlot*>(t->dev.feat),
              reinterpret_cast<double*>(const_cast<unsigned char*>(t->dev.dense)), static_cast<const uint32_t*>(t->d_feat_dst.p),
              static_cast<const int64_t*>(tr->feat_coef.p), n_feat, static_cast<const double*>(tr->w.p));
    CU(cudaGetLastError());
    return LT_OK;
}

extern "C" int lt_trainer_create(lt_tables* t, int32_t func, const uint16_t* text, const int32_t* sent_off, int32_t n_sent,
                                 const lt_pathset* gold, int64_t n_coef, const int64_t* feat_coef, const double* coef,
                                 lt_trainer** out) {
    if (!t || !out || !gold || !sent_off || n_sent < 0 || n_coef < 0) return fail(LT_ERR_INVALID, "bad argument");
    *out = nullptr;
    if (int rc = check_trigram_func(t, func)) return rc;
    if (gold->tables != t) return fail(LT_ERR_INVALID, "the gold path set belongs to other tables");
    if (gold->n_paths != n_sent) return fail(LT_ERR_INVALID, "%d gold paths for %d sentences", gold->n_paths, n_sent);
    if (sent_off[0] != 0) return fail(LT_ERR_INVALID, "sent_off[0] must be 0");
    for (int32_t i = 0; i < n_sent; ++i)
        if (sent_off[i + 1] < sent_off[i]) return fail(LT_ERR_INVALID, "sent_off is not monotone at %d", i);
    const int64_t n_units = sent_off[n_sent];
    const int64_t n_feat = (int64_t)t->feat_dst.size();
    if ((n_units > 0 && !text) || (n_feat > 0 && !feat_coef) || (n_coef > 0 && !coef)) return fail(LT_ERR_INVALID, "null input pointer");
    for (int64_t i = 0; i < n_feat; ++i) {
        if (feat_coef[i] < -1 || feat_coef[i] >= n_coef)
            return fail(LT_ERR_INVALID, "feat_coef[%lld] = %lld is outside [-1, %lld)", (long long)i, (long long)feat_coef[i], (long long)n_coef);
        if (feat_coef[i] >= 0 && t->feat_func[(size_t)i] != func)
            return fail(LT_ERR_INVALID, "feature %lld belongs to scorer %d, not to the trained scorer %d", (long long)i, t->feat_func[(size_t)i], func);
    }
    ON_DEVICE(t->device);
    lt_trainer* tr = new lt_trainer();
    tr->tables = t;
    tr->device = t->device;
    tr->gold = gold;
    tr->func = func;
    tr->n_sent = n_sent;
    tr->n_coef = n_coef;
    tr->sent_off.assign(sent_off, sent_off + n_sent + 1);
    int rc = upload_once(tr->text, text, (size_t)n_units * 2);
    if (rc == LT_OK) rc = upload_once(tr->off, sent_off, (size_t)(n_sent + 1) * 4);
    if (rc == LT_OK) rc = upload_once(tr->feat_coef, feat_coef, (size_t)n_feat * 8);
    if (rc == LT_OK) rc = upload_once(tr->w, coef, (size_t)n_coef * 8);
    if (rc == LT_OK) rc = zeroed(tr->u, (size_t)n_coef * 8);
    if (rc == LT_OK) rc = zeroed(tr->acc, (size_t)n_coef * 8);
    if (rc == LT_OK) rc = zeroed(tr->differs, (size_t)n_sent);
    if (rc == LT_OK) rc = zeroed(tr->mistakes, 8);
    if (rc == LT_OK) rc = zeroed(tr->prefix_words, (size_t)n_sent * 4);
    if (rc == LT_OK) {
        const std::vector<double> nan((size_t)std::max(1, n_sent), std::numeric_limits<double>::quiet_NaN());
        rc = upload_once(tr->violation, nan.data(), nan.size() * 8);
    }
    if (rc == LT_OK) rc = ensure(tr->gscore, (size_t)std::max<int64_t>(1, gold->n_words) * 8);
    if (rc == LT_OK) {
        tr->gold_off.resize((size_t)n_sent + 1);
        tr->full_last.assign((size_t)n_sent, 1);
        if (cudaMemcpy(tr->gold_off.data(), gold->off.p, tr->gold_off.size() * 8, cudaMemcpyDeviceToHost) != cudaSuccess)
            rc = fail(LT_ERR_CUDA, "reading the gold offsets failed");
    }
    if (rc == LT_OK) rc = upload_feat_dst(t);
    if (rc == LT_OK) rc = scatter_trainer_weights(tr, nullptr);
    if (rc == LT_OK && cudaEventCreate(&tr->done) != cudaSuccess) rc = fail(LT_ERR_CUDA, "cudaEventCreate failed");
    if (rc == LT_OK && cudaDeviceSynchronize() != cudaSuccess) rc = fail(LT_ERR_CUDA, "writing the initial weights failed");
    if (rc != LT_OK) {
        lt_trainer_destroy(tr);
        return rc;
    }
    *out = tr;
    return LT_OK;
}

// Decode the slice on the batch's stream (its text copied device to device into the batch's own buffers, so that
// the batch does not point into the trainer), wait once for the lattice-overflow check, then compare with the gold
// range and apply the update without leaving the device.
extern "C" int lt_trainer_step(lt_trainer* tr, lt_batch* b, int32_t first, int32_t count, int32_t beam_size) {
    if (!tr || !b) return fail(LT_ERR_INVALID, "null argument");
    lt_tables* t = tr->tables;
    if (b->tables != t) return fail(LT_ERR_INVALID, "the batch belongs to other tables");
    if (count < 1 || first < 0 || (int64_t)first + count > tr->n_sent)
        return fail(LT_ERR_INVALID, "sentences [%d, %lld) are not a non-empty range of the %d corpus sentences", first,
                    (long long)first + count, tr->n_sent);
    if (beam_size < 1 || beam_size > LT_MAX_BEAM) return fail(LT_ERR_INVALID, "beam_size must be in 1..%d", LT_MAX_BEAM);
    if (b->cons) return fail(LT_ERR_INVALID, "the batch has constraints bound: a trainer step searches without them");
    ON_DEVICE(t->device);
    cudaStream_t st = b->own_stream;
    const int32_t* off = tr->sent_off.data() + first;
    const int64_t n_units = (int64_t)off[count] - off[0];
    int32_t max_units = 0;
    for (int32_t i = 0; i < count; ++i) max_units = std::max(max_units, off[i + 1] - off[i]);
    if (int rc = ensure(b->text, (size_t)std::max<int64_t>(1, n_units) * 2)) return rc;
    if (int rc = ensure(b->sent_off, (size_t)(count + 1) * 4)) return rc;
    if (n_units) CU(cudaMemcpyAsync(b->text.p, static_cast<const uint16_t*>(tr->text.p) + off[0], (size_t)n_units * 2, cudaMemcpyDeviceToDevice, st));
    LT_LAUNCH(rebase_offsets, (unsigned)std::min<int64_t>(((int64_t)count + 256) / 256, (int64_t)t->sm_count), 256, 0, st,
              static_cast<const int32_t*>(tr->off.p), first, count, static_cast<int32_t*>(b->sent_off.p));
    CU(cudaGetLastError());
    b->launches += 1;
    bind_batch(b, static_cast<const uint16_t*>(b->text.p), static_cast<const int32_t*>(b->sent_off.p), count, n_units, max_units, st);
    if (int rc = launch_lattice(b, st)) return rc;
    b->beam = beam_size;
    b->search_cons = nullptr;
    // (the flag holds through the reruns resolve may launch; later searches of the batch keep the usual trail)
    b->hbm_trail = tr->mode != LT_UPDATE_FULL;
    int rc = launch_beam(b, st, false);
    if (rc == LT_OK) rc = resolve(b);
    b->hbm_trail = false;
    if (rc) return rc;

    PerceptronArgs A{};
    if (int rc = search_and_gold(b, tr->gold, &A.sg)) return rc;
    A.sg.gold_off += first;                       // gold offsets are absolute word indices: the slice's paths start there
    if (int rc = ensure(t->d_counts, n_hits(t) * 8)) return rc;
    CU(cudaMemsetAsync(t->d_counts.p, 0, n_hits(t) * 8, st));
    A.func = tr->func;
    A.counts = static_cast<unsigned long long*>(t->d_counts.p);
    A.differs = static_cast<uint8_t*>(tr->differs.p) + first;
    A.n_differ = static_cast<unsigned long long*>(tr->mistakes.p);
    if (tr->mode == LT_UPDATE_FULL) {
        LT_LAUNCH(perceptron_kernel, warp_grid(t, count), 256, 0, st, t->dev, A);
    } else {
        if (int rc = ensure(tr->chain, (size_t)std::max<int64_t>(1, n_units) * sizeof(lt_edge))) return rc;
        ViolationArgs V{};
        V.pc = A;
        V.mode = tr->mode;
        V.beam = beam_size;
        V.trail = static_cast<const uint64_t*>(b->trail.p);
        V.edges = static_cast<const lt_edge*>(b->edges.p);
        V.gscore = static_cast<double*>(tr->gscore.p);
        V.chain = static_cast<lt_edge*>(tr->chain.p);
        V.prefix_words = static_cast<int32_t*>(tr->prefix_words.p) + first;
        V.violation = static_cast<double*>(tr->violation.p) + first;
        LT_LAUNCH(violation_kernel, warp_grid(t, count), 256, 0, st, t->dev, V);
    }
    CU(cudaGetLastError());
    b->launches += 1;
    std::fill(tr->full_last.begin() + first, tr->full_last.begin() + first + count, tr->mode == LT_UPDATE_FULL ? 1 : 0);

    const int64_t step = ++tr->steps;
    const int64_t n_feat = (int64_t)t->feat_dst.size();
    const int64_t cap = (int64_t)t->sm_count * 16;
    if (n_feat > 0) {
        LT_LAUNCH(gather_coef_counts, (unsigned)std::min<int64_t>((n_feat + 255) / 256, cap), 256, 0, st, A.counts,
                  static_cast<const uint32_t*>(t->d_feat_dst.p), static_cast<const int64_t*>(tr->feat_coef.p), n_feat, feat_slots(t),
                  static_cast<unsigned long long*>(tr->acc.p));
        CU(cudaGetLastError());
        b->launches += 1;
    }
    if (tr->n_coef > 0) {
        LT_LAUNCH(apply_coef_delta, (unsigned)std::min<int64_t>((tr->n_coef + 255) / 256, cap), 256, 0, st,
                  static_cast<unsigned long long*>(tr->acc.p), tr->n_coef, (long long)(step - 1), static_cast<double*>(tr->w.p),
                  static_cast<double*>(tr->u.p));
        CU(cudaGetLastError());
        b->launches += 1;
    }
    if (int rc = scatter_trainer_weights(tr, st)) return rc;
    if (n_feat > 0) b->launches += 1;
    CU(cudaEventRecord(tr->done, st));
    return LT_OK;
}

extern "C" int lt_trainer_fetch(lt_trainer* tr, double* coef, double* averaged, int64_t* steps, int64_t* mistakes, uint8_t* differs) {
    if (!tr) return fail(LT_ERR_INVALID, "null argument");
    ON_DEVICE(tr->tables->device);
    CU(cudaEventSynchronize(tr->done));
    const size_t n = (size_t)tr->n_coef;
    if (coef && n) CU(cudaMemcpy(coef, tr->w.p, n * 8, cudaMemcpyDeviceToHost));
    if (averaged && n) {
        // mean of the weights after steps 1 .. T: (T * w_T - sum_t (t - 1) * delta_t) / T
        std::vector<double> u(n);
        CU(cudaMemcpy(averaged, tr->w.p, n * 8, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(u.data(), tr->u.p, n * 8, cudaMemcpyDeviceToHost));
        if (tr->steps > 0)
            for (size_t c = 0; c < n; ++c) averaged[c] = averaged[c] - u[c] / (double)tr->steps;
    }
    if (steps) *steps = tr->steps;
    if (mistakes) {
        unsigned long long m = 0;
        CU(cudaMemcpy(&m, tr->mistakes.p, 8, cudaMemcpyDeviceToHost));
        *mistakes = (int64_t)m;
    }
    if (differs && tr->n_sent) CU(cudaMemcpy(differs, tr->differs.p, (size_t)tr->n_sent, cudaMemcpyDeviceToHost));
    return LT_OK;
}

extern "C" int lt_trainer_set_update(lt_trainer* tr, int32_t mode) {
    if (!tr) return fail(LT_ERR_INVALID, "null argument");
    if (mode != LT_UPDATE_FULL && mode != LT_UPDATE_EARLY && mode != LT_UPDATE_MAX_VIOLATION)
        return fail(LT_ERR_INVALID, "unknown update mode %d", mode);
    tr->mode = mode;
    return LT_OK;
}

extern "C" int lt_trainer_fetch_update(lt_trainer* tr, int32_t* prefix_words, double* violation) {
    if (!tr) return fail(LT_ERR_INVALID, "null argument");
    ON_DEVICE(tr->tables->device);
    CU(cudaEventSynchronize(tr->done));
    const size_t n = (size_t)tr->n_sent;
    if (n == 0) return LT_OK;
    std::vector<uint8_t> differs(n);
    CU(cudaMemcpy(differs.data(), tr->differs.p, n, cudaMemcpyDeviceToHost));
    if (prefix_words) CU(cudaMemcpy(prefix_words, tr->prefix_words.p, n * 4, cudaMemcpyDeviceToHost));
    if (violation) CU(cudaMemcpy(violation, tr->violation.p, n * 8, cudaMemcpyDeviceToHost));
    // a FULL step updates a differing sentence on its whole gold path
    for (size_t i = 0; i < n; ++i) {
        if (!tr->full_last[i]) continue;
        if (prefix_words) prefix_words[i] = differs[i] ? (int32_t)(tr->gold_off[i + 1] - tr->gold_off[i]) : 0;
        if (violation) violation[i] = std::numeric_limits<double>::quiet_NaN();
    }
    return LT_OK;
}
