// violation.cuh — early and max-violation perceptron updates (Collins and Roark 2004; Huang, Fayong and Guo 2012)
// read from the back-pointers of the step's search (lt_trainer_set_update).
//
// The step's beam kernel keeps its trail in HBM: entry (e, r) = (edge reference, span, parent rank) of rank r at end
// position e, every rank the search kept (beam.cuh).  Ranks it did not fill hold the host's 0xFF memset: span byte
// 0xFF > LT_WINDOW.  For a sentence that differs, has status LT_SENT_OK and whose gold words 1..W tile [0, L) with
// ends e_1 < ... < e_W = L:
//   R_m  the ranks at e_m whose hypothesis equals gold words 1..m on (b, e, tags, morphemes); R_0 = {0} (BOS).
//        Rank r is in R_m when its entry is filled, spans e_m - e_{m-1}, has its parent in R_{m-1} and its edge
//        equals gold word m by content (a lattice may hold equal edges: either copy counts).
//   G_m  gold words 1..m scored as lt_pathset_eval scores them; B_m the rank-0 hypothesis at e_m, followed back
//        through the trail and rescored the same way — bit for bit the score the search gave it.
//   m*   EARLY: the first m with R_m empty, else W.  MAX_VIOLATION: argmax of B_m - G_m over the m with 0 not in
//        R_m, ties to the larger m.
// The update is phi(gold words 1..m*) - phi(rank-0 hypothesis at e_{m*}); a trigram feature of a word depends only
// on the words before it, so the prefix's features are its share of the whole path's.  Every other sentence is
// updated as perceptron_kernel updates it.
#pragma once
#include "evaluate.cuh"

namespace lt {

struct ViolationArgs {
    PerceptronArgs pc;
    int32_t mode;               // LT_UPDATE_EARLY or LT_UPDATE_MAX_VIOLATION
    int32_t beam;
    const uint64_t* trail;      // [(n_units) * beam] the search's HBM back-pointers
    const lt_edge* edges;       // the batch's lattice
    double* gscore;             // scratch: G_m at gold word m - 1 [gold n_words]
    lt_edge* chain;             // scratch: a rank-0 hypothesis, last word first, at the sentence's offset [n_units]
    int32_t* prefix_words;      // [n_sent] m*: 0 when the sentence did not differ, W for a full update
    double* violation;          // [n_sent] B_{m*} - G_{m*}, NaN without an update or for a full fallback
};

__device__ __forceinline__ bool same_word(const EdgeView& k, const EdgeView& g) {
    return k.b == g.b && k.e == g.e && k.tag0 == g.tag0 && k.tag1 == g.tag1 && h2_same(k.mk, g.mk) && h2_same(k.m1, g.m1);
}

// Sequence.add over n words in order (path_eval_kernel's sum); prefix[w], when given, gets the sum up to word w.
template <class Load>
__device__ __forceinline__ double sum_words(const DevTables& T, int n, int lane, Load load, double* prefix) {
    double s = 0.0;
    walk_words(T, n, lane, load, [&](int w, bool valid, const EdgeView& k, const PathCtx& c) {
        uint32_t hit[9];
        const double inc = valid ? path_increment(T, k, c, -1, hit) : 0.0;
        const int m = min(32, n - (w - lane));
        double mine = 0.0;
        for (int l = 0; l < m; ++l) {
            s = __dadd_rn(__dadd_rn(s, __shfl_sync(kFull, inc, l)), 0.0);
            if (l == lane) mine = s;
        }
        if (prefix && valid) prefix[w] = mine;
    });
    return s;
}

// delta per hit of scorer `func` over n words (perceptron_kernel's counting)
template <class Load>
__device__ __forceinline__ void count_words(const DevTables& T, int n, int lane, int func, Load load, unsigned long long* counts,
                                            unsigned long long delta) {
    walk_words(T, n, lane, load, [&](int, bool valid, const EdgeView& k, const PathCtx& c) {
        if (!valid) return;
        uint32_t hit[9];
        path_hits(T, k, c, func, hit);
        #pragma unroll
        for (int i = 0; i < 9; ++i)
            if (hit[i] != kNoHit) atomicAdd(counts + hit[i], delta);
    });
}

// The rank-0 hypothesis at end position e as lattice records (unknown words as the beam's path walk makes them),
// last word first, into chain[0 .. n); -> n.  Lane 0 follows the back-pointers.
__device__ __forceinline__ int rank0_chain(const ViolationArgs& A, int s0, int e, int lane, lt_edge* chain) {
    int n = 0;
    if (lane == 0) {
        int r = 0;
        while (e > 0) {
            const uint64_t t = A.trail[(size_t)(s0 + e - 1) * A.beam + r];
            const uint32_t eref = (uint32_t)t, span = (uint32_t)((t >> 32) & 0xFFu);
            // Rank 0 is filled at every end position 1..L (an unknown word from the window's first begin is always a
            // candidate), so this only stops a walk on a corrupt trail instead of looping.
            if (span == 0u || span > (uint32_t)LT_WINDOW) break;
            chain[n++] = eref == kTrailUnk ? unknown_record(e - (int)span, e) : A.edges[eref];
            r = (int)((t >> 40) & 0xFFu);
            e -= (int)span;
        }
    }
    __syncwarp();
    return __shfl_sync(kFull, n, 0);
}

__global__ void __launch_bounds__(256) violation_kernel(const __grid_constant__ DevTables T, const __grid_constant__ ViolationArgs A) {
    const int lane = threadIdx.x & 31;
    const int warps = (int)(gridDim.x * blockDim.x) >> 5;
    const SearchAndGold& sg = A.pc.sg;
    const double nan = __longlong_as_double(0x7FF8000000000000ll);
    for (int s = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); s < sg.n_sent; s += warps) {
        const bool ok = sg.status[s] == LT_SENT_OK;
        const int64_t go = sg.gold_off[s];
        const int W = (int)(sg.gold_off[s + 1] - go);
        const lt_edge* gold = sg.gold_edges + go;
        const int s0 = sg.sent_off[s], s1 = sg.sent_off[s + 1];
        const lt_edge* pred = sg.path_edges + sg.path_off[s];
        const int P = ok ? (int)(sg.path_off[s + 1] - sg.path_off[s]) : 0;
        uint16_t* ch = sg.ch + s0;
        uint64_t* ha = sg.ha + s0 + s;
        uint64_t* hb = sg.hb + s0 + s;
        const int L = ok ? stage_sentence_hashes(sg.text, s0, s1, lane, ch, ha, hb) : 0;
        const SentView pv{ch, ha, hb, nullptr, sg.imp};
        const SentView gv{nullptr, nullptr, nullptr, nullptr, sg.gold_hashes};
        auto load_gold = [&](int w, EdgeView& k) {
            unpack_edge(ldg16(gold + w), k);
            edge_hashes_inline<1>(T, gv, k, true);
        };
        lt_edge* chain = A.chain + s0;
        int n_chain = 0;
        auto load_chain = [&](int w, EdgeView& k) {
            unpack_edge(*reinterpret_cast<const uint4*>(chain + (n_chain - 1 - w)), k);
            edge_hashes_inline<1>(T, pv, k, true);
        };

        // does the prediction differ: exactly perceptron_kernel's test
        bool differ = !ok || P != W;
        for (int base = 0; base < P && !differ; base += 32) {
            const int w = base + lane;
            bool mismatch = false;
            if (w < P) {
                EdgeView k, g;
                unpack_edge(ldg16(pred + w), k);
                edge_hashes_inline<1>(T, pv, k, true);
                load_gold(w, g);
                mismatch = !same_word(k, g);
            }
            differ = __ballot_sync(kFull, mismatch) != 0u;
        }

        // does the gold path tile [0, L) with non-empty words (else: the full update)
        bool tiles = differ && ok && W > 0;
        int prev_e = 0;
        for (int base = 0; base < W && tiles; base += 32) {
            const int w = base + lane;
            const uint32_t x = w < W ? ldg16(gold + w).x : 0u;
            const int b = (int)(x & 0xFFFFu), e = (int)(x >> 16);
            int pe = __shfl_up_sync(kFull, e, 1);
            if (lane == 0) pe = prev_e;
            tiles = __ballot_sync(kFull, w < W && (b != pe || e <= b || e > L || (w == W - 1 && e != L))) == 0u;
            prev_e = __shfl_sync(kFull, e, 31);
        }

        int mstar = differ ? W : 0;
        double vio = nan;
        if (tiles) {
            sum_words(T, W, lane, load_gold, A.gscore + go);
            __syncwarp();
            uint64_t R = 1ull;                  // R_0 = {BOS}
            int e_prev = 0;
            double best = 0.0;
            mstar = 0;
            for (int m = 1; m <= W; ++m) {
                EdgeView g;
                load_gold(m - 1, g);
                if (R != 0ull) {
                    uint64_t next = 0ull;
                    for (int r0 = 0; r0 < A.beam; r0 += 32) {
                        const int r = r0 + lane;
                        bool in = false;
                        if (r < A.beam) {
                            const uint64_t t = A.trail[(size_t)(s0 + g.e - 1) * A.beam + r];
                            const uint32_t eref = (uint32_t)t, span = (uint32_t)((t >> 32) & 0xFFu), parent = (uint32_t)((t >> 40) & 0xFFu);
                            // (the span test rejects before the edge load; same_word's b comparison implies it)
                            if (span <= (uint32_t)LT_WINDOW && span == (uint32_t)(g.e - e_prev) && parent < 64u && ((R >> parent) & 1ull)) {
                                EdgeView k;
                                if (eref == kTrailUnk) unknown_edge(g.e - (int)span, g.e, k);
                                else unpack_edge(ldg16(A.edges + eref), k);
                                edge_hashes_inline<1>(T, pv, k, true);
                                in = same_word(k, g);
                            }
                        }
                        next |= (uint64_t)__ballot_sync(kFull, in) << r0;
                    }
                    R = next;
                }
                e_prev = g.e;
                if (A.mode == LT_UPDATE_EARLY) {
                    if (R == 0ull || m == W) {
                        mstar = m;
                        break;
                    }
                } else if (!(R & 1ull)) {
                    n_chain = rank0_chain(A, s0, g.e, lane, chain);
                    const double v = __dadd_rn(sum_words(T, n_chain, lane, load_chain, nullptr), -A.gscore[go + m - 1]);
                    if (mstar == 0 || v >= best) {
                        best = v;
                        mstar = m;
                    }
                    __syncwarp();               // the chain is rebuilt for the next m
                }
            }
            // 0 is in R_W only when the best path is the gold path, which does not differ: m* = 0 cannot happen here.
            // Should it, the update is the full one and, as for every full update, no violation is reported.
            const bool none = mstar == 0;
            if (none) mstar = W;
            const int e_star = (int)(ldg16(gold + mstar - 1).x >> 16);
            n_chain = rank0_chain(A, s0, e_star, lane, chain);
            if (!none)
                vio = A.mode == LT_UPDATE_EARLY ? __dadd_rn(sum_words(T, n_chain, lane, load_chain, nullptr), -A.gscore[go + mstar - 1]) : best;
            count_words(T, mstar, lane, A.pc.func, load_gold, A.pc.counts, 1ull);
            count_words(T, n_chain, lane, A.pc.func, load_chain, A.pc.counts, ~0ull);      // -1
        } else if (differ) {
            count_words(T, W, lane, A.pc.func, load_gold, A.pc.counts, 1ull);
            if (ok) count_words(T, P, lane, A.pc.func, [&](int w, EdgeView& k) {
                unpack_edge(ldg16(pred + w), k);
                edge_hashes_inline<1>(T, pv, k, true);
            }, A.pc.counts, ~0ull);
        }
        if (lane == 0) {
            A.pc.differs[s] = differ ? 1 : 0;
            if (differ) atomicAdd(A.pc.n_differ, 1ull);
            A.prefix_words[s] = mstar;
            A.violation[s] = vio;
        }
        __syncwarp();
    }
}

}  // namespace lt
