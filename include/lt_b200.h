/*
 * lt_b200.h — C ABI of the B200-native lattice-tagger decode path (liblt_b200.so).
 *
 * The reference (lovit/lattice_based_tagger) is pure Python and has no FFI; its boundary for this
 * path is `Tagger.__init__` / `Tagger.tag` (lattice_tagger/tagger/tagger.py:47-78).  The entry
 * points below are what a binding for that boundary calls (INTEGRATION.md shows the ctypes stub):
 *
 *   lt_tables_create   <- Tagger.__init__: dictionary + rules + MorphemeLookup.max_len
 *                         (tagger.py:47-66, dictionary/lookup.py:99-132), the score functions
 *                         (beam/score_funcs.py:18-144) and the trainer's weight format
 *                         (trainer/train.py:34-37), compiled into device-resident tables.
 *   lt_tag_batch_host  <- Tagger.tag for a batch of sentences in HOST memory
 *                         (tagger.py:68-78 = sentence_lookup_as_begin_index + beam_search).
 *   lt_lattice / lt_beam  the same two stages on buffers already resident in HBM
 *                         (dictionary/lookup.py:344-369 ; beam/beam.py:5-61).
 *   lt_pathset_eval    <- the score classes' `evaluate(seq)` hooks (beam/score_funcs.py) and
 *                         SimpleTrigramEncoder.encode_sequence (features/feature.py:62-68) on given paths.
 *   lt_perceptron_delta <- the trainer's epoch (trainer/train.py:61-65): phi(gold) - phi(predicted).
 *   lt_evaluate        <- comparing the tagger's output with an annotated corpus (the trainer's loss,
 *                         word-level matches, and why a wrong sentence is wrong).
 *   lt_trainer_*       <- an online, averaged perceptron in mini-batches: the weights and their running
 *                         average stay on the device between steps.
 *   lt_constraints_*   <- spans the caller already knows to be words (with or without their tag), kept by
 *                         the beam search itself (lt_batch_set_constraints).
 *
 * Plain pointers and sizes only.  No function throws; each returns LT_OK or an LT_ERR_* code and
 * lt_last_error() returns the message of the calling thread's last failure.
 */
#ifndef LT_B200_H
#define LT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LT_ABI_VERSION 8

/* return codes */
#define LT_OK            0
#define LT_ERR_INVALID   1   /* bad argument / malformed table description            */
#define LT_ERR_CUDA      2   /* a CUDA runtime call failed (message has the details)   */
#define LT_ERR_CAPACITY  3   /* caller-provided output buffer too small                */
#define LT_ERR_COLLISION 4   /* two distinct table keys share a 128-bit hash, or a key
                                hashes to the reserved fingerprint 0 (2^-64 per key)    */

/* per-sentence status (the reference's error behaviour, tagger.py:73-78) */
#define LT_SENT_OK        0
#define LT_SENT_NO_EDGES  1  /* non-empty sentence without any dictionary edge: the reference
                                raises IndexError (lookup.py:362-363 + beam.py:33)              */
#define LT_SENT_BAD_SPACE 2  /* whitespace other than U+0020: `str.split()` and
                                `str.replace(' ','')` disagree in the reference; rejected       */
#define LT_SENT_TOO_LONG  3  /* more code units than lt_tables_max_sentence_units(): skipped, the
                                rest of the batch is tagged                                     */
#define LT_SENT_UNSUPPORTED_CHAR 4  /* set by host bindings for text that has no UTF-16 BMP form
                                (the library itself never sees such a sentence)                 */
#define LT_SENT_BAD_CONSTRAINT 5    /* a constrained search (lt_batch_set_constraints): a constraint of the
                                sentence ends beyond its last syllable; no path, the rest of the
                                batch is tagged                                                 */

/* eojeol lookup that builds the lattice (dictionary/lookup.py), lt_batch_set_lookup():
 *   MORPHEME  MorphemeLookup  (lookup.py:99-132, :212-279) — what Tagger.tag always uses (tagger.py:60)
 *   LR        LRLookup(prefer_exact_match=True)   (lookup.py:75-85, :171-210)
 *   LR_ALL    LRLookup(prefer_exact_match=False)
 *   WORD      WordLookup(prefer_exact_match=True) (lookup.py:87-97, :134-169)
 *   WORD_ALL  WordLookup(prefer_exact_match=False)                                             */
#define LT_LOOKUP_MORPHEME 0
#define LT_LOOKUP_LR       1
#define LT_LOOKUP_LR_ALL   2
#define LT_LOOKUP_WORD     3
#define LT_LOOKUP_WORD_ALL 4
#define LT_LOOKUP_EXACT    5  /* MorphemeDictionary.lookup of the whole eojeol alone (dictionary.py:304-312) */

#define LT_WINDOW   8        /* beam_search max_len, beam/beam.py:5                              */
#define LT_MAX_BEAM 64
#define LT_MAX_TAGS 29       /* tag sets are 29-bit masks next to 3 lemmatizer bits */
#define LT_MAX_FUNCS 8
#define LT_NO_TAG   0xFF
#define LT_NO_RULE  0xFFFFFFFFu

/* fixed tag ids (lattice_tagger/tagset.py:1-15); dictionaries may add ids 13..28 */
enum { LT_TAG_NOUN = 0, LT_TAG_PRONOUN, LT_TAG_NUMBER, LT_TAG_JOSA, LT_TAG_ADJECTIVE, LT_TAG_VERB,
       LT_TAG_EOMI, LT_TAG_ADVERB, LT_TAG_DETERMINER, LT_TAG_EXCLAMATION, LT_TAG_BOS, LT_TAG_EOS,
       LT_TAG_UNK };

/* lt_edge.flags */
#define LT_EDGE_IS_L   0x01  /* Word.is_l                                                        */
#define LT_EDGE_UNK    0x02  /* unknown word synthesised by the beam (beam.py:36-38)             */
#define LT_EDGE_LEMMA  0x04  /* two-morpheme word from the lemmatizer (dictionary.py:311-312)    */
#define LT_EDGE_SKIP2  0x08  /* lemma: the eomi continues at word[split+2:] (2/3-syllable keys,
                                lemmatizer.py:109) instead of word[split+1:]                     */

#define LT_EDGE_EXPLICIT 0x10 /* imported lattice (lt_lattice_import): word / morph0 / morph1 are the
                                strings 3*rule, 3*rule+1, 3*rule+2 given with the import           */
#define LT_EDGE_FORCED 0x20  /* forced word of a tagged constraint whose span has no lattice edge of that
                                tag: word = morph0 = chars[b:e], no morph1, tag0 = the constraint's
                                tag, len = e - b (lt_batch_set_constraints)                       */

/* One lattice edge = the reference's `Word` (dictionary/dictionary.py:169) in 16 bytes.
 * word  = chars[b:e]
 * morph0/morph1: single-morpheme edge: morph0 = word, morph1 = None.
 *   lemma edge, rule == LT_NO_RULE (plain split): morph0 = word[:split+1], morph1 = word[split+1:]
 *   lemma edge, rule = r: morph0 = word[:split] + stem_r,
 *                         morph1 = eomi_r + word[split + (SKIP2 ? 2 : 1):]                      */
typedef struct lt_edge {
    uint16_t b, e;       /* syllable span in the space-stripped sentence                        */
    uint16_t len;        /* Word.len — not always e-b (lookup.py:201-202)                       */
    uint8_t  tag0, tag1; /* tag ids; tag1 = LT_NO_TAG for single-morpheme edges                 */
    uint32_t rule;       /* index into the flattened rule list, or LT_NO_RULE                   */
    uint16_t split;      /* lemma edges: syllables of the surface before the conjugation point  */
    uint8_t  flags;
    uint8_t  reserved;
} lt_edge;

/* Score program: the BeamScoreFunctions list in evaluation order (score_funcs.py:50-54). */
#define LT_FUNC_REG     1    /* RegularizationScore: p0=unknown_penalty p1=known_preference p2=syllable_penalty */
#define LT_FUNC_MPREF   2    /* MorphemePreferenceScore                                          */
#define LT_FUNC_WPREF   3    /* WordPreferenceScore                                              */
#define LT_FUNC_TRIGRAM 4    /* SimpleTrigramFeatureScore                                        */
typedef struct lt_func {
    int32_t kind;
    int32_t reserved;
    double  p[3];
} lt_func;

/* Table description handed to lt_tables_create.  Strings are UTF-16 code units (every character
 * of the reference's resources is in the BMP); `*_off` arrays have one more entry than strings. */
typedef struct lt_tables_desc {
    int32_t abi_version;            /* LT_ABI_VERSION */
    int32_t n_tags;                 /* ids in use, <= LT_MAX_TAGS */

    /* dictionary: distinct strings with the tag sets they belong to (dictionary.py:227-242) */
    int64_t         n_dict;
    const uint16_t* dict_chars;
    const int64_t*  dict_off;       /* n_dict + 1 */
    const uint32_t* dict_tagmask;   /* bit t: string in tag_to_morphs[tag t]                    */
    const uint8_t*  dict_lemma;     /* bit0 in .verbs, bit1 in .adjectives, bit2 in .eomis
                                       (captured separately, dictionary.py:300-302)             */
    int32_t         n_tag_order;    /* dictionary iteration order of the tags (get_tags)        */
    const uint8_t*  tag_order;
    int32_t         max_len;        /* MorphemeLookup.max_len (lookup.py:123-132)               */
    int32_t         reserved0;

    /* conjugation rules (dictionary.py:365-378); keys of 1..3 syllables, rules in tuple order */
    int64_t         n_rule_keys;
    const uint16_t* rule_key_chars; /* 3 code units per key, zero padded                        */
    const uint8_t*  rule_key_len;
    const uint8_t*  rule_k3_first;  /* 3-syllable key iterates before its 2-syllable prefix
                                       in {word[i:i+2], word[i:i+3]} (lemmatizer.py:107)        */
    const int64_t*  rule_first;     /* n_rule_keys + 1: rules of key i = [first[i], first[i+1]) */
    int64_t         n_rules;
    const uint16_t* rule_chars;     /* stems and eomis, concatenated                            */
    const int64_t*  rule_stem_off;  /* n_rules + 1 entries: stem i = [stem_off[i], eomi_off[i])    */
    const int64_t*  rule_eomi_off;  /* n_rules entries:     eomi i = [eomi_off[i], stem_off[i+1])  */

    /* score program */
    int32_t         n_funcs;
    int32_t         reserved1;
    const lt_func*  funcs;

    /* feature / preference strings (distinct) */
    int64_t         n_fstr;
    const uint16_t* fstr_chars;
    const int64_t*  fstr_off;       /* n_fstr + 1 */

    /* trigram features (features/feature.py:94-121) of the LT_FUNC_TRIGRAM entries.
     * template: 0..8; s0,s1,s2 string ids (-1 unused); a0,a1 integers (tag ids, len, is_l):
     *  0 (s0=wj.word, s1=wk.word, a0=tk)   1 (s0=wj.word, a0=tk)   2 (a0=tj, s0=wk.word, a1=tk)
     *  3 (a0=tj, a1=tk)   4 (a0=len)   5 (s0=wk.word, a0=tk, a1=is_l)   6 (a0=len)
     *  7 (s0=wi.word, s1=wj.word, s2=wk.word)   8 (s0=w?.morph0, s1=wk.morph0)                 */
    int64_t         n_feat;
    const uint8_t*  feat_func;      /* index into funcs[] of the owning scorer                  */
    const uint8_t*  feat_template;
    const int32_t*  feat_s;         /* 3 per feature */
    const int32_t*  feat_a;         /* 2 per feature */
    const double*   feat_weight;

    /* preference entries of the LT_FUNC_MPREF / LT_FUNC_WPREF scorers: (tag, string) -> value */
    int64_t         n_pref;
    const uint8_t*  pref_func;
    const uint8_t*  pref_tag;
    const int32_t*  pref_s;
    const double*   pref_value;
} lt_tables_desc;

/* Work counters of one batch (SURVEY.md §8d); they define the algorithmic byte counts. */
typedef struct lt_counters {
    uint64_t sentences;
    uint64_t L;    /* syllables                                                                */
    uint64_t P;    /* dictionary string probes the reference semantics require                 */
    uint64_t E;    /* dictionary edges                                                          */
    uint64_t T;    /* scored transitions                                                        */
    uint64_t F;    /* feature tuples generated                                                  */
    uint64_t Bk;   /* kept beam entries                                                         */
    uint64_t W;    /* words on the returned paths                                               */
} lt_counters;

/* Device-time of the last batch, measured with CUDA events on the batch's stream. */
typedef struct lt_timings {
    float ms_h2d, ms_lattice, ms_reserved0, ms_reserved1, ms_beam, ms_pack, ms_d2h, ms_total;
} lt_timings;

/* State of a batch workspace: sticky buffer capacities, how often a batch had to be rerun with
 * larger buffers, kernels launched so far, launch shapes of the last batch. */
typedef struct lt_info {
    int64_t launches;            /* kernels launched by this workspace so far (cumulative)            */
    int64_t edge_cap;            /* lattice edge buffer capacity (records)                             */
    int64_t n_edges;             /* dictionary edges of the last batch                                 */
    int32_t reruns;              /* grow-and-rerun rounds so far (cumulative)                          */
    int32_t hcap, retry_hcap;    /* lattice staging capacity per warp: main pass, retry pass (0 = off) */
    int32_t retried;             /* sentences of the last batch that went through the retry pass       */
    int32_t unit_limit;          /* = lt_tables_max_sentence_units()                                   */
    int32_t lattice_warps, lattice_ctas_per_sm, lattice_smem;
    int32_t beam_warps, beam_ctas_per_sm, beam_smem, beam_trail_smem;
    int32_t sm_count;
    int32_t reserved[3];
} lt_info;

typedef struct lt_tables lt_tables;   /* immutable device tables; shareable between batches */
typedef struct lt_batch  lt_batch;    /* device workspace + stream state of one in-flight batch */

const char* lt_last_error(void);
int  lt_abi_version(void);

int  lt_tables_create(const lt_tables_desc* desc, int device, lt_tables** out);
void lt_tables_destroy(lt_tables* tables);
/* bytes of device memory held by the tables */
int64_t lt_tables_device_bytes(const lt_tables* tables);
/* Longest sentence (UTF-16 code units, spaces included) the kernels can hold with these tables; it
 * shrinks with the longest dictionary string (at most 4088).  Longer sentences of a batch get
 * LT_SENT_TOO_LONG, the others are tagged. */
int32_t lt_tables_max_sentence_units(const lt_tables* tables);

/* New coefficients for the SAME features the tables were created with (desc->feat_* order): the trainer's
 * epoch (trainer/train.py:44-65 changes `coefficients`, never the feature dictionary).  Weights are written
 * in place on the device; nothing is re-hashed.  No batch may be in flight on these tables. */
int  lt_tables_update_weights(lt_tables* tables, const double* weights, int64_t n_weights);

int  lt_batch_create(lt_tables* tables, lt_batch** out);
void lt_batch_destroy(lt_batch* batch);
/* which eojeol lookup the following lt_lattice* calls enumerate (LT_LOOKUP_*, default MORPHEME) */
int  lt_batch_set_lookup(lt_batch* batch, int32_t mode);

/* Tagger.tag over a batch in HOST memory: copies `text` / `sent_off` to the device, builds the
 * lattices, runs the beam search, copies the best paths back.
 *   text      UTF-16 code units of all sentences, spaces (U+0020) included
 *   sent_off  n_sent + 1 offsets into text
 *   path_off  out, n_sent + 1: words of sentence s are path_edges[path_off[s] : path_off[s+1]]
 *             (BOS / EOS not included)
 *   path_edges out, capacity path_cap records (sent_off[n_sent] always suffices)
 *   scores    out, n_sent fp64 path scores;  status out, n_sent LT_SENT_* codes               */
int  lt_tag_batch_host(lt_batch* batch, const uint16_t* text, const int32_t* sent_off,
                       int32_t n_sent, int32_t beam_size,
                       int32_t* path_off, lt_edge* path_edges, int64_t path_cap,
                       double* scores, int32_t* status);

/* The two stages on DEVICE-resident inputs, asynchronous on `stream` (a cudaStream_t).
 * lt_lattice builds the CSR lattice into the batch workspace; lt_beam consumes it.            */
int  lt_lattice(lt_batch* batch, const uint16_t* d_text, const int32_t* d_sent_off,
                int32_t n_sent, int64_t n_units, int32_t max_sent_units, void* stream);
int  lt_beam(lt_batch* batch, int32_t beam_size, void* stream);
/* Both stages in one call (= lt_lattice then lt_beam): Tagger.tag for N sentences already in HBM
 * (tagger.py:68-78), results fetched with lt_paths_fetch.                                     */
int  lt_tag_batch_device(lt_batch* batch, const uint16_t* d_text, const int32_t* d_sent_off,
                         int32_t n_sent, int64_t n_units, int32_t max_sent_units, int32_t beam_size,
                         void* stream);

/* sentence_lookup_as_begin_index (dictionary/lookup.py:344-369) over a batch in HOST memory:
 * copies `text` / `sent_off` to the device and builds the lattices; fetch with lt_lattice_fetch. */
int  lt_lattice_host(lt_batch* batch, const uint16_t* text, const int32_t* sent_off, int32_t n_sent);

/* A lattice built by the CALLER (beam_search's `bindex` argument, beam/beam.py:5): sentences in host
 * memory plus their edges in the layout lt_lattice_fetch returns — sorted by (sentence, end, begin,
 * order within the span), end_off[sent_off[s] + e - 1 .. + e] bracketing the edges of sentence s that end
 * at syllable e.  Edges flagged LT_EDGE_EXPLICIT name their strings instead of deriving them from the
 * text: edge.rule = i, and strings 3i, 3i+1, 3i+2 of (str_chars, str_off) are its word, morph0 and
 * morph1 (empty when there is none).  lt_beam / lt_beam_kbest then search it.                    */
int  lt_lattice_import(lt_batch* batch, const uint16_t* text, const int32_t* sent_off, int32_t n_sent,
                       const lt_edge* edges, const int64_t* end_off,
                       const uint16_t* str_chars, const int64_t* str_off, int64_t n_strings);

/* beam_search keeping ALL survivors of the last position (its return value, beam/beam.py:59-61),
 * not only matures[0]: lt_beam_kbest instead of lt_beam, results with lt_kbest_fetch (the best path
 * stays available through lt_paths_fetch as well).  lt_tag_batch_host_kbest = text from host memory
 * + lt_lattice + lt_beam_kbest. */
int  lt_beam_kbest(lt_batch* batch, int32_t beam_size, void* stream);
int  lt_tag_batch_host_kbest(lt_batch* batch, const uint16_t* text, const int32_t* sent_off,
                             int32_t n_sent, int32_t beam_size);
int  lt_kbest_size(lt_batch* batch, int64_t* n_words);
/* n_best[s] survivors of sentence s (<= beam, 0 when status[s] != LT_SENT_OK), best first in the
 * reference's order; survivor r of sentence s is path_edges[path_off[s*beam+r] : path_off[s*beam+r+1]]
 * with score scores[s*beam+r]; path_off has n_sent*beam + 1 entries, scores n_sent*beam.          */
int  lt_kbest_fetch(lt_batch* batch, int32_t* n_best, int32_t* path_off, lt_edge* path_edges,
                    int64_t path_cap, double* scores, int32_t* status);

/* Results of the last lt_lattice / lt_beam on this batch (these synchronise the stream). */
int  lt_lattice_size(lt_batch* batch, int64_t* n_edges);
/* edges sorted by (sentence, e, b, reference order); end_off[sent_off[s] + e - 1 .. + e] bracket
 * the edges of sentence s that end at syllable e (end_off has n_units + 1 entries)            */
int  lt_lattice_fetch(lt_batch* batch, lt_edge* edges, int64_t edge_cap, int64_t* end_off);
int  lt_paths_size(lt_batch* batch, int64_t* n_words);
int  lt_paths_fetch(lt_batch* batch, int32_t* path_off, lt_edge* path_edges, int64_t path_cap,
                    double* scores, int32_t* status);

/* per-sentence status / syllable count of the last lattice (either pointer may be NULL) */
int  lt_lattice_status(lt_batch* batch, int32_t* status, int32_t* sent_len);

int  lt_batch_info(lt_batch* batch, lt_info* out);
int  lt_batch_counters(lt_batch* batch, lt_counters* out);
int  lt_batch_timings(lt_batch* batch, lt_timings* out);
/* Per-stage CUDA events on / off for the batches to come (the first lt_batch_timings call switches them on).
 * They are recorded on the batch's stream between its kernels, which run one after the other either way.       */
int  lt_batch_set_stage_timing(lt_batch* batch, int32_t on);

/* Word paths given by the caller (a gold analysis, candidates from elsewhere), device-resident, tied to one
 * lt_tables.  Path p is edges[path_off[p] .. path_off[p+1]), in order, BOS / EOS left out (path_off has
 * n_paths + 1 entries, path_off[0] = 0).  Every edge is LT_EDGE_EXPLICIT: its strings 3*rule, 3*rule+1,
 * 3*rule+2 of (str_chars, str_off) are word, morph0 and morph1 (empty when there is none), as in
 * lt_lattice_import; they are hashed once, here.  Spans, Word.len and tags need not be anything the search
 * could produce (tag ids below n_tags). */
typedef struct lt_pathset lt_pathset;
int  lt_pathset_create(lt_tables* tables, int32_t n_paths, const lt_edge* edges, const int64_t* path_off,
                       const uint16_t* str_chars, const int64_t* str_off, int64_t n_strings, lt_pathset** out);
void lt_pathset_destroy(lt_pathset* paths);

/* scores[p] = the score of path p under the tables' score program, bit for bit what the beam computes for
 * the path (BeamScoreFunctions over every transition, Sequence.add in word order; EOS adds nothing).
 * With feat_off != NULL also the features of trigram scorer `func` that fire (SimpleTrigramEncoder.
 * encode_sequence): word w (index over all words of the set) has feat_idx[feat_off[w] .. feat_off[w+1])
 * (feat_off: n_words + 1 entries), indices in lt_tables_desc feature order, by template.  9 * n_words
 * always suffices for feat_cap.  `func` is read only with feat_off.  Runs on the batch's stream; synchronous. */
int  lt_pathset_eval(lt_batch* batch, const lt_pathset* paths, int32_t func, double* scores,
                     int64_t* feat_off, int32_t* feat_idx, int64_t feat_cap);

/* One perceptron step against the best paths of the batch's last lt_tag_batch_host / lt_beam, with gold path
 * s for sentence s (gold->n_paths = the batch's sentences).  Sentence s differs when its status is not
 * LT_SENT_OK or its best path is not gold path s word for word on (b, e, morph0, morph1, tag0, tag1);
 * Word.len and is_l are not compared.  For every sentence that differs: delta += phi(gold) - phi(best), the
 * second term only when the status is LT_SENT_OK; phi = counts of trigram scorer func's features.
 *   delta     out, n_delta = lt_tables_desc.n_feat counts in desc order (exact integers)
 *   differs   out, one flag per sentence;  n_differ  out, sentences that differ
 * The count buffer belongs to the tables: no other lt_perceptron_delta on the same tables may run meanwhile. */
int  lt_perceptron_delta(lt_batch* batch, const lt_pathset* gold, int32_t func, int64_t* delta, int64_t n_delta,
                         uint8_t* differs, int64_t* n_differ);

/* lt_evaluate: the class of a sentence */
#define LT_EVAL_CORRECT      0  /* status LT_SENT_OK and the best path is the gold path (the negation of
                                   lt_perceptron_delta's `differs`)                                  */
#define LT_EVAL_FAILED       1  /* status is not LT_SENT_OK                                          */
#define LT_EVAL_UNREACHABLE  2  /* the gold path is not in the search space of beam_search          */
#define LT_EVAL_SEARCH_ERROR 3  /* reachable, and its image scores higher than the path found        */
#define LT_EVAL_MODEL_ERROR  4  /* reachable, and its image scores at most the found path's score    */

/* lt_evaluate: why a gold word is outside the search space (the first check it fails, in this order) */
#define LT_GOLD_OK             0
#define LT_GOLD_BREAKS_TILING  1  /* does not begin where the previous word ends (0 for the first word),
                                     ends beyond the sentence, or is the last word and does not end at
                                     its last syllable                                                   */
#define LT_GOLD_BEYOND_WINDOW  2  /* e - b > LT_WINDOW                                                   */
#define LT_GOLD_NOT_IN_LATTICE 3  /* no lattice edge of its (b, e) equals it on b, e, tag0, tag1, morph0,
                                     morph1; where the lattice has no edge of that span at all, it is not
                                     the beam's unknown word (tag0 Unk, no tag1, morph0 = the span's
                                     syllables, no morph1)                                               */
#define LT_GOLD_UNK_AFTER_UNK  4  /* tag0 Unk right after a tag0-Unk word, and b != max(0, e - LT_WINDOW)
                                     (beam/beam.py:44-45)                                               */
#define LT_GOLD_UNCHECKED   0xFF  /* the sentence's status is not LT_SENT_OK                              */

/* lt_evaluate: counts[LT_EVAL_N_COUNTS * s + i] */
#define LT_EVAL_GOLD_WORDS 0
#define LT_EVAL_PRED_WORDS 1      /* 0 unless the status is LT_SENT_OK                                  */
#define LT_EVAL_SEG        2      /* predicted words equal to a gold word on b, e                        */
#define LT_EVAL_TAG        3      /* ... on b, e, tag0, tag1                                             */
#define LT_EVAL_FULL       4      /* ... on b, e, tag0, tag1, morph0, morph1                              */
#define LT_EVAL_GOLD_UNITS 5      /* (morph0, tag0) per word, plus (morph1, tag1) when tag1 is set        */
#define LT_EVAL_PRED_UNITS 6
#define LT_EVAL_UNIT_MATCH 7      /* units of words equal on b, e whose morpheme and tag are equal        */
#define LT_EVAL_N_COUNTS   8

/* The best paths of the batch's last search (lt_tag_batch_host, lt_tag_batch_device, lt_beam, lt_beam_kbest,
 * also over an imported lattice) against gold path s for sentence s (gold->n_paths = the batch's sentences;
 * every gold path has b < e and strictly increasing b).  Per sentence:
 *   sent_class   LT_EVAL_* (required)
 *   counts       LT_EVAL_N_COUNTS int32 (LT_EVAL_GOLD_WORDS ...), or NULL
 *   gold_scores  the score of the gold path's image, NaN unless the gold path is reachable, or NULL
 *   word_reason  per gold word (gold->n_words) LT_GOLD_*, or NULL
 * A gold path is reachable when the status is LT_SENT_OK, every word passes the LT_GOLD_* checks, and the path
 * is not empty unless the sentence is.  Its image takes for each word the first equal lattice edge of its end
 * position's bucket (or the beam's unknown-word record), and its score is bit for bit lt_pathset_eval of the
 * image, the search's own score when the image is the path the search found.  Runs on the batch's stream;
 * synchronous. */
int  lt_evaluate(lt_batch* batch, const lt_pathset* gold, uint8_t* sent_class, int32_t* counts,
                 double* gold_scores, uint8_t* word_reason);

/* Mini-batch perceptron training on the device.  The trainer keeps the weights in coefficient space, w[n_coef]
 * (indexed like the encoder's feature_dic, which need not be one-to-one), and u[n_coef] for the average.  Step
 * t = 1, 2, ... decodes sentences [first, first + count) of the corpus with the current tables, takes delta as
 * lt_perceptron_delta does (per sentence that differs: phi(gold) - phi(best), only phi(gold) when the status is
 * not LT_SENT_OK; desc feature f of `func` adds to coefficient feat_coef[f]), then
 *     w += delta,   u += (t - 1) * delta,
 * and writes w[feat_coef[f]] into the tables for every feature f of `func` with feat_coef[f] >= 0 (hashed slots
 * and dense blocks).  A step without a mistake still counts.  The averaged weights after T steps are
 * w - u / T, the mean of the weights after steps 1 .. T.  Counts are exact integers, so w and u are the same
 * whatever the order of the atomic adds.
 *
 * lt_trainer_create  corpus `text` / `sent_off` (n_sent + 1 offsets, sent_off[0] = 0, non-decreasing) in host
 *                    memory, uploaded once; `gold` one path per corpus sentence (gold->n_paths == n_sent), on the
 *                    same tables, and it must outlive the trainer; `func` a trigram scorer;
 *                    feat_coef[desc->n_feat] the coefficient of each desc feature of `func` (-1: not trained, its
 *                    weight stays), -1 for every feature of another scorer; coef[n_coef] = w_0, written into the
 *                    tables here (synchronous, no batch may be in flight on the tables).
 * lt_trainer_step    one step on `batch` (same tables): the slice is copied and searched on the batch's own stream
 *                    (one host wait, for the lattice-overflow check), then compared and applied there without a
 *                    copy to or from the host.  Afterwards the batch holds the slice as its last search:
 *                    lt_paths_fetch, lt_evaluate etc. work on it, also after lt_trainer_destroy.  The step writes
 *                    the tables and the tables' count buffer: no other search, lt_perceptron_delta or trainer step
 *                    on the same tables may run meanwhile, and lt_tables_update_weights afterwards rewrites every
 *                    weight, dense blocks included.
 * lt_trainer_fetch   waits for the last step; any pointer may be NULL.  coef / averaged: n_coef doubles
 *                    (averaged = w while no step has run); steps; mistakes: sentences that differed, summed over
 *                    all steps; differs[n_sent]: per corpus sentence, from the last step that covered it (0 before). */
typedef struct lt_trainer lt_trainer;
int  lt_trainer_create(lt_tables* tables, int32_t func, const uint16_t* text, const int32_t* sent_off, int32_t n_sent,
                       const lt_pathset* gold, int64_t n_coef, const int64_t* feat_coef, const double* coef,
                       lt_trainer** out);
int  lt_trainer_step(lt_trainer* trainer, lt_batch* batch, int32_t first, int32_t count, int32_t beam_size);
int  lt_trainer_fetch(lt_trainer* trainer, double* coef, double* averaged, int64_t* steps, int64_t* mistakes,
                      uint8_t* differs);
void lt_trainer_destroy(lt_trainer* trainer);

/* The update a trainer step makes for a sentence that differs and has status LT_SENT_OK (every other sentence is
 * updated as above in every mode; which sentences differ, the mistakes and the w / u bookkeeping do not change).
 * Let gold words 1..W end at e_1 < ... < e_W = L (e_0 = 0), R_m the ranks the search kept at end position e_m whose
 * hypothesis equals gold words 1..m on (b, e, tags, morphemes) (R_0 = {0}), B_m the score of rank 0 at e_m and G_m
 * the score of gold words 1..m as lt_pathset_eval sums it.  The update is phi(gold words 1..m*) - phi(the rank-0
 * hypothesis at e_{m*}) with
 *   LT_UPDATE_FULL           m* = W: phi(gold) - phi(best path), the default
 *   LT_UPDATE_EARLY          m* = the first m with R_m empty, else W (Collins and Roark 2004)
 *   LT_UPDATE_MAX_VIOLATION  m* = the m with 0 not in R_m that maximises B_m - G_m, ties to the larger m
 *                            (Huang, Fayong and Guo 2012)
 * A gold path that does not tile [0, L) with non-empty words (lt_evaluate: LT_GOLD_BREAKS_TILING) gets m* = W.
 * EARLY and MAX_VIOLATION steps keep the search's back-pointers in HBM and read them there.
 *
 * lt_trainer_set_update    the mode of the steps that follow; LT_ERR_INVALID for an unknown mode.
 * lt_trainer_fetch_update  waits for the last step; per corpus sentence, from the last step that covered it (either
 *                          pointer may be NULL): prefix_words[n_sent] = m* (0 when the sentence did not differ or was
 *                          never covered, W for a full update, also when the status is not LT_SENT_OK);
 *                          violation[n_sent] = B_{m*} - G_{m*}, NaN where there was no update, a FULL step, or the
 *                          tiling fallback. */
#define LT_UPDATE_FULL          0
#define LT_UPDATE_EARLY         1
#define LT_UPDATE_MAX_VIOLATION 2
int  lt_trainer_set_update(lt_trainer* trainer, int32_t mode);
int  lt_trainer_fetch_update(lt_trainer* trainer, int32_t* prefix_words, double* violation);

/* Constrained search: spans the caller already knows to be words.  A constraint of a sentence is (b, e, tag): b, e
 * syllable offsets in the space-stripped sentence (the coordinates of lt_edge.b / .e), 1 <= e - b <= LT_WINDOW, and
 * tag a tag id below n_tags other than BOS, EOS and Unk, or LT_NO_TAG for "any word".  A sentence's constraints are
 * sorted by b and do not overlap (c[i].e <= c[i+1].b); they may cross eojeol boundaries.  The search is beam_search
 * with three changes to the candidates of end e and begin b (DESIGN.md, "Constrained search"):
 *   1. (b, e) is blocked when a constraint c overlaps it without being equal to it (b < c.e, c.b < e, (b, e) != (c.b,
 *      c.e)): no lattice edge and no unknown word.  Positions strictly inside a constrained span keep no hypothesis.
 *   2. (b, e) == (c.b, c.e): the span's lattice edges with tag0 == c.tag (all of them for LT_NO_TAG), in lattice
 *      order.  If there is none: with LT_NO_TAG the usual unknown word; with a tag, one LT_EDGE_FORCED word, is_l set
 *      when b is the first syllable of an eojeol.
 *   3. An unknown word may follow an unknown word only from the first begin the constraints leave open: the smallest
 *      b in [max(0, e - LT_WINDOW), e) for which (b, e) is not blocked (without constraints: beam.py:44-45).
 * Every sentence with status LT_SENT_OK then has a path, and it has a word on each constrained span with its tag.
 *
 * lt_constraints_create   constraint set of n_sent sentences: sentence s has cons[cons_off[s] .. cons_off[s+1]),
 *                         cons_off has n_sent + 1 entries starting at 0.  LT_ERR_INVALID, naming the sentence and the
 *                         index, for offsets that are not monotone, constraints that are unsorted or overlap, a span
 *                         outside 1..LT_WINDOW syllables or a tag the search cannot give a word.  A constraint ending
 *                         beyond its sentence is found by the search: LT_SENT_BAD_CONSTRAINT.
 * lt_batch_set_constraints binds the set (NULL: none) for the searches that follow on the batch: lt_beam,
 *                         lt_beam_kbest, lt_tag_batch_host, lt_tag_batch_host_kbest, lt_tag_batch_device, imported
 *                         lattices included.  The set must outlive its binding and the fetch of those searches'
 *                         results.  A search of a batch whose n_sent differs from the set's returns LT_ERR_INVALID
 *                         before any launch.  The statuses lt_paths_fetch / lt_kbest_fetch return are the search's
 *                         (with LT_SENT_BAD_CONSTRAINT); lt_lattice_status keeps the lattice's.
 * lt_evaluate and lt_perceptron_delta after a constrained search, and lt_trainer_step on a batch with constraints
 * bound, return LT_ERR_INVALID: their results are defined on the unconstrained search space. */
typedef struct lt_constraint {
    uint16_t b, e;
    uint8_t  tag;        /* tag id, or LT_NO_TAG */
    uint8_t  reserved[3];
} lt_constraint;
typedef struct lt_constraints lt_constraints;
int  lt_constraints_create(lt_tables* tables, int32_t n_sent, const lt_constraint* cons, const int64_t* cons_off,
                           lt_constraints** out);
void lt_constraints_destroy(lt_constraints* cons);
int  lt_batch_set_constraints(lt_batch* batch, const lt_constraints* cons);

#ifdef __cplusplus
}
#endif
#endif /* LT_B200_H */
