"""Host compile step: dictionary + rules + score functions -> device tables.

This is where `Tagger.__init__` of the reference (`tagger/tagger.py:47-66`) does its set-up: it
keeps the dictionary, builds `MorphemeLookup` (which derives `max_len`,
`dictionary/lookup.py:110-113,123-132`) and stores the score functions.  Here the same inputs are
flattened into the plain arrays of `lt_tables_desc` (include/lt_b200.h) and handed to
`lt_tables_create`, which hashes them into the GPU-resident tables.

Three facts of the reference depend on the running process and are therefore read from the live
objects, never re-derived (SURVEY App. A Q1-Q3): the iteration order of `tag_to_morphs`, the
order of each rule tuple, and the iteration order of the two-element set
`{word[i:i+2], word[i:i+3]}` for every pair of rule keys where it can matter.
"""

import ctypes

import numpy as np

from . import _native
from .tagset import Adjective, Adverb, Determiner, Exclamation, Noun, Number, Verb
from .tagset import BUILTIN_TAGS, MAX_TAGS

DEFAULT_STANDALONES = (Noun, Adverb, Exclamation, Determiner, Number)   # dictionary/lookup.py:104-105
OTHER_TAG = '\x00other'         # device id for tags of an imported lattice that the tables have never seen


class UnsupportedScoreFunction(ValueError):
    pass


def _encode_units(strings):
    """Concatenate strings into UTF-16 code units; returns (uint16 array, int64 offsets).

    Every string must consist of BMP characters (one code unit per Python character) — true for
    all of the reference's resources (SURVEY App. B).
    """
    lengths = np.fromiter((len(s) for s in strings), dtype=np.int64, count=len(strings))
    offsets = np.zeros(len(strings) + 1, dtype=np.int64)
    np.cumsum(lengths, out=offsets[1:])
    raw = ''.join(strings).encode('utf-16-le', 'surrogatepass')
    units = np.frombuffer(raw, dtype='<u2')
    if units.size != int(offsets[-1]):
        bad = next(s for s in strings if len(s.encode('utf-16-le', 'surrogatepass')) != 2 * len(s))
        raise ValueError('characters outside the Basic Multilingual Plane are not supported: %r' % bad)
    if units.size == 0:
        units = np.zeros(1, dtype='<u2')
    return np.ascontiguousarray(units), offsets


def _is_bmp(s):
    return all(ord(c) < 0x10000 for c in s)


class _StringTable:
    def __init__(self):
        self.ids = {}
        self.strings = []

    def add(self, s):
        idx = self.ids.get(s)
        if idx is None:
            idx = len(self.strings)
            self.ids[s] = idx
            self.strings.append(s)
        return idx


def _as_index(x):
    """Python-equality normalisation of a numeric feature component: True == 1 == 1.0."""
    if isinstance(x, (bool, int, np.integer)):
        return int(x)
    if isinstance(x, (float, np.floating)) and float(x).is_integer():
        return int(x)
    return None


class CompiledTables:
    """Owns the `lt_tables` handle plus the host-side lists needed to turn packed results back
    into `Word`s (tag names, flattened rules)."""

    def __init__(self, dictionary, score_funcs, device=0, k3_first=None, extra_tags=()):
        if not hasattr(dictionary, 'rules'):
            raise ValueError('dictionary must be MorphemeDictionary')         # lookup.py:101-102
        self._lib = _native.load()
        self._keep = []
        self.device = device
        self.handle = None

        tag_to_morphs = dictionary.tag_to_morphs
        self.tag_names = list(BUILTIN_TAGS)
        tag_ids = {t: i for i, t in enumerate(self.tag_names)}
        # (`extra_tags`: tags of caller-built lattices — beam_search's `bindex` — that no dictionary lists;
        # OTHER_TAG stands for any further tag: no feature or preference can name it)
        for tag in list(tag_to_morphs) + list(extra_tags):
            if tag not in tag_ids:
                tag_ids[tag] = len(self.tag_names)
                self.tag_names.append(tag)
        self.other_tag_id = tag_ids.get(OTHER_TAG)
        if len(self.tag_names) > MAX_TAGS:
            raise ValueError('at most %d distinct tags are supported, dictionary has %d'
                             % (MAX_TAGS, len(self.tag_names)))
        self.tag_ids = tag_ids

        desc = _native.lt_tables_desc()
        desc.abi_version = _native.LT_ABI_VERSION
        desc.n_tags = len(self.tag_names)
        self._pack_dictionary(desc, dictionary)
        self._pack_rules(desc, dictionary.rules, k3_first)
        self._pack_scores(desc, score_funcs)

        handle = ctypes.c_void_p()
        _native.check(self._lib.lt_tables_create(ctypes.byref(desc), int(device), ctypes.byref(handle)))
        self.handle = handle
        self._keep = []          # the library copied everything it needs

    # -- dictionary ------------------------------------------------------------------------------
    def _pack_dictionary(self, desc, dictionary):
        tag_to_morphs = dictionary.tag_to_morphs
        index = {}
        masks = []
        strings = []

        def slot(s):
            i = index.get(s)
            if i is None:
                i = len(strings)
                index[s] = i
                strings.append(s)
                masks.append([0, 0])
            return i

        for tag, morphs in tag_to_morphs.items():
            bit = 1 << self.tag_ids[tag]
            for m in morphs:
                masks[slot(m)][0] |= bit
        # the lemmatizer reads these three attributes, not tag_to_morphs (dictionary.py:300-302)
        for bit, attr in ((1, 'verbs'), (2, 'adjectives'), (4, 'eomis')):
            for m in getattr(dictionary, attr, ()) or ():
                masks[slot(m)][1] |= bit

        # MorphemeLookup._find_max_len (lookup.py:123-132); max() of an empty set raises ValueError
        wanted = set(DEFAULT_STANDALONES) | {Verb, Adjective}
        max_len = 0
        for tag, morphs in tag_to_morphs.items():
            if tag in wanted:
                max_len = max(max_len, max(len(m) for m in morphs))
        self.max_len = max_len

        units, offsets = _encode_units(strings)
        mask_arr = np.asarray(masks, dtype=np.int64).reshape(-1, 2)
        tagmask = np.ascontiguousarray(mask_arr[:, 0].astype(np.uint32))
        lemma = np.ascontiguousarray(mask_arr[:, 1].astype(np.uint8))
        order = np.asarray([self.tag_ids[t] for t in tag_to_morphs], dtype=np.uint8)
        if order.size == 0:
            order = np.zeros(1, dtype=np.uint8)
        self._keep += [units, offsets, tagmask, lemma, order]
        desc.n_dict = len(strings)
        desc.dict_chars = _native.ptr(units)
        desc.dict_off = _native.ptr(offsets)
        desc.dict_tagmask = _native.ptr(tagmask if tagmask.size else np.zeros(1, np.uint32))
        desc.dict_lemma = _native.ptr(lemma if lemma.size else np.zeros(1, np.uint8))
        desc.n_tag_order = len(tag_to_morphs)
        desc.tag_order = _native.ptr(order)
        desc.max_len = int(max_len)
        self.n_dict = len(strings)

    # -- rules -----------------------------------------------------------------------------------
    def _pack_rules(self, desc, rules, k3_first):
        keys = [k for k in rules if isinstance(k, str) and 1 <= len(k) <= 3 and _is_bmp(k)]
        key_chars = np.zeros((max(1, len(keys)), 3), dtype='<u2')
        key_len = np.zeros(max(1, len(keys)), dtype=np.uint8)
        k3_flags = np.zeros(max(1, len(keys)), dtype=np.uint8)
        first = np.zeros(len(keys) + 1, dtype=np.int64)
        flat = []
        pieces = []
        for i, key in enumerate(keys):
            key_chars[i, :len(key)] = [ord(c) for c in key]
            key_len[i] = len(key)
            if len(key) == 3 and key[:2] in rules:
                if k3_first is not None and key in k3_first:
                    k3_flags[i] = 1 if k3_first[key] else 0
                else:
                    # observe the set order exactly as lemmatizer.py:107 builds it
                    k2 = key[:2]
                    k3_flags[i] = 1 if next(iter({k2, key})) == key else 0
            for stem, eomi in rules[key]:
                flat.append((stem, eomi))
                pieces.append(stem)
                pieces.append(eomi)
            first[i + 1] = len(flat)
        units, offsets = _encode_units(pieces)
        stem_off = np.ascontiguousarray(offsets[0::2])              # n_rules + 1 entries
        eomi_off = np.ascontiguousarray(offsets[1::2]) if flat else np.zeros(1, dtype=np.int64)
        self.rules_flat = flat
        self._keep += [key_chars, key_len, k3_flags, first, units, stem_off, eomi_off]
        desc.n_rule_keys = len(keys)
        desc.rule_key_chars = _native.ptr(key_chars)
        desc.rule_key_len = _native.ptr(key_len)
        desc.rule_k3_first = _native.ptr(k3_flags)
        desc.rule_first = _native.ptr(first)
        desc.n_rules = len(flat)
        desc.rule_chars = _native.ptr(units)
        desc.rule_stem_off = _native.ptr(stem_off)
        desc.rule_eomi_off = _native.ptr(eomi_off)

    # -- score program -----------------------------------------------------------------------------
    def _pack_scores(self, desc, score_funcs):
        funcs = list(getattr(score_funcs, 'funcs', None) or [])
        if not funcs and score_funcs is not None and not hasattr(score_funcs, 'funcs'):
            raise UnsupportedScoreFunction('score_funcs must be a BeamScoreFunctions')
        if len(funcs) > _native.LT_MAX_FUNCS:
            raise UnsupportedScoreFunction('at most %d score functions are supported' % _native.LT_MAX_FUNCS)
        prog = (_native.lt_func * max(1, len(funcs)))()
        self._weight_source = []
        self._desc_sources = None
        self._funcs = funcs
        strings = _StringTable()
        feat_func, feat_tmpl, feat_s, feat_a, feat_w = [], [], [], [], []
        pref_func, pref_tag, pref_s, pref_v = [], [], [], []
        tag_ids = self.tag_ids
        self.n_features = 0

        for f, func in enumerate(funcs):
            kind = type(func).__name__
            if kind == 'RegularizationScore':
                prog[f].kind = _native.LT_FUNC_REG
                prog[f].p[0] = float(func.unknown_penalty)
                prog[f].p[1] = float(func.known_preference)
                prog[f].p[2] = float(func.syllable_penalty)
            elif kind in ('MorphemePreferenceScore', 'WordPreferenceScore'):
                is_m = kind == 'MorphemePreferenceScore'
                prog[f].kind = _native.LT_FUNC_MPREF if is_m else _native.LT_FUNC_WPREF
                table = func.tag_to_morph if is_m else func.tag_to_word
                for tag, entries in table.items():
                    if tag not in tag_ids:
                        continue                      # no word can carry this tag
                    for s, value in entries.items():
                        if not isinstance(s, str) or not _is_bmp(s):
                            continue
                        pref_func.append(f)
                        pref_tag.append(tag_ids[tag])
                        pref_s.append(strings.add(s))
                        pref_v.append(float(value))
            elif kind == 'SimpleTrigramFeatureScore':
                prog[f].kind = _native.LT_FUNC_TRIGRAM
                if func.encoder is None:
                    raise UnsupportedScoreFunction('SimpleTrigramFeatureScore needs an encoder')
                if type(func.encoder).__name__ != 'SimpleTrigramEncoder':
                    raise UnsupportedScoreFunction(
                        'only SimpleTrigramEncoder features have a device implementation, got %s'
                        % type(func.encoder).__name__)
                feature_dic = func.encoder.feature_dic
                coef = func.coefficients
                if isinstance(coef, np.ndarray) and coef.dtype.kind == 'f' and coef.dtype != np.float64:
                    raise UnsupportedScoreFunction(
                        'coefficients must be float64 (numpy sums %s differently)' % coef.dtype)
                coef = np.asarray(coef, dtype=np.float64)
                if len(coef) != len(feature_dic):
                    raise ValueError('Encoder and coefficients have different size features')
                self.n_features += len(feature_dic)
                self._pack_feature_dic(f, feature_dic, coef, strings, feat_func, feat_tmpl, feat_s, feat_a, feat_w)
            else:
                raise UnsupportedScoreFunction(
                    'score function %s has no device implementation (supported: RegularizationScore, '
                    'MorphemePreferenceScore, WordPreferenceScore, SimpleTrigramFeatureScore); '
                    'there is no CPU fallback' % kind)

        units, offsets = _encode_units(strings.strings)

        def joined(parts, dtype, width=None):
            if not parts:
                return np.zeros((0, width) if width else 0, dtype=dtype)
            return np.concatenate(parts).astype(dtype, copy=False)
        a_func = joined(feat_func, np.uint8)
        a_tmpl = joined(feat_tmpl, np.uint8)
        a_s = joined(feat_s, np.int32, 3).reshape(-1, 3)
        a_a = joined(feat_a, np.int32, 2).reshape(-1, 2)
        a_w = joined(feat_w, np.float64)
        n_feat = int(a_func.size)
        p_func = np.asarray(pref_func, dtype=np.uint8)
        p_tag = np.asarray(pref_tag, dtype=np.uint8)
        p_s = np.asarray(pref_s, dtype=np.int32)
        p_v = np.asarray(pref_v, dtype=np.float64)
        arrays = [units, offsets, a_func, a_tmpl, a_s, a_a, a_w, p_func, p_tag, p_s, p_v]
        arrays = [np.ascontiguousarray(a) if a.size else np.zeros(4, dtype=a.dtype) for a in arrays]
        units, offsets, a_func, a_tmpl, a_s, a_a, a_w, p_func, p_tag, p_s, p_v = arrays
        if len(strings.strings) == 0:
            offsets = np.zeros(1, dtype=np.int64)
        self._keep += arrays + [prog, offsets]
        desc.n_funcs = len(funcs)
        desc.funcs = ctypes.cast(prog, ctypes.c_void_p)
        desc.n_fstr = len(strings.strings)
        desc.fstr_chars = _native.ptr(units)
        desc.fstr_off = _native.ptr(offsets)
        desc.n_feat = n_feat
        self.n_desc = n_feat
        desc.feat_func = _native.ptr(a_func)
        desc.feat_template = _native.ptr(a_tmpl)
        desc.feat_s = _native.ptr(a_s)
        desc.feat_a = _native.ptr(a_a)
        desc.feat_weight = _native.ptr(a_w)
        desc.n_pref = len(pref_func)
        desc.pref_func = _native.ptr(p_func)
        desc.pref_tag = _native.ptr(p_tag)
        desc.pref_s = _native.ptr(p_s)
        desc.pref_value = _native.ptr(p_v)

    # (template, tuple length) -> kinds of the components after the template id:
    #   's' string (word / morpheme), 't' tag name, 'n' small integer, 'l' is_l flag
    _TEMPLATES = {(0, 4): 'sst', (1, 3): 'st', (2, 4): 'tst', (3, 3): 'tt', (4, 2): 'n', (5, 4): 'stl',
                  (6, 2): 'n', (7, 4): 'sss', (8, 3): 'ss'}
    # where each component goes in (feat_s[0..2], feat_a[0..1]) — include/lt_b200.h, lt_tables_desc
    _SLOTS = {0: ('s0', 's1', 'a0'), 1: ('s0', 'a0'), 2: ('a0', 's0', 'a1'), 3: ('a0', 'a1'), 4: ('a0',),
              5: ('s0', 'a0', 'a1'), 6: ('a0',), 7: ('s0', 's1', 's2'), 8: ('s0', 's1')}

    def _pack_feature_dic(self, f, feature_dic, coef, strings, feat_func, feat_tmpl, feat_s, feat_a, feat_w):
        """Feature tuples (features/feature.py:94-121) -> (template, string ids, integers).

        A key that cannot equal any tuple the templates generate (wrong arity or types, a tag no
        word can carry) is dropped: `_filter` (feature.py:28-29) would never select it either.
        Works column-wise per template, so that a 10 M-entry dictionary packs in seconds: the keys
        of one template are transposed once and each component column is mapped as a whole.
        """
        tag_ids = self.tag_ids
        groups = {}
        for key, idx in feature_dic.items():
            if type(key) is not tuple or not key:
                continue
            tmpl = key[0]
            if type(tmpl) is not int:
                tmpl = _as_index(tmpl)
            slot = (tmpl, len(key))
            group = groups.get(slot)
            if group is None:
                if slot not in self._TEMPLATES:
                    continue
                group = groups[slot] = ([], [])
            group[0].append(key)
            group[1].append(idx)

        def string_ids(column):
            ids = strings.ids
            out = np.empty(len(column), dtype=np.int64)
            for pos, x in enumerate(column):
                i = ids.get(x)
                if i is None:
                    i = strings.add(x) if type(x) is str and _is_bmp(x) else -1
                out[pos] = i
            return out

        for (tmpl, _), (keys, idxs) in groups.items():
            kinds = self._TEMPLATES[(tmpl, len(keys[0]))]
            columns = list(zip(*keys))[1:]
            n = len(keys)
            cols = {'s0': np.full(n, -1, np.int64), 's1': np.full(n, -1, np.int64), 's2': np.full(n, -1, np.int64),
                    'a0': np.zeros(n, np.int64), 'a1': np.zeros(n, np.int64)}
            ok = np.ones(n, dtype=bool)
            for kind, where, column in zip(kinds, self._SLOTS[tmpl], columns):
                if kind == 's':
                    vals = string_ids(column)
                    ok &= vals >= 0
                elif kind == 't':
                    vals = np.fromiter((tag_ids.get(x, -1) if type(x) is str else -1 for x in column), dtype=np.int64, count=n)
                    ok &= vals >= 0
                else:
                    vals = np.fromiter((-1 if v is None else v for v in map(_as_index, column)), dtype=np.int64, count=n)
                    ok &= (vals >= 0) & (vals < (1 << 24))
                    if kind == 'l':
                        ok &= vals <= 1
                cols[where] = vals
            keep = np.nonzero(ok)[0]
            source = np.asarray(idxs, dtype=np.int64)[keep]
            self._weight_source.append((f, source))          # where each packed weight comes from (update_weights)
            weights = np.asarray(coef, dtype=np.float64)[source]
            feat_func.append(np.full(len(keep), f, dtype=np.uint8))
            feat_tmpl.append(np.full(len(keep), tmpl, dtype=np.uint8))
            feat_s.append(np.stack([cols['s0'][keep], cols['s1'][keep], cols['s2'][keep]], axis=1).astype(np.int32))
            feat_a.append(np.stack([np.where(ok, cols['a0'], 0)[keep], np.where(ok, cols['a1'], 0)[keep]], axis=1).astype(np.int32))
            feat_w.append(weights)

    def desc_sources(self):
        """Per feature of `lt_tables_desc` (the order of device feature indices and of a perceptron delta):
        (index of its scorer in the score program, its `feature_dic` index)."""
        if self._desc_sources is None:
            funcs = [np.full(len(source), f, dtype=np.int64) for f, source in self._weight_source]
            if funcs:
                self._desc_sources = (np.concatenate(funcs), np.concatenate([source for _, source in self._weight_source]))
            else:
                self._desc_sources = (np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64))
        return self._desc_sources

    def update_weights(self):
        """Write the scorers' CURRENT `coefficients` into the device tables in place (same features, new
        weights — the trainer's epoch).  Nothing is re-hashed: `lt_tables_update_weights`."""
        parts = []
        for f, source in self._weight_source:
            coef = np.asarray(self._funcs[f].coefficients, dtype=np.float64)
            if len(coef) != len(self._funcs[f].encoder.feature_dic):
                raise ValueError('Encoder and coefficients have different size features')
            parts.append(coef[source])
        weights = np.ascontiguousarray(np.concatenate(parts)) if parts else np.zeros(0, dtype=np.float64)
        _native.check(self._lib.lt_tables_update_weights(self.handle, _native.ptr(weights) if weights.size else None, int(weights.size)))

    def device_bytes(self):
        return int(self._lib.lt_tables_device_bytes(self.handle))

    def close(self):
        if self.handle is not None and self._lib is not None:
            self._lib.lt_tables_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
