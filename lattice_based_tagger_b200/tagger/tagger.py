"""`Tagger` — the drop-in boundary of the decode path.

Same constructor and `tag()` signature as the reference (`tagger/tagger.py:47-48,68`); `tag()`
returns a `Sequence` whose `.sequences` is the word list BOS .. EOS, `.score` the path score and
`.num_unk` the trailing-unknown count.  Added for the GPU: `tag_batch()` (many sentences per
call — the unit the kernels are built for), `tag_batch_kbest()` (every beam survivor, the
return value of the reference's `beam_search`), `lattice_batch()` (the lattice alone, i.e.
`sentence_lookup_as_begin_index`, `dictionary/lookup.py:344-369`), `score_paths()` / `encode_paths()`
(given paths) and `evaluate()` (the output against gold analyses).

All work happens in `liblt_b200.so`: the sentences go to the device as raw UTF-16 text, the
lattice and beam kernels run there, and packed 16-byte word records come back.  Nothing is
computed on the host besides packing strings and rebuilding `Word` tuples; without the library
or a CUDA device the constructor raises.
"""

from .. import _native
from ..dictionary import BaseMorphemeDictionary, Word
from ..dictionary.lookup import EojeolLookup, MorphemeLookup, begin_index
from ..engine import Engine, PackedSequences, pack_sentences  # noqa: F401  (pack_sentences is part of this module's surface)
from ..tagset import BOS, EOS


def _inner_words(paths):
    """`Sequence`s or [BOS, ..., EOS] word lists -> the words between BOS and EOS of each."""
    from ..beam.beam import Sequence
    out = []
    for path in paths:
        words = path.sequences if isinstance(path, Sequence) else path
        if not isinstance(words, (list, tuple)) or len(words) < 2:
            raise ValueError('a path is a Sequence or a [BOS, ..., EOS] word list, got %r' % (path,))
        words = [w if isinstance(w, Word) else Word._make(w) if isinstance(w, tuple) and len(w) == len(Word._fields) else None
                 for w in words]
        if any(w is None for w in words) or words[0].tag0 != BOS or words[-1].tag0 != EOS:
            raise ValueError('a path is a Sequence or a [BOS, ..., EOS] word list, got %r' % (path,))
        out.append(words[1:-1])
    return out


def _trigram_func(score_funcs, scorer=None):
    """(index in the score program, scorer) of `scorer`, by default the first SimpleTrigramFeatureScore."""
    from ..beam import SimpleTrigramFeatureScore
    funcs = list(getattr(score_funcs, 'funcs', None) or [])
    for f, func in enumerate(funcs):
        if (func is scorer) if scorer is not None else isinstance(func, SimpleTrigramFeatureScore):
            if not isinstance(func, SimpleTrigramFeatureScore):
                raise ValueError('%r is not a SimpleTrigramFeatureScore' % (func,))
            return f, func
    if scorer is None:
        raise ValueError('the tagger has no SimpleTrigramFeatureScore')
    raise ValueError('the scorer is not one of the tagger\'s score functions')


class Tagger:
    """
    >>> funcs = BeamScoreFunctions(RegularizationScore(unknown_penalty=-.1, known_preference=0.5))
    >>> tagger = Tagger(DemoMorphemeDictionary(), score_funcs=funcs)
    >>> tagger.tag('너무너무너무는 아이오아이의 노래 입니다').score
    15.5

    `lookup`: the reference accepts the argument and then always builds `MorphemeLookup`
    (`tagger.py:57-62`); any string does the same here.  An `EojeolLookup` object — `LRLookup`,
    `WordLookup`, `MorphemeLookup`, with their `prefer_exact_match` / `flatten` options — selects
    that enumeration on the device instead (the options the argument was meant for).
    """

    def __init__(self, dictionary='base', lookup='subword_lookup', encoder=None, score_funcs=None,
                 device=0, k3_first=None, extra_tags=()):
        if isinstance(dictionary, str):
            dictionary = BaseMorphemeDictionary()
        self.dictionary = dictionary
        self.score_funcs = score_funcs
        self.device = device
        self._k3_first = k3_first
        self._lookup_arg = lookup
        # tags no dictionary word carries that given paths may name (`score_paths`, the trainer's gold paths)
        self._extra_tags = tuple(extra_tags)
        self._engine = None
        self.eojeol_lookup = None
        self.refresh()

    # -- device state ------------------------------------------------------------------------------
    def refresh(self):
        """(Re)compile the device tables — call after mutating the dictionary or the weights."""
        self.close()
        self._engine = Engine(self.dictionary, self.score_funcs, self.device, self._k3_first, extra_tags=self._extra_tags)
        if isinstance(self._lookup_arg, EojeolLookup):
            self.eojeol_lookup = self._lookup_arg
        else:
            self.eojeol_lookup = MorphemeLookup(self.dictionary, device=self.device)
        # the lookup object shares this tagger's tables (its own would be a second copy of the dictionary)
        self.eojeol_lookup._attach(self._engine, self._engine.tables.max_len)
        self._engine.set_lookup(self.eojeol_lookup.mode)

    def update_weights(self):
        """After changing the `coefficients` of the tagger's trigram scorers (same `feature_dic`): write them
        to the device tables in place — much cheaper than `refresh()`, which recompiles everything."""
        self._engine.tables.update_weights()

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # handles the C-ABI level tools (bench.py, tests) use directly
    @property
    def _lib(self):
        return self._engine._lib

    @property
    def _batch(self):
        return self._engine.batch

    @property
    def _tables(self):
        return self._engine.tables

    # -- the reference's API ---------------------------------------------------------------------------
    def tag(self, sent, beam_size=5, ensure_normalize=True, debug=False, constraints=None):
        """`constraints`: this sentence's list for `tag_batch`'s `constraints=`."""
        if debug:
            if constraints is not None:
                raise ValueError('tag(debug=True) does not support constraints')
            self.trace(sent, beam_size)
        return self.tag_batch([sent], beam_size=beam_size, constraints=None if constraints is None else [constraints])[0]

    # -- batched API -----------------------------------------------------------------------------------
    def tag_batch(self, sents, beam_size=5, errors='raise', lazy=True, constraints=None):
        """Tag many sentences in one device pass; returns one `Sequence` per sentence.

        A sentence the reference cannot tag — no dictionary edge at all, `IndexError` there
        (`lookup.py:362-363` + `beam.py:33`) — raises the same here, or yields `None` with
        `errors='none'`; so do the inputs this implementation rejects per sentence (whitespace
        other than U+0020, characters outside the BMP, sentences beyond the device limit:
        `ValueError`).  The result is a `PackedSequences`: a list whose `Sequence` / `Word` objects
        are built when an item is read (`lazy=False`: a plain list, all built at once).

        `constraints`: one list per sentence (`None` or `[]`: none) of `(b, e)` or `(b, e, tag_name)` spans,
        syllable offsets in the space-stripped sentence, sorted and not overlapping, at most 8 syllables each.  The
        search keeps each span as one word — a lattice word of that tag, or of any tag for `(b, e)`; where the
        lattice has none, an unknown word for `(b, e)` and the word `Word(surface, surface, None, tag, None, e - b,
        b, e, is_l)` for a tag — and no word crosses a span's boundary (DESIGN.md, "Constrained search").  A
        malformed list raises `ValueError` before anything runs.
        """
        if self.score_funcs is None:
            raise TypeError("'NoneType' object is not callable")      # what beam.py:47 raises
        sents = list(sents)
        if self.eojeol_lookup.flatten:
            if constraints is not None:
                raise ValueError('constraints are not supported with a flatten=True lookup')
            best = [None if s is None else s[0] for s in self._kbest_flattened(sents, beam_size, errors)]
            return best
        packed = self._engine.tag_packed(sents, beam_size, constraints)
        if errors == 'raise':
            status = packed[3]
            if status.any():
                bad = int(status.nonzero()[0][0])
                self._engine._raise_for(int(status[bad]), bad)
        if not lazy:
            return self._engine.unpack(sents, packed, errors)
        return PackedSequences(self._engine, sents, packed, errors)

    def tag_batch_packed(self, sents, beam_size=5, constraints=None):
        """The C-ABI call alone: returns (path_off, path_edges, scores, status) numpy arrays."""
        if constraints is not None and self.eojeol_lookup.flatten:
            raise ValueError('constraints are not supported with a flatten=True lookup')
        return self._engine.tag_packed(list(sents), beam_size, constraints)

    def tag_batch_kbest(self, sents, beam_size=5, errors='raise', constraints=None):
        """Every survivor of the beam per sentence, best first — what the reference's `beam_search`
        returns (`beam/beam.py:59-61`); `tag_batch(...)[i]` is `tag_batch_kbest(...)[i][0]`."""
        if self.score_funcs is None:
            raise TypeError("'NoneType' object is not callable")
        sents = list(sents)
        if self.eojeol_lookup.flatten:
            if constraints is not None:
                raise ValueError('constraints are not supported with a flatten=True lookup')
            return self._kbest_flattened(sents, beam_size, errors)
        packed = self._engine.kbest_packed(sents, beam_size, constraints=constraints)
        return self._engine.unpack_kbest(sents, packed, beam_size, errors)

    def _kbest_flattened(self, sents, beam_size, errors):
        # flatten=True (flatten_words, dictionary.py:114-167): the device builds the lattice, the two-morpheme
        # words are split on the host, and the flattened lattice goes back as an imported one
        lattices = self.eojeol_lookup.lookup_batch(sents, errors=errors)
        usable = [(i, s, lat) for i, (s, lat) in enumerate(zip(sents, lattices)) if lat is not None]
        packed = self._engine.kbest_packed([s for _, s, _ in usable], beam_size, imported=[lat for _, _, lat in usable])
        got = self._engine.unpack_kbest([s for _, s, _ in usable], packed, beam_size, errors, self._engine._imported_words)
        out = [None] * len(sents)
        for (i, _, _), seqs in zip(usable, got):
            out[i] = seqs
        return out

    def trace(self, sent, beam_size=5):
        """`tag(debug=True)`: prints the hypotheses kept at every end position, best first.  (The
        reference prints every grown hypothesis before the beam is cut, `beam/beam.py:53-57`; the
        device keeps only the survivors, so those are what can be shown.)  The beam at end position
        e depends on nothing to its right, so it is the search result of the e-syllable prefix of
        the sentence's lattice — one k-best pass over all prefixes."""
        words = self.eojeol_lookup.lookup_batch([sent])[0]
        chars = sent.replace(' ', '')
        prefixes, lattices = [], []
        for e in range(1, len(chars) + 1):
            prefixes.append(chars[:e])
            lattices.append([w for w in words if w.e <= e])
        if not prefixes:
            return
        packed = self._engine.kbest_packed(prefixes, beam_size, imported=lattices)
        kept = self._engine.unpack_kbest(prefixes, packed, beam_size, 'none', self._engine._imported_words)
        for e, seqs in enumerate(kept, 1):
            print('\n{}\nEnd point = {}, len(kept) = {}\n'.format('-' * 40, e, len(seqs or ())))
            for seq in seqs or ():
                seq.sequences = seq.sequences[:-1]        # the hypotheses of an inner position carry no EOS
                seq.num_unk = 0
                for w in reversed(seq.sequences):
                    if w.tag0 != 'Unknown':
                        break
                    seq.num_unk += 1
                print(seq, end='\n\n')

    # -- given paths ---------------------------------------------------------------------------------
    def score_paths(self, paths):
        """The score the model gives each path (float64 array): what the score classes' `evaluate(seq)`
        computes in the reference, on the device, bit for bit the arithmetic of the search.  A path is a
        `Sequence` or a [BOS, ..., EOS] word list; it need not be one the search could find."""
        if self.score_funcs is None:
            raise TypeError("'NoneType' object is not callable")
        pathset = self._engine.upload_paths(_inner_words(paths))
        try:
            return self._engine.eval_paths(pathset)[0]
        finally:
            pathset.close()

    def encode_paths(self, paths, scorer=None):
        """Per path the list `scorer.encoder.encode_sequence(words)` returns (feature-dictionary indices of
        the trigram features that fire, word by word, template order), computed on the device.  `scorer`:
        one of the tagger's `SimpleTrigramFeatureScore`s, by default the first."""
        func, scorer = _trigram_func(self.score_funcs, scorer)
        words = _inner_words(paths)
        pathset = self._engine.upload_paths(words)
        try:
            _, feat_off, feat_idx = self._engine.eval_paths(pathset, func)
        finally:
            pathset.close()
        desc_func, desc_fdic = self._engine.tables.desc_sources()
        fdic = desc_fdic[feat_idx].tolist()
        offs = feat_off.tolist()
        out, w = [], 0
        for path in words:
            out.append([fdic[offs[i]:offs[i + 1]] for i in range(w, w + len(path))])
            w += len(path)
        return out

    def evaluate(self, sents, golds, beam_size=5):
        """Tag `sents` and compare each best path with its gold path (`golds[i]`: a `Sequence` or a [BOS, ...,
        EOS] word list, as for `score_paths`), all on the device: one decode, one upload of the gold paths, one
        `lt_evaluate`.  Returns an `Evaluation`: per-sentence classes (correct, failed, unreachable, search
        error, model error), word-level precision / recall / F1, the model's score of each reachable gold path,
        and per gold word why it is outside the search space (`missing_words()` lists the dictionary's gaps).

        Gold words must have b < e with b increasing along the path.  A `flatten=True` lookup is not supported:
        its lattices hold single-morpheme words only, while gold words may have two."""
        from ..compile import _is_bmp
        from .evaluation import evaluate_pathset, ordered
        if self.score_funcs is None:
            raise TypeError("'NoneType' object is not callable")
        if self.eojeol_lookup.flatten:
            raise ValueError('evaluate() does not support a flatten=True lookup: its lattices hold single-morpheme words')
        sents = list(sents)
        golds = _inner_words(golds)
        if len(sents) != len(golds):
            raise ValueError('%d sentences but %d gold paths' % (len(sents), len(golds)))
        bad = [i for i, s in enumerate(sents) if not _is_bmp(s)]
        if bad:
            raise ValueError(self._engine._status_message(_native.LT_SENT_UNSUPPORTED_CHAR, bad[0]))
        if not ordered(golds):
            raise ValueError('every gold word needs b < e, and b must increase along its path')
        pathset = self._engine.upload_paths(golds)
        try:
            return evaluate_pathset(self._engine, sents, golds, pathset, beam_size)
        finally:
            pathset.close()

    def unpack(self, sents, packed, errors='raise'):
        return self._engine.unpack(sents, packed, errors)

    def edges_to_words(self, chars, edges):
        """Packed `lt_edge` records -> `Word` tuples (include/lt_b200.h documents the encoding)."""
        return self._engine.records_to_words(chars, edges.tolist())

    def lattice_batch(self, sents):
        """`sentence_lookup_as_begin_index` for every sentence: list of (words, bindex).

        `words` = [BOS] + dictionary edges + [EOS]; edges come grouped by end position then begin
        position, each (begin, end) group in the reference's order (the order `beam_search`
        observes); `bindex` is `[]` for a sentence without any dictionary edge
        (`lookup.py:362-363`).
        """
        sents = list(sents)
        out = []
        for sent, real in zip(sents, self.eojeol_lookup.lookup_batch(sents)):
            m = len(sent.replace(' ', ''))
            words = [Word(BOS, BOS, None, BOS, None, 0, 0, 0, False)] + real
            words.append(Word(EOS, EOS, None, EOS, None, 0, m, m, False))
            out.append((words, begin_index(m, real)))
        return out

    def counters(self):
        """Work counters of the last batch (SURVEY §8d): L, P, E, T, F, Bk, W."""
        return self._engine.counters()

    def timings(self):
        """Device times of the last batch by stage (first call only switches timing on)."""
        return self._engine.timings()

    def set_stage_timing(self, on):
        """Per-stage events between the kernels of a batch on / off for the batches to come."""
        self._engine.set_stage_timing(on)

    def info(self):
        """Workspace state: buffer capacities, reruns, kernel launches so far, launch shapes."""
        return self._engine.info()
