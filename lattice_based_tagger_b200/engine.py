"""`Engine` — one set of device tables plus a batch workspace, and the packing / unpacking between
Python strings / `Word` tuples and the C ABI's flat arrays (include/lt_b200.h).

Everything that computes runs in `liblt_b200.so`: an `Engine` only flattens its inputs, calls the
library and rebuilds `Word` / `Sequence` objects from the packed 16-byte records.  `Tagger`, the
eojeol-lookup classes (`dictionary/lookup.py`), `MorphemeDictionary.lookup / lemmatize`,
`analyze_morphology` and `beam_search` are thin layers over it.
"""

import contextlib
import ctypes
from collections.abc import Sequence as _SequenceABC

import numpy as np

from . import _native
from .compile import CompiledTables, _encode_units
from .tagset import BOS, EOS, Unk

_STATUS_MESSAGES = {
    _native.LT_SENT_BAD_SPACE: 'sentence %d contains whitespace other than U+0020',
    _native.LT_SENT_TOO_LONG: 'sentence %d is longer than the %d code units the device kernels hold',
    _native.LT_SENT_UNSUPPORTED_CHAR: 'sentence %d contains characters outside the Basic Multilingual Plane, '
                                      'which the device text format (UTF-16 code units) does not support',
    _native.LT_SENT_BAD_CONSTRAINT: 'sentence %d has a constraint that ends beyond its last syllable',
}


def _word_class():
    from .dictionary.dictionary import Word
    return Word


def _sequence_class():
    from .beam.beam import Sequence
    return Sequence


def pack_sentences(sents, unsupported=None):
    """list[str] -> (uint16 text, int32 offsets); spaces stay in the text (the kernels strip them).

    A sentence with characters outside the BMP has no one-unit-per-character UTF-16 form: with
    `unsupported` (a list) its index is recorded there and it travels as an empty sentence, so that
    the rest of the batch is tagged; without it the call raises `ValueError`.
    """
    n = len(sents)
    raw = ''.join(sents).encode('utf-16-le', 'surrogatepass')
    lengths = np.fromiter(map(len, sents), dtype=np.int64, count=n)
    offsets = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lengths, out=offsets[1:])
    if len(raw) != 2 * int(offsets[-1]):
        bad = [i for i, s in enumerate(sents) if len(s.encode('utf-16-le', 'surrogatepass')) != 2 * len(s)]
        if unsupported is None:
            raise ValueError(_STATUS_MESSAGES[_native.LT_SENT_UNSUPPORTED_CHAR] % bad[0])
        unsupported.extend(bad)
        sents = list(sents)
        for i in bad:
            sents[i] = ''
        raw = ''.join(sents).encode('utf-16-le', 'surrogatepass')
        lengths = np.fromiter(map(len, sents), dtype=np.int64, count=n)
        np.cumsum(lengths, out=offsets[1:])
    if offsets[-1] >= 2 ** 31:
        raise ValueError('batch holds %d code units; split it (limit 2^31)' % offsets[-1])
    text = np.frombuffer(raw, dtype='<u2')
    if text.size == 0:
        text = np.zeros(1, dtype='<u2')
    return np.ascontiguousarray(text), offsets.astype(np.int32)


class PackedSequences(_SequenceABC):
    """Result of `tag_batch`: behaves like `list[Sequence | None]`, but a sentence's `Sequence` (its
    `Word` tuples, BOS .. EOS) is only built when that item is read.  The packed arrays the device
    returned stay available as `.path_off`, `.path_edges`, `.scores`, `.status`."""

    def __init__(self, engine, sents, packed, errors):
        self._engine = engine
        self._sents = sents
        self.path_off, self.path_edges, self.scores, self.status = packed
        self._errors = errors
        self._cache = {}

    def __len__(self):
        return len(self._sents)

    def __getitem__(self, index):
        if isinstance(index, slice):
            return [self[i] for i in range(*index.indices(len(self)))]
        n = len(self)
        if index < 0:
            index += n
        if not 0 <= index < n:
            raise IndexError('list index out of range')
        if index not in self._cache:
            self._cache[index] = self._engine.sequence_at(self._sents[index], self, index, self._errors)
        return self._cache[index]

    def __eq__(self, other):
        if isinstance(other, (list, tuple, PackedSequences)):
            return len(self) == len(other) and all(a == b for a, b in zip(self, other))
        return NotImplemented

    def __repr__(self):
        return 'PackedSequences(%d sentences, %d words)' % (len(self), len(self.path_edges))

    def materialize(self):
        """All items as a plain list (one bulk conversion, faster than reading them one by one)."""
        return self._engine.unpack(self._sents, (self.path_off, self.path_edges, self.scores, self.status), self._errors)


class Engine:
    """Device tables of (dictionary, score functions) + one batch workspace."""

    def __init__(self, dictionary, score_funcs=None, device=0, k3_first=None, extra_tags=()):
        self._lib = _native.load()
        self.device = device
        self.tables = CompiledTables(dictionary, score_funcs, device, k3_first, extra_tags=extra_tags)
        handle = ctypes.c_void_p()
        _native.check(self._lib.lt_batch_create(self.tables.handle, ctypes.byref(handle)))
        self.batch = handle
        self._mode = _native.LT_LOOKUP_MORPHEME
        self.unit_limit = int(self._lib.lt_tables_max_sentence_units(self.tables.handle))

    def close(self):
        if getattr(self, 'batch', None) is not None:
            self._lib.lt_batch_destroy(self.batch)
            self.batch = None
        if getattr(self, 'tables', None) is not None:
            self.tables.close()
            self.tables = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- lookups ---------------------------------------------------------------------------------
    def set_lookup(self, mode):
        if mode != self._mode:
            _native.check(self._lib.lt_batch_set_lookup(self.batch, int(mode)))
            self._mode = mode

    # -- constraints -------------------------------------------------------------------------------
    def pack_constraints(self, sents, constraints):
        """Per sentence a list of `(b, e)` / `(b, e, tag_name)` spans the search must keep as words (`None` or `[]`:
        none) -> (`lt_constraint` records, int64 offsets).  Every malformed list raises `ValueError`: a count that
        is not one list per sentence, items that are not such tuples, b >= e, spans longer than the window or
        beyond the sentence's syllables, unsorted or overlapping spans, BOS / EOS / Unknown or a tag the tables do
        not know."""
        if len(constraints) != len(sents):
            raise ValueError('%d constraint lists for %d sentences' % (len(constraints), len(sents)))
        tag_ids = self.tables.tag_ids
        rec, off = [], [0]
        for i, (sent, items) in enumerate(zip(sents, constraints)):
            n_syl = len(sent.replace(' ', ''))
            prev_b, prev_e = -1, 0
            for k, item in enumerate(items or ()):
                where = 'sentence %d, constraint %d' % (i, k)
                if not isinstance(item, (tuple, list)) or len(item) not in (2, 3):
                    raise ValueError('%s: %r is not (b, e) or (b, e, tag)' % (where, item))
                b, e = item[0], item[1]
                tag = item[2] if len(item) == 3 else None
                if not all(isinstance(x, int) and not isinstance(x, bool) for x in (b, e)):
                    raise ValueError('%s: b and e must be integers, got %r' % (where, item))
                if not 0 <= b < e:
                    raise ValueError('%s: needs 0 <= b < e, got (%d, %d)' % (where, b, e))
                if e - b > _native.LT_WINDOW:
                    raise ValueError('%s: span (%d, %d) is longer than the %d-syllable window' % (where, b, e, _native.LT_WINDOW))
                if e > n_syl:
                    raise ValueError('%s: span (%d, %d) ends beyond the sentence\'s %d syllables' % (where, b, e, n_syl))
                if b < prev_b:
                    raise ValueError('%s: constraints must be sorted by b' % where)
                if b < prev_e:
                    raise ValueError('%s: span (%d, %d) overlaps the previous one' % (where, b, e))
                if tag is None:
                    tag_id = _native.LT_NO_TAG
                elif tag in (BOS, EOS, Unk):
                    raise ValueError('%s: %r is not a tag a constraint can ask for' % (where, tag))
                elif tag not in tag_ids:
                    raise ValueError('%s: tag %r is unknown to the compiled tables' % (where, tag))
                else:
                    tag_id = tag_ids[tag]
                rec.append((b, e, tag_id, (0, 0, 0)))
                prev_b, prev_e = b, e
            off.append(len(rec))
        cons = np.array(rec, dtype=_native.CONSTRAINT_DTYPE) if rec else np.zeros(1, dtype=_native.CONSTRAINT_DTYPE)
        return cons, np.array(off, dtype=np.int64)

    @contextlib.contextmanager
    def constrained(self, sents, constraints):
        """Within the block the batch's searches keep `constraints` (see `pack_constraints`; `None`: no binding):
        the set is validated, uploaded and bound here, and unbound and freed on the way out.  Fetch the results
        inside the block."""
        if constraints is None:
            yield
            return
        cons, off = self.pack_constraints(sents, constraints)
        handle = ctypes.c_void_p()
        _native.check(self._lib.lt_constraints_create(self.tables.handle, len(sents), _native.ptr(cons), _native.ptr(off),
                                                      ctypes.byref(handle)))
        try:
            _native.check(self._lib.lt_batch_set_constraints(self.batch, handle))
            try:
                yield
            finally:
                self._lib.lt_batch_set_constraints(self.batch, None)
        finally:
            self._lib.lt_constraints_destroy(handle)

    # -- tagging -----------------------------------------------------------------------------------
    def tag_packed(self, sents, beam_size, constraints=None):
        """The C-ABI call alone: (path_off, path_edges, scores, status) numpy arrays.  `constraints`: see
        `pack_constraints`."""
        if not 1 <= beam_size <= _native.LT_MAX_BEAM:
            raise ValueError('beam_size must be in 1..%d' % _native.LT_MAX_BEAM)
        unsupported = []
        text, offsets = pack_sentences(sents, unsupported)
        n = len(sents)
        cap = max(1, int(offsets[-1]))
        path_off = np.zeros(n + 1, dtype=np.int32)
        path_edges = np.empty(cap, dtype=_native.EDGE_DTYPE)
        scores = np.zeros(max(1, n), dtype=np.float64)
        status = np.zeros(max(1, n), dtype=np.int32)
        with self.constrained(sents, constraints):
            _native.check(self._lib.lt_tag_batch_host(
                self.batch, _native.ptr(text), _native.ptr(offsets), n, int(beam_size),
                _native.ptr(path_off), _native.ptr(path_edges), cap, _native.ptr(scores), _native.ptr(status)))
        for i in unsupported:
            status[i] = _native.LT_SENT_UNSUPPORTED_CHAR
        return path_off, path_edges[:int(path_off[n])], scores[:n], status[:n]

    def kbest_packed(self, sents, beam_size, imported=None, constraints=None):
        """All survivors: (n_best, path_off, path_edges, scores, status); `path_off` / `scores` are
        indexed by sentence * beam_size + rank.  With `imported` the lattice is the caller's.
        `constraints`: see `pack_constraints`."""
        if not 1 <= beam_size <= _native.LT_MAX_BEAM:
            raise ValueError('beam_size must be in 1..%d' % _native.LT_MAX_BEAM)
        n = len(sents)
        unsupported = []
        with self.constrained(sents, constraints):
            if imported is None:
                text, offsets = pack_sentences(sents, unsupported)
                _native.check(self._lib.lt_tag_batch_host_kbest(self.batch, _native.ptr(text), _native.ptr(offsets), n, int(beam_size)))
            else:
                self.import_lattice(sents, imported)
                _native.check(self._lib.lt_beam_kbest(self.batch, int(beam_size), None))
            total = ctypes.c_int64()
            _native.check(self._lib.lt_kbest_size(self.batch, ctypes.byref(total)))
            n_best = np.zeros(max(1, n), dtype=np.int32)
            path_off = np.zeros(n * beam_size + 1, dtype=np.int32)
            path_edges = np.empty(max(1, total.value), dtype=_native.EDGE_DTYPE)
            scores = np.zeros(max(1, n * beam_size), dtype=np.float64)
            status = np.zeros(max(1, n), dtype=np.int32)
            _native.check(self._lib.lt_kbest_fetch(self.batch, _native.ptr(n_best), _native.ptr(path_off), _native.ptr(path_edges),
                                                   path_edges.size, _native.ptr(scores), _native.ptr(status)))
        for i in unsupported:
            status[i] = _native.LT_SENT_UNSUPPORTED_CHAR
            n_best[i] = 0
        return n_best[:n], path_off, path_edges[:total.value], scores[:n * beam_size], status[:n]

    # -- lattices ----------------------------------------------------------------------------------
    def lattice_packed(self, sents):
        """(edges, end_off, offsets, status): the edges of all sentences sorted by (sentence, end,
        begin, reference order) and the CSR index over (sentence offset + end - 1)."""
        unsupported = []
        text, offsets = pack_sentences(sents, unsupported)
        n = len(sents)
        n_units = int(offsets[-1])
        _native.check(self._lib.lt_lattice_host(self.batch, _native.ptr(text), _native.ptr(offsets), n))
        n_edges = ctypes.c_int64()
        _native.check(self._lib.lt_lattice_size(self.batch, ctypes.byref(n_edges)))
        edges = np.empty(max(1, n_edges.value), dtype=_native.EDGE_DTYPE)
        end_off = np.zeros(n_units + 1, dtype=np.int64)
        _native.check(self._lib.lt_lattice_fetch(self.batch, _native.ptr(edges), edges.size, _native.ptr(end_off)))
        status = np.zeros(max(1, n), dtype=np.int32)
        _native.check(self._lib.lt_lattice_status(self.batch, _native.ptr(status), None))
        for i in unsupported:
            status[i] = _native.LT_SENT_UNSUPPORTED_CHAR
        return edges[:n_edges.value], end_off, offsets, status[:n]

    def lattice_words(self, sents, errors='raise'):
        """Per sentence the dictionary edges as `Word`s, grouped by end position then begin position,
        each (begin, end) group in the reference's order."""
        sents = list(sents)
        edges, end_off, offsets, status = self.lattice_packed(sents)
        records = edges.tolist()
        ends = end_off.tolist()
        offs = offsets.tolist()
        out = []
        for i, sent in enumerate(sents):
            st = int(status[i])
            if st not in (_native.LT_SENT_OK, _native.LT_SENT_NO_EDGES):
                if errors == 'raise':
                    raise ValueError(self._status_message(st, i))
                out.append(None)
                continue
            chars = sent.replace(' ', '')
            out.append(self.records_to_words(chars, records[ends[offs[i]]:ends[offs[i + 1]]]))
        return out

    def pack_words(self, words):
        """`Word`s -> LT_EDGE_EXPLICIT records (record i names strings 3i, 3i+1, 3i+2: word, morph0,
        morph1) and those strings as UTF-16: (edges, units, str_off, n_strings).  A tag the tables do not
        know, a string outside the BMP or a field outside the record's range raises `ValueError`."""
        tag_ids = self.tables.tag_ids
        other = self.tables.other_tag_id
        rec, strings = [], []
        for idx, w in enumerate(words):
            if not 0 <= w.len < 65536:
                raise ValueError('Word.len %r is outside 0..65535' % (w.len,))
            if not (0 <= w.b < 65536 and 0 <= w.e < 65536):
                raise ValueError('Word span [%r, %r) is outside 0..65535' % (w.b, w.e))
            tag0 = tag_ids.get(w.tag0, other)
            tag1 = 0xFF if w.tag1 is None else tag_ids.get(w.tag1, other)
            if tag0 is None or tag1 is None:
                raise ValueError('tag %r / %r is unknown to the compiled tables' % (w.tag0, w.tag1))
            flags = (_native.LT_EDGE_EXPLICIT | (_native.LT_EDGE_IS_L if w.is_l else 0) |
                     (_native.LT_EDGE_LEMMA if w.tag1 is not None else 0))
            rec.append((w.b, w.e, int(w.len), tag0, tag1, idx, 0, flags, 0))
            strings += [w.word, w.morph0, w.morph1 or '']
        edges = np.array(rec, dtype=_native.EDGE_DTYPE) if rec else np.zeros(1, dtype=_native.EDGE_DTYPE)
        units, str_off = _encode_units(strings)
        return edges, units, str_off, len(strings)

    def import_lattice(self, sents, lattices):
        """Upload caller-built lattices (`lattices[i]` = iterable of `Word`s of sentence i, any order)
        for `lt_beam*`; returns the flat list of the imported `Word`s (index = record.rule)."""
        text, offsets = pack_sentences(sents)
        n = len(sents)
        n_units = int(offsets[-1])
        flat = []
        end_off = np.zeros(n_units + 1, dtype=np.int64)
        for i, words in enumerate(lattices):
            m = len(sents[i].replace(' ', ''))
            base, top = int(offsets[i]), int(offsets[i + 1])
            usable = []
            for order, w in enumerate(words or ()):
                # only spans inside the sentence can be used by the search (beam.py:30-33); zero-width words
                # (flatten_words produces them) are never expanded
                if 0 <= w.b < w.e <= m:
                    usable.append((w.e, w.b, order, w))
            usable.sort(key=lambda t: t[:3])
            counts = np.zeros(top - base, dtype=np.int64)
            start = len(flat)
            for e, _, _, w in usable:
                flat.append(w)
                counts[e - 1] += 1
            if top > base:
                end_off[base + 1:top + 1] = start + np.cumsum(counts)
        edges, units, str_off, n_strings = self.pack_words(flat)
        _native.check(self._lib.lt_lattice_import(self.batch, _native.ptr(text), _native.ptr(offsets), n, _native.ptr(edges),
                                                  _native.ptr(end_off), _native.ptr(units), _native.ptr(str_off), n_strings))
        self._imported_words = flat
        return flat

    # -- given paths -----------------------------------------------------------------------------------
    def upload_paths(self, paths):
        """`paths[p]` = the `Word`s of path p without BOS / EOS -> a `PathSet` on these tables."""
        return PathSet(self, paths)

    def trainer(self, sents, gold, func, n_coef, feat_coef, coef, update='full'):
        """A `DeviceTrainer` over `sents` (gold path i for sentence i) training scorer index `func` with `update`
        ('full', 'early' or 'max_violation')."""
        return DeviceTrainer(self, sents, gold, func, n_coef, feat_coef, coef, update)

    def eval_paths(self, pathset, func=None):
        """lt_pathset_eval: (scores, feat_off, feat_idx); the features (of scorer index `func`, desc order)
        only with `func`, else (scores, None, None)."""
        n = pathset.n_paths
        scores = np.zeros(max(1, n), dtype=np.float64)
        if func is None:
            _native.check(self._lib.lt_pathset_eval(self.batch, pathset.handle, -1, _native.ptr(scores), None, None, 0))
            return scores[:n], None, None
        feat_off = np.zeros(pathset.n_words + 1, dtype=np.int64)
        feat_idx = np.zeros(max(1, 9 * pathset.n_words), dtype=np.int32)
        _native.check(self._lib.lt_pathset_eval(self.batch, pathset.handle, int(func), _native.ptr(scores),
                                                _native.ptr(feat_off), _native.ptr(feat_idx), feat_idx.size))
        return scores[:n], feat_off, feat_idx[:int(feat_off[-1])]

    def perceptron_delta(self, gold, func):
        """lt_perceptron_delta against the last search: (delta in desc order, differs, n_differ)."""
        n_feat = self.tables.n_desc
        delta = np.zeros(max(1, n_feat), dtype=np.int64)
        differs = np.zeros(max(1, gold.n_paths), dtype=np.uint8)
        n_differ = ctypes.c_int64()
        _native.check(self._lib.lt_perceptron_delta(self.batch, gold.handle, int(func), _native.ptr(delta), n_feat,
                                                    _native.ptr(differs), ctypes.byref(n_differ)))
        return delta[:n_feat], differs[:gold.n_paths].astype(bool), int(n_differ.value)

    def evaluate(self, gold):
        """lt_evaluate against the last search: (sent_class uint8 [n], counts int32 [n, LT_EVAL_N_COUNTS],
        gold_scores float64 [n] (NaN unless reachable), word_reason uint8 [gold.n_words])."""
        n = gold.n_paths
        sent_class = np.zeros(max(1, n), dtype=np.uint8)
        counts = np.zeros((max(1, n), _native.LT_EVAL_N_COUNTS), dtype=np.int32)
        gold_scores = np.zeros(max(1, n), dtype=np.float64)
        word_reason = np.zeros(max(1, gold.n_words), dtype=np.uint8)
        _native.check(self._lib.lt_evaluate(self.batch, gold.handle, _native.ptr(sent_class), _native.ptr(counts),
                                            _native.ptr(gold_scores), _native.ptr(word_reason)))
        return sent_class[:n], counts[:n], gold_scores[:n], word_reason[:gold.n_words]

    # -- unpacking -----------------------------------------------------------------------------------
    def _status_message(self, st, index):
        msg = _STATUS_MESSAGES.get(st, 'sentence %d could not be tagged')
        return msg % ((index, self.unit_limit) if st == _native.LT_SENT_TOO_LONG else index)

    def _raise_for(self, st, index):
        if st == _native.LT_SENT_NO_EDGES:
            raise IndexError('list index out of range')       # as the reference does (lookup.py:362-363 + beam.py:33)
        raise ValueError(self._status_message(st, index))

    def records_to_words(self, chars, records, imported=None):
        """Packed `lt_edge` tuples -> `Word` tuples (include/lt_b200.h documents the encoding)."""
        Word = _word_class()
        names = self.tables.tag_names
        rules = self.tables.rules_flat
        lemma_flag, is_l_flag, explicit = _native.LT_EDGE_LEMMA, _native.LT_EDGE_IS_L, _native.LT_EDGE_EXPLICIT
        new = tuple.__new__            # Word is a namedtuple: skips the per-call length check of _make
        words = []
        for b, e, length, tag0, tag1, rule, split, flags, _ in records:
            if flags & explicit:
                words.append(imported[rule])
                continue
            surface = chars[b:e]
            is_l = (flags & is_l_flag) != 0
            if flags & lemma_flag:
                if rule == _native.LT_NO_RULE:
                    morph0, morph1 = surface[:split + 1], surface[split + 1:]
                else:
                    stem, eomi = rules[rule]
                    skip = 2 if flags & _native.LT_EDGE_SKIP2 else 1
                    morph0, morph1 = surface[:split] + stem, eomi + surface[split + skip:]
                words.append(new(Word, (surface, morph0, morph1, names[tag0], names[tag1], length, b, e, is_l)))
            else:
                words.append(new(Word, (surface, surface, None, names[tag0], None, length, b, e, is_l)))
        return words

    def _sequence(self, sent, records, score, imported=None):
        Word = _word_class()
        chars = sent.replace(' ', '')
        n = len(chars)
        words = [Word(BOS, BOS, None, BOS, None, 0, 0, 0, False)]
        words += self.records_to_words(chars, records, imported)
        words.append(Word(EOS, EOS, None, EOS, None, 0, n, n, False))
        # adding EOS resets the trailing-unknown count (beam.py:113 with tag0 == EOS)
        return _sequence_class()(words, score, 0)

    def sequence_at(self, sent, packed, index, errors):
        st = int(packed.status[index])
        if st != _native.LT_SENT_OK:
            if errors == 'raise':
                self._raise_for(st, index)
            return None
        lo, hi = int(packed.path_off[index]), int(packed.path_off[index + 1])
        return self._sequence(sent, packed.path_edges[lo:hi].tolist(), float(packed.scores[index]))

    def unpack(self, sents, packed, errors='raise'):
        path_off, path_edges, scores, status = packed
        # one conversion for the whole batch (per-sentence numpy slicing dominates otherwise)
        offs = path_off.tolist()
        records = path_edges.tolist()
        score_list = scores.tolist()
        status_list = status.tolist()
        out = []
        for i, sent in enumerate(sents):
            st = status_list[i]
            if st != _native.LT_SENT_OK:
                if errors == 'raise':
                    self._raise_for(st, i)
                out.append(None)
                continue
            out.append(self._sequence(sent, records[offs[i]:offs[i + 1]], score_list[i]))
        return out

    def unpack_kbest(self, sents, packed, beam_size, errors='raise', imported=None):
        """list (per sentence) of list of `Sequence` — every survivor, best first (beam.py:59-61)."""
        n_best, path_off, path_edges, scores, status = packed
        offs = path_off.tolist()
        records = path_edges.tolist()
        score_list = scores.tolist()
        out = []
        for i, sent in enumerate(sents):
            st = int(status[i])
            if st != _native.LT_SENT_OK:
                if errors == 'raise':
                    self._raise_for(st, i)
                out.append(None)
                continue
            base = i * beam_size
            out.append([self._sequence(sent, records[offs[base + r]:offs[base + r + 1]], score_list[base + r], imported)
                        for r in range(int(n_best[i]))])
        return out

    # -- instrumentation -------------------------------------------------------------------------------
    def counters(self):
        c = _native.lt_counters()
        _native.check(self._lib.lt_batch_counters(self.batch, ctypes.byref(c)))
        return c.as_dict()

    def timings(self):
        t = _native.lt_timings()
        _native.check(self._lib.lt_batch_timings(self.batch, ctypes.byref(t)))
        return t.as_dict()

    def set_stage_timing(self, on):
        """Per-stage CUDA events between the kernels of a batch on / off."""
        _native.check(self._lib.lt_batch_set_stage_timing(self.batch, 1 if on else 0))

    def info(self):
        i = _native.lt_info()
        _native.check(self._lib.lt_batch_info(self.batch, ctypes.byref(i)))
        return i.as_dict()


class PathSet:
    """Word paths on the device (`lt_pathset`), tied to one `Engine`'s tables: packed once, then scored,
    featurized or compared with the engine's search results as often as needed."""

    def __init__(self, engine, paths):
        self._lib = engine._lib
        self.tables = engine.tables
        self.handle = None
        lengths = [len(p) for p in paths]
        off = np.zeros(len(paths) + 1, dtype=np.int64)
        np.cumsum(lengths, out=off[1:])
        edges, units, str_off, n_strings = engine.pack_words([w for p in paths for w in p])
        handle = ctypes.c_void_p()
        _native.check(self._lib.lt_pathset_create(self.tables.handle, len(paths), _native.ptr(edges), _native.ptr(off),
                                                  _native.ptr(units), _native.ptr(str_off), n_strings, ctypes.byref(handle)))
        self.handle = handle
        self.n_paths = len(paths)
        self.n_words = int(off[-1])
        self.path_off = off

    def close(self):
        if self.handle is not None:
            self._lib.lt_pathset_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceTrainer:
    """Mini-batch perceptron on the device (`lt_trainer`), tied to one `Engine`: the corpus `sents` and its gold
    `PathSet` (which must stay open while the trainer lives) go up once; `step(first, count, beam_size)` decodes
    sentences [first, first + count) on the engine's batch and updates the weights there; `fetch()` brings them
    back.  `feat_coef[i]`: the coefficient of desc feature i (`CompiledTables.desc_sources` order) of scorer
    `func`, -1 for the others; `coef`: the initial weights, written into the tables at once.  `update` ('full',
    'early' or 'max_violation', see `lt_trainer_set_update`) applies to the steps that follow and may be changed
    between them with `set_update`."""

    UPDATE_MODES = {'full': _native.LT_UPDATE_FULL, 'early': _native.LT_UPDATE_EARLY,
                    'max_violation': _native.LT_UPDATE_MAX_VIOLATION}

    def __init__(self, engine, sents, gold, func, n_coef, feat_coef, coef, update='full'):
        self._lib = engine._lib
        self._engine = engine
        self.handle = None
        text, offsets = pack_sentences(sents)
        feat_coef = np.ascontiguousarray(feat_coef, dtype=np.int64)
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        if len(coef) != n_coef:
            raise ValueError('%d initial weights for %d coefficients' % (len(coef), n_coef))
        if len(feat_coef) != engine.tables.n_desc:
            raise ValueError('feat_coef has %d entries, the tables %d features' % (len(feat_coef), engine.tables.n_desc))
        if update not in self.UPDATE_MODES:         # (before lt_trainer_create, which writes coef into the tables)
            raise ValueError('update must be one of %s, got %r' % (', '.join(self.UPDATE_MODES), update))
        handle = ctypes.c_void_p()
        _native.check(self._lib.lt_trainer_create(
            engine.tables.handle, int(func), _native.ptr(text), _native.ptr(offsets), len(sents), gold.handle, int(n_coef),
            _native.ptr(feat_coef) if feat_coef.size else None, _native.ptr(coef) if coef.size else None, ctypes.byref(handle)))
        self.handle = handle
        self.n_sent = len(sents)
        self.n_coef = int(n_coef)
        self.set_update(update)

    def set_update(self, update):
        """The update of the following steps: 'full', 'early' or 'max_violation'."""
        if update not in self.UPDATE_MODES:
            raise ValueError('update must be one of %s, got %r' % (', '.join(self.UPDATE_MODES), update))
        _native.check(self._lib.lt_trainer_set_update(self.handle, self.UPDATE_MODES[update]))

    def step(self, first, count, beam_size):
        _native.check(self._lib.lt_trainer_step(self.handle, self._engine.batch, int(first), int(count), int(beam_size)))

    def fetch(self):
        """-> (coef, averaged, steps, mistakes, differs): the weights, their mean over the steps so far, the number
        of steps, of mistaken sentences summed over them, and per sentence whether its last step got it wrong."""
        coef = np.zeros(max(1, self.n_coef), dtype=np.float64)
        averaged = np.zeros_like(coef)
        differs = np.zeros(max(1, self.n_sent), dtype=np.uint8)
        steps, mistakes = ctypes.c_int64(), ctypes.c_int64()
        _native.check(self._lib.lt_trainer_fetch(self.handle, _native.ptr(coef), _native.ptr(averaged), ctypes.byref(steps),
                                                 ctypes.byref(mistakes), _native.ptr(differs)))
        return coef[:self.n_coef], averaged[:self.n_coef], int(steps.value), int(mistakes.value), differs[:self.n_sent].astype(bool)

    def update_info(self):
        """-> (prefix_words int32 [n_sent], violation float64 [n_sent]) per sentence, from the last step that covered
        it: the gold words the update took (0: no update, W: the whole path) and B - G at that prefix, the score of
        the best hypothesis minus the gold prefix's (NaN without an update, for a full step or a gold path that
        does not tile the sentence)."""
        prefix = np.zeros(max(1, self.n_sent), dtype=np.int32)
        violation = np.zeros(max(1, self.n_sent), dtype=np.float64)
        _native.check(self._lib.lt_trainer_fetch_update(self.handle, _native.ptr(prefix), _native.ptr(violation)))
        return prefix[:self.n_sent], violation[:self.n_sent]

    def close(self):
        if self.handle is not None:
            self._lib.lt_trainer_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
