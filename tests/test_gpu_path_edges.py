"""The given-path kernels (csrc/paths.cuh) where they can go wrong: paths across the 32-word chunks a warp
walks, path sets and batches larger than the device's warps (the grid-stride loops), the perceptron step
on paths of more than two chunks, after every kind of search, on sentences the search could not tag and
with two trigram scorers, and the feature-buffer contract of lt_pathset_eval.  Every result is compared
with == against a plain host reference: the oracle's score program summed word by word in Python floats,
`SimpleTrigramEncoder.encode_sequence`, and the perceptron's host loop (`_same_path`, +-1.0 per feature
index).

The `check_*` functions take their sizes as arguments: tests/test_emulated_kernels.py runs them through the
SIMT emulator at smaller sizes, and tests/fuzz_emulated.py runs `check_path_stage` on every seed."""

import importlib.util
import os
import random

import numpy as np
import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native, synth
from lattice_based_tagger_b200.dictionary import Word
from lattice_based_tagger_b200.trainer.train import _same_path, train_epoch
from oracle import lattice_oracle as lo
from tests import _cases
from tests.test_gpu_paths import BOS, _dense_features, _eos, _oracle_score, _random_paths, _reference_epoch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTEXT_TAGS = ('Noun', 'Adverb', 'Adjective', 'Verb')           # kCtxMask (beam.cuh)
BOUNDARY_LENGTHS = (0, 1, 2, 31, 32, 33, 63, 64, 65, 96, 97, 300)
KINDS = ('context', 'unknown', 'lemma', 'long', 'plain')
# the fields of a word that _same_path compares, and the ones it does not
DIFFERING = ('boundary', 'tag0', 'tag1', 'morph0', 'morph1')
SAME = ('len', 'is_l', 'word')


def _scorers(funcs):
    return [f for f in funcs if isinstance(f, pkg.beam.SimpleTrigramFeatureScore)]


def _alphabet(case):
    return sorted({c for morphs in case['tag_to_morphs'].values() for m in morphs for c in m})


def _word(rng, kind, b, case, alphabet):
    """One word of a synthetic path at begin position b: a context-tagged word (templates 8 and the context
    flag), an unknown word of len 1..9 (template 6 through min(8, len)), a lemma word (morph1), a word of
    len >= 64 (template 4 hashed instead of dense; 64 itself is the first such length) or any word."""
    def text(n):
        return ''.join(rng.choice(alphabet) for _ in range(n))
    if kind == 'unknown':
        n = rng.randint(1, 9)
        s = text(n)
        return Word(s, s, None, 'Unknown', None, n, b, b + n, False)
    if kind == 'lemma':
        stem, eomi = text(rng.randint(1, 2)), text(rng.randint(1, 2))
        s = stem + eomi
        return Word(s, stem + rng.choice('다가'), eomi, rng.choice(['Verb', 'Adjective']), 'Eomi', len(s), b, b + len(s),
                    rng.random() < 0.5)
    tag = rng.choice(CONTEXT_TAGS) if kind == 'context' else rng.choice(case['tags'] + ['Unknown'])
    morphs = case['tag_to_morphs'].get(tag)
    s = rng.choice(morphs) if morphs and rng.random() < 0.7 else text(rng.randint(1, 4))
    n = rng.choice([63, 64, 64, 65, 130, 65535]) if kind == 'long' else len(s)
    return Word(s, s, None, tag, None, n, b, b + len(s), rng.random() < 0.3)


def boundary_paths(case, rng, per_length=6, lengths=BOUNDARY_LENGTHS):
    """`per_length` [BOS, ..., EOS] paths of each length; any kind of word anywhere, and around every chunk
    boundary (word positions 28..35 mod 32) mostly the kinds whose context crosses it."""
    alphabet = _alphabet(case)
    paths = []
    for n in lengths:
        for _ in range(per_length):
            words, b = [], 0
            for pos in range(n):
                near = pos >= 28 and (pos % 32 >= 28 or pos % 32 <= 3)
                kind = rng.choice(KINDS[:4] if near else KINDS)
                words.append(_word(rng, kind, b, case, alphabet))
                b = words[-1].e
            paths.append([BOS] + words + [_eos(b)])
    return paths


def _assert_boundary_coverage(paths):
    """The paths do what the test needs at some chunk boundary: an unknown word j whose capped length differs
    from the word before it (template 6 of the next chunk's first word), context tags on both sides, and a
    word of len 64."""
    unk = ctx = False
    for p in paths:
        words = p[1:-1]
        for first in range(32, len(words), 32):
            j, i, k = words[first - 1], words[first - 2], words[first]
            unk |= j.tag0 == 'Unknown' and min(8, j.len) != min(8, i.len)
            ctx |= k.tag0 in CONTEXT_TAGS and j.tag0 in CONTEXT_TAGS
    assert unk and ctx
    assert any(w.len == 64 for p in paths for w in p)


def _program(case, full, paths, rng, program):
    reg = next(f for f in full.funcs if isinstance(f, pkg.beam.RegularizationScore))
    prefs = [f for f in full.funcs if isinstance(f, (pkg.beam.MorphemePreferenceScore, pkg.beam.WordPreferenceScore))]
    if program == 'reg_trigram':
        return [reg] + _dense_features(paths, rng)
    assert program == 'all'
    return prefs[:1] + _dense_features(paths, rng) + [reg] + prefs[1:]


def _check_paths(tagger, funcs, paths):
    """score_paths against the oracle, encode_paths against encode_sequence, each distinct path computed once
    on the host."""
    oracle = lo.ScoreProgram(pkg.beam.BeamScoreFunctions(*funcs))
    scores, codes = {}, {}
    for p in paths:
        if id(p) not in scores:
            scores[id(p)] = _oracle_score(oracle, p)
    assert tagger.score_paths(paths).tolist() == [scores[id(p)] for p in paths]
    for scorer in _scorers(funcs):
        for p in paths:
            if (id(p), id(scorer)) not in codes:
                codes[id(p), id(scorer)] = scorer.encoder.encode_sequence(p)
        assert tagger.encode_paths(paths, scorer) == [codes[id(p), id(scorer)] for p in paths]


def _boundary_setup(seed, program, per_length, lengths=BOUNDARY_LENGTHS):
    rng = random.Random(seed)
    case = _cases.random_case(seed, n_sent=4, prefs=True)
    dictionary, full = _cases.build_objects(case, pkg)
    paths = boundary_paths(case, rng, per_length, lengths)
    funcs = _program(case, full, paths, rng, program)
    return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(*funcs)), funcs, paths


# ---- a. chunk boundaries, the path grid's stride, the feature buffer -----------------------------------

def check_chunk_boundaries(seed, program, per_length=6):
    tagger, funcs, paths = _boundary_setup(seed, program, per_length)
    _assert_boundary_coverage(paths)
    _check_paths(tagger, funcs, paths)
    hits = [len(x) for p in tagger.encode_paths(paths) for x in p]
    assert max(hits) >= 8


@pytest.mark.parametrize('seed', [21, 22])
@pytest.mark.parametrize('program', ['reg_trigram', 'all'])
def test_chunk_boundaries(seed, program):
    check_chunk_boundaries(seed, program)


def check_path_grid_stride(seed, per_length=3):
    """More paths than the launch has warps (2 * sm_count * 64 + 7 against sm_count * 8 CTAs of 8 warps):
    every warp takes several paths in turn, empty ones and paths of up to 300 words among them."""
    tagger, funcs, pool = _boundary_setup(seed, 'all', per_length)
    short = [p for p in pool if len(p) <= 4]
    long = [p for p in pool if len(p) > 34]
    n = 2 * tagger.info()['sm_count'] * 64 + 7
    paths = [long[(p // 5) % len(long)] if p % 5 == 2 else short[p % len(short)] for p in range(n)]
    assert sum(len(p) == 2 for p in paths) > n // 5
    _check_paths(tagger, funcs, paths)


def test_path_set_beyond_the_device_warps():
    check_path_grid_stride(23)


def test_feature_buffer_capacity():
    """lt_pathset_eval fills the caller's buffer when it holds exactly the hits, refuses one less with
    LT_ERR_CAPACITY, and its per-word offsets skip empty paths."""
    tagger, funcs, pool = _boundary_setup(24, 'reg_trigram', 1, lengths=(0, 3, 33, 64))
    scorer = _scorers(funcs)[0]
    empty = [BOS, _eos(0)]
    paths = [pool[1], empty, pool[2], empty, empty, pool[3], empty]
    codes = [x for p in paths for x in scorer.encoder.encode_sequence(p)]
    total = sum(len(x) for x in codes)
    engine = tagger._engine
    pathset = engine.upload_paths([p[1:-1] for p in paths])
    lib, func = tagger._lib, funcs.index(scorer)
    n_words = pathset.n_words
    assert n_words == len(codes)
    scores = np.zeros(len(paths))
    feat_off = np.full(n_words + 1, -7, dtype=np.int64)
    feat_idx = np.full(total + 1, -7, dtype=np.int32)

    def call(cap):
        return lib.lt_pathset_eval(tagger._batch, pathset.handle, func, _native.ptr(scores), _native.ptr(feat_off),
                                   _native.ptr(feat_idx), cap)
    assert call(total - 1) == 3                   # LT_ERR_CAPACITY
    assert call(total) == 0
    pathset.close()
    assert feat_off.tolist() == np.concatenate([[0], np.cumsum([len(x) for x in codes])]).tolist()
    desc_func, desc_fdic = engine.tables.desc_sources()
    assert (desc_func[feat_idx[:total]] == func).all()
    assert desc_fdic[feat_idx[:total]].tolist() == [i for x in codes for i in x]
    assert feat_idx[total] == -7


# ---- the perceptron step: host reference and gold paths ----------------------------------------------

def host_delta(golds, predicted, encoder):
    """The perceptron's host loop: (phi(gold) - phi(predicted) summed over the sentences whose prediction
    differs, per feature_dic index; the differs flags)."""
    want = np.zeros(max(encoder.feature_dic.values(), default=-1) + 1)
    differs = []
    for g, seq in zip(golds, predicted):
        d = seq is None or not _same_path(seq.sequences, g)
        differs.append(d)
        if d:
            for idxs in encoder.encode_sequence(g):
                np.add.at(want, idxs, 1.0)
            if seq is not None:
                for idxs in encoder.encode_sequence(seq.sequences):
                    np.add.at(want, idxs, -1.0)
    return want, differs


def check_delta(engine, pathset, golds, predicted, func, encoder):
    """lt_perceptron_delta after the engine's last search (whose best paths are `predicted`) against the host
    loop; -> the host's differs flags."""
    delta, differs, n_differ = engine.perceptron_delta(pathset, func)
    desc_func, desc_fdic = engine.tables.desc_sources()
    want, want_differs = host_delta(golds, predicted, encoder)
    got = np.zeros_like(want)
    mine = desc_func == func
    np.add.at(got, desc_fdic[mine], delta[mine].astype(np.float64))
    assert differs.tolist() == want_differs
    assert n_differ == sum(want_differs)
    assert got.tolist() == want.tolist()
    return want_differs


def change_field(words, pos, field, tags):
    """A copy of the [BOS, ..., EOS] path `words` with one field of inner word `pos` changed ('boundary': the
    boundary between it and its right neighbour, or its left one for the last word, moves by one)."""
    out = list(words)
    i = pos + 1
    w = out[i]
    if field == 'boundary':
        a = i if i + 1 < len(out) - 1 else i - 1
        assert a >= 1, 'a one-word path has no boundary to move'
        x, y = out[a], out[a + 1]
        shift = -1 if x.e - x.b > 1 else 1
        out[a], out[a + 1] = x._replace(e=x.e + shift), y._replace(b=y.b + shift)
    elif field == 'tag0':
        out[i] = w._replace(tag0=next(t for t in tags if t != w.tag0))
    elif field == 'tag1':
        out[i] = w._replace(tag1='Eomi' if w.tag1 is None else next(t for t in tags if t != w.tag1))
    elif field in ('morph0', 'morph1', 'word'):
        out[i] = w._replace(**{field: (getattr(w, field) or '') + '가'})
    elif field == 'len':
        out[i] = w._replace(len=w.len + 1)
    else:
        out[i] = w._replace(is_l=not w.is_l)
    return out


def near_misses(words, tags, positions=(0, 31, 32, 33, 64)):
    """(gold path, whether it differs from `words`) for every field at each position, and at the last word."""
    n = len(words) - 2
    out = []
    for pos in sorted({p for p in positions if p < n} | ({n - 1} if n else set())):
        for field in DIFFERING + SAME:
            if field == 'boundary' and n < 2:
                continue
            out.append((change_field(words, pos, field, tags), field in DIFFERING))
    return out


def _tilings(sent, tagger, rng, n):
    """n random tilings of `sent` (and the empty path)."""
    return _random_paths({'sentences': [sent], 'tags': _tags(tagger)}, tagger, rng, n)


def _tags(tagger):
    return [t for t in tagger._engine.tables.tag_names if t not in ('BOS', 'EOS')]


def long_sentences(case, n, min_syllables, limit):
    """n sentences of at least `min_syllables` syllables and fewer than `limit` UTF-16 units, each the case's
    sentences joined by spaces from a different start."""
    pool = [s.strip() for s in case['sentences'] if s.strip()]
    out = []
    for start in range(n):
        parts, k = [], start
        while sum(len(p.replace(' ', '')) for p in parts) < min_syllables:
            parts.append(pool[k % len(pool)])
            k += 1
        sent = ' '.join(parts)
        assert len(sent) < limit
        out.append(sent)
    return out


def _trained_tagger(seed, n_long, min_syllables, two_trigrams=False):
    """A tagger over a random case whose trigram features cover the reg-only search's paths and random
    tilings of long sentences; -> (tagger, funcs, case, long sentences, rng)."""
    rng = random.Random(seed)
    case = _cases.random_case(seed, n_sent=30, prefs=two_trigrams, max_sent_len=40)
    dictionary, full = _cases.build_objects(case, pkg)
    reg = next(f for f in full.funcs if isinstance(f, pkg.beam.RegularizationScore))
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    sents = long_sentences(case, n_long, min_syllables, probe.info()['unit_limit'])
    seen = [s.sequences for s in probe.tag_batch(sents, errors='none') if s is not None]
    for sent in sents:
        seen += _tilings(sent, probe, rng, 2)
    probe.close()
    if two_trigrams:
        pref = next(f for f in full.funcs if isinstance(f, pkg.beam.MorphemePreferenceScore))
        first, last = _dense_features(seen, rng, 2)
        funcs = [first, pref, reg, last]
    else:
        funcs = [reg] + _dense_features(seen, rng)
    return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(*funcs)), funcs, case, sents, rng


# ---- b. the perceptron on long sentences ---------------------------------------------------------------

def check_long_sentences(seed, n_long=3, min_syllables=200, beam_size=5):
    """Predictions of more than 64 words against themselves, random tilings and every one-field change at
    words 0, 31, 32, 33, 64 and the last: _same_path's fields make the sentence differ, len / is_l / word
    do not."""
    tagger, funcs, case, sents, rng = _trained_tagger(seed, n_long, min_syllables)
    scorer = _scorers(funcs)[0]
    predicted = tagger.tag_batch(sents, beam_size, errors='none')
    assert max(len(s.sequences) for s in predicted) > 66
    tags = _tags(tagger)
    batch, golds, expect = [], [], []
    for sent, seq in zip(sents, predicted):
        for gold, differs in [(list(seq.sequences), False)] + near_misses(seq.sequences, tags):
            golds.append(gold)
            expect.append(differs)
        for gold in _tilings(sent, tagger, rng, 3):
            golds.append(gold)
            expect.append(True)
        batch += [sent] * (len(golds) - len(batch))
    engine = tagger._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    predicted = engine.unpack(batch, engine.tag_packed(batch, beam_size), 'none')
    assert check_delta(engine, pathset, golds, predicted, funcs.index(scorer), scorer.encoder) == expect
    pathset.close()


@pytest.mark.parametrize('seed', [31, 32])
def test_perceptron_on_long_sentences(seed):
    check_long_sentences(seed)


# ---- c. batch states -------------------------------------------------------------------------------------

def _mixed_batch(tagger, case, sents, rng, beam_size, too_long=True):
    """Long sentences, each with its prediction, a near miss and a tiling as gold paths, and sentences the
    search does not tag: too long, empty, spaces only, no dictionary edge."""
    limit = tagger.info()['unit_limit']
    alphabet = _alphabet(case)
    predicted = tagger.tag_batch(sents, beam_size, errors='none')
    tags = _tags(tagger)
    batch, golds = [], []
    for sent, seq in zip(sents, predicted):
        n = len(seq.sequences) - 2
        miss = change_field(seq.sequences, rng.choice([p for p in (31, 32, 33, n - 1) if 0 <= p < n]),
                            rng.choice(DIFFERING + SAME), tags)
        golds += [list(seq.sequences), miss] + _tilings(sent, tagger, rng, 1)[1:]
        batch += [sent] * (len(golds) - len(batch))
    no_edge = case['sentences'][-1]
    beyond = alphabet[0] * (limit + 3)
    unknown = [BOS, Word(alphabet[0] * 3, alphabet[0] * 3, None, 'Unknown', None, 3, 0, 3, False), _eos(3)]
    for sent, gold in ((beyond, unknown), ('', [BOS, _eos(0)]), ('', unknown), ('   ', [BOS, _eos(0)]),
                       ('   ', unknown), (no_edge, unknown), (no_edge, [BOS, _eos(0)]))[0 if too_long else 1:]:
        batch.append(sent)
        golds.append(gold)
    return batch, golds


def _search(tagger, batch, beam_size, search):
    """Runs one kind of search on the batch; -> its best path per sentence (Sequence or None)."""
    engine = tagger._engine
    if search in ('tag', 'rerun'):
        packed = engine.tag_packed(batch, beam_size)
        assert set(packed[3].tolist()) >= {_native.LT_SENT_OK, _native.LT_SENT_NO_EDGES}
        assert _native.LT_SENT_TOO_LONG in packed[3] or search == 'rerun'
        return engine.unpack(batch, packed, 'none')
    imported = None
    if search == 'imported':
        imported = [words or [] for words in tagger.eojeol_lookup.lookup_batch(batch, errors='none')]
    packed = engine.kbest_packed(batch, beam_size, imported=imported)
    kept = engine.unpack_kbest(batch, packed, beam_size, 'none', engine._imported_words if imported else None)
    return [seqs[0] if seqs else None for seqs in kept]


def check_after_search(search, n_long=2, min_syllables=150, beam_size=4):
    """One gold path set against the best paths of each kind of search: lt_tag_batch_host, the k-best search,
    the k-best search over an imported lattice (string hashes from the import) and a search that outgrew its
    buffers and ran again; features of scorer 0 and of scorer 3 of [trigram, preference, regulariser,
    trigram] (the preference entries share the trigram features' table), each counted twice in turn."""
    tagger, funcs, case, sents, rng = _trained_tagger(41, n_long, min_syllables, two_trigrams=True)
    # (with staging areas this small, a batch sized for a sentence at the unit limit cannot grow them far
    # enough: the forced rerun leaves the too-long sentence out)
    batch, golds = _mixed_batch(tagger, case, sents, rng, beam_size, too_long=search != 'rerun')
    engine = tagger._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    predicted = _search(tagger, batch, beam_size, search)
    if search == 'rerun':
        assert tagger.info()['reruns'] > 0
    first = [check_delta(engine, pathset, golds, predicted, f, funcs[f].encoder) for f in (0, 3, 0)]
    assert first[0] == first[2] and any(first[0]) and not all(first[0])
    pathset.close()


@pytest.mark.parametrize('search', ['tag', 'kbest', 'imported', 'rerun'])
def test_perceptron_after_each_search(monkeypatch, search):
    if search == 'rerun':
        monkeypatch.setenv('LT_HIT_CAP', '8')
        monkeypatch.setenv('LT_EDGE_CAP', '16')
    check_after_search(search)


def check_batch_sequence(n_big=400, n_long=2, min_syllables=150, beam_size=4):
    """One tagger through a large batch, then a 3-sentence batch (stale scratch of the larger one), then new
    weights written in place (update_weights) and new weights compiled afresh (refresh)."""
    tagger, funcs, case, sents, rng = _trained_tagger(42, n_long, min_syllables, two_trigrams=True)
    batch, golds = _mixed_batch(tagger, case, sents, rng, beam_size)
    big = [i % len(batch) for i in range(n_big)]
    small = [0, 1, len(batch) - 1]
    rounds = [(big, None), (small, None), (small, 'update_weights'), (big[:len(batch)], 'refresh')]
    for which, change in rounds:
        if change:
            for f in (0, 3):
                funcs[f].coefficients = np.asarray([rng.choice([-2.0, 0.5, 1.0, 3.0]) for _ in funcs[f].coefficients])
            getattr(tagger, change)()
        sub_batch, sub_golds = [batch[i] for i in which], [golds[i] for i in which]
        engine = tagger._engine
        pathset = engine.upload_paths([g[1:-1] for g in sub_golds])
        predicted = engine.unpack(sub_batch, engine.tag_packed(sub_batch, beam_size), 'none')
        for f in (3, 0):
            check_delta(engine, pathset, sub_golds, predicted, f, funcs[f].encoder)
        pathset.close()


def test_perceptron_batch_sequence():
    check_batch_sequence()


# ---- d. the full C2 workload -----------------------------------------------------------------------------

@pytest.fixture(scope='module')
def c2_corpus():
    """C2's sentences, its feature dictionary, and gold paths from a tagger with those features and other
    seeded weights (profiles/tools/train_epoch.py)."""
    cfg, dictionary, sents = synth.build_workload('c2')
    beam = cfg['beam']
    reg = pkg.beam.RegularizationScore()
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    ok = [s for s, st in zip(sents, probe.tag_batch_packed(sents, beam)[3]) if st == 0]
    feature_dic, _ = synth.make_features(ok[:1000], lambda s: probe.tag_batch(s, beam, errors='none'), probe.lattice_batch,
                                         cfg['n_feat'], list(dictionary.tag_to_morphs), seed=3)
    probe.close()
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
    other = np.random.default_rng(11).normal(0.0, 1.0, len(feature_dic))
    teacher = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder, other)))
    taught = list(teacher.tag_batch(sents, beam, errors='none'))
    teacher.close()
    return beam, dictionary, reg, encoder, sents, taught


def test_perceptron_on_the_c2_workload(c2_corpus):
    """Every C2 sentence, repeated until the batch has more sentences than
    the launch has warps."""
    beam, dictionary, reg, encoder, sents, taught = c2_corpus
    coef = np.random.default_rng(12).normal(0.0, 1.0, len(encoder.feature_dic))
    student = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder, coef)))
    golds = [list(seq.sequences) if seq is not None else [BOS, _eos(0)] for seq in taught]
    reps = -(-2 * student.info()['sm_count'] * 64 // len(sents))
    want, want_differs = host_delta(golds, student.tag_batch(sents, beam, errors='none'), encoder)
    assert 0 < sum(want_differs) < len(sents)
    engine = student._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds] * reps)
    engine.tag_packed(sents * reps, beam)
    delta, differs, n_differ = engine.perceptron_delta(pathset, 1)
    pathset.close()
    desc_func, desc_fdic = engine.tables.desc_sources()
    got = np.zeros_like(want)
    np.add.at(got, desc_fdic[desc_func == 1], delta[desc_func == 1].astype(np.float64))
    assert differs.tolist() == want_differs * reps
    assert n_differ == reps * sum(want_differs)
    assert got.tolist() == (want * reps).tolist()


def test_train_epoch_many_to_one_on_the_c2_workload(c2_corpus):
    """One trainer epoch over the C2 annotation with a feature dictionary that maps three features to each
    index, against the host epoch."""
    beam, dictionary, reg, encoder, sents, taught = c2_corpus
    spec = importlib.util.spec_from_file_location('_train_epoch_tool', os.path.join(ROOT, 'profiles', 'tools', 'train_epoch.py'))
    tool = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tool)
    pairs = [tool.annotation(s, seq.sequences[1:-1]) for s, seq in zip(sents, taught) if seq is not None]
    pairs = [p for p in pairs if p is not None]
    n = max(1, len(encoder.feature_dic) // 3)
    many = pkg.features.SimpleTrigramEncoder({k: i % n for k, i in encoder.feature_dic.items()})
    coef = np.random.default_rng(13).normal(0.0, 1.0, len(encoder.feature_dic))

    def tagger():
        return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(many)))
    coef_dev, loss_dev = train_epoch(pairs, many, tagger(), coef, 1, False, beam_size=beam)
    coef_ref, loss_ref = _reference_epoch(pairs, many, tagger(), coef, beam)
    assert loss_dev == loss_ref > 0
    assert coef_dev.tolist() == coef_ref.tolist()


# ---- the path stage of tests/fuzz_emulated.py --------------------------------------------------------------

def check_path_stage(case, funcs, tagger, seed, beam_size):
    """score_paths / encode_paths on random tilings of the case's sentences, and the perceptron step with gold
    paths that are the prediction, a one-field near miss of it (at a chunk boundary when the path is long
    enough) or a random tiling."""
    rng = random.Random(seed ^ 0x9A7)
    _check_paths(tagger, list(funcs.funcs), _random_paths(case, tagger, rng))
    sents = case['sentences']
    predicted = tagger.tag_batch(sents, beam_size, errors='none')
    tags = _tags(tagger)
    golds = []
    for sent, seq in zip(sents, predicted):
        r = rng.random()
        n = -1 if seq is None else len(seq.sequences) - 2
        if n < 0 or r < 0.25:
            golds.append(_tilings(sent, tagger, rng, 1)[-1])
        elif n == 0 or r < 0.4:
            golds.append(list(seq.sequences))
        else:
            pos = [p for p in (31, 32, 33, 64, n - 1) if p < n]
            fields = DIFFERING + SAME if n > 1 else DIFFERING[1:] + SAME
            golds.append(change_field(seq.sequences, rng.choice(pos), rng.choice(fields), tags))
    engine = tagger._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    predicted = engine.unpack(sents, engine.tag_packed(sents, beam_size), 'none')
    for f, scorer in enumerate(funcs.funcs):
        if isinstance(scorer, pkg.beam.SimpleTrigramFeatureScore):
            check_delta(engine, pathset, golds, predicted, f, scorer.encoder)
    pathset.close()
