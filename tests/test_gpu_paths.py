"""Given paths on the device: `Tagger.score_paths` / `encode_paths` (lt_pathset_eval) against the search's own
scores, the oracle's transition arithmetic and `SimpleTrigramEncoder.encode_sequence`; the perceptron step
(lt_perceptron_delta) and the trainer epoch built on it against the host loop they replace."""

import ctypes
import random

import numpy as np
import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native, synth
from lattice_based_tagger_b200.dictionary import Word
from lattice_based_tagger_b200.dictionary.text import text_to_words
from lattice_based_tagger_b200.trainer import train
from lattice_based_tagger_b200.trainer.train import _same_path, _surface, fit_parameter, train_epoch
from oracle import lattice_oracle as lo
from tests import _cases, _golden

pytestmark = pytest.mark.gpu

BOS = Word('BOS', 'BOS', None, 'BOS', None, 0, 0, 0, False)


def _eos(n):
    return Word('EOS', 'EOS', None, 'EOS', None, 0, n, n, False)


def _oracle_score(program, words):
    words = [tuple(w) for w in words]
    score = 0
    for i in range(1, len(words) - 1):
        score = score + program.increment(None if i == 1 else words[i - 2], words[i - 1], words[i])
    return score


# ---- the search's own paths ----------------------------------------------------------------------------

@pytest.mark.parametrize('name', ['demo_morph', 'base_c1', 'random_1000', 'random_1003', 'random_1007', 'random_1012'])
def test_scores_of_searched_paths(name):
    payload = _golden.load(name)
    case = payload['case']
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs, k3_first=payload['k3_first'])
    sents = case['sentences']
    best = [s for s in tagger.tag_batch(sents, beam_size=5, errors='none') if s is not None]
    got = tagger.score_paths(best)
    assert got.dtype == np.float64 and len(got) == len(best)
    assert got.tolist() == [s.score for s in best]
    survivors = [seq for seqs in tagger.tag_batch_kbest(sents, beam_size=7, errors='none') if seqs for seq in seqs]
    assert tagger.score_paths(survivors).tolist() == [s.score for s in survivors]


@pytest.fixture(scope='module')
def c2_sample():
    cfg, dictionary, sents = synth.build_workload('c2', n_sent=400)
    reg = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore())
    reg_tagger = pkg.Tagger(dictionary, score_funcs=reg)
    feature_dic, coef = synth.make_features(
        sents, lambda s: reg_tagger.tag_batch(s, cfg['beam'], errors='none'), reg_tagger.lattice_batch,
        cfg['n_feat'], list(dictionary.tag_to_morphs), seed=3)
    reg_tagger.close()
    funcs = pkg.beam.BeamScoreFunctions(
        pkg.beam.RegularizationScore(),
        pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    return cfg, dictionary, funcs, sents


def test_scores_of_searched_paths_c2(c2_sample):
    cfg, dictionary, funcs, sents = c2_sample
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    best = [s for s in tagger.tag_batch(sents, cfg['beam'], errors='none') if s is not None]
    assert tagger.score_paths(best).tolist() == [s.score for s in best]
    survivors = [seq for seqs in tagger.tag_batch_kbest(sents[:100], cfg['beam'], errors='none') if seqs for seq in seqs]
    assert tagger.score_paths(survivors).tolist() == [s.score for s in survivors]
    encoder = funcs.funcs[1].encoder
    assert tagger.encode_paths(best[:100]) == [encoder.encode_sequence(s.sequences) for s in best[:100]]


# ---- arbitrary paths -----------------------------------------------------------------------------------

def _random_paths(case, tagger, rng, n_paths=40):
    """Random tilings of the case's sentences: lattice words, unknown words of any width (beyond 8 too), lemma
    words, Word.len != e - b, both is_l values, and the empty path."""
    tags = case['tags']
    paths = [[BOS, _eos(0)]]
    lattices = tagger.lattice_batch(case['sentences'])
    for _ in range(n_paths):
        sent = rng.choice(case['sentences'])
        chars = sent.replace(' ', '')
        if not chars:
            continue
        words = lattices[case['sentences'].index(sent)][0][1:-1]
        by_span = {}
        for w in words:
            by_span.setdefault((w.b, w.e), []).append(w)
        path, b = [], 0
        while b < len(chars):
            starts = [w for (wb, _), ws in by_span.items() if wb == b for w in ws]
            r = rng.random()
            if starts and r < 0.5:
                w = rng.choice(starts)
            else:
                e = min(len(chars), b + rng.randint(1, 12))
                surface = chars[b:e]
                if r < 0.75:
                    w = Word(surface, surface, None, 'Unknown', None, e - b, b, e, False)
                else:
                    split = rng.randint(1, max(1, len(surface)))
                    w = Word(surface, surface[:split] + rng.choice('가나'), rng.choice('다요') + surface[split:],
                             rng.choice(['Verb', 'Adjective']), 'Eomi', e - b, b, e, False)
            if rng.random() < 0.2:
                w = w._replace(len=rng.randint(0, 70))
            if rng.random() < 0.3:
                w = w._replace(is_l=not w.is_l)
            if rng.random() < 0.1:
                w = w._replace(tag0=rng.choice(tags))
            path.append(w)
            b = w.e
        paths.append([BOS] + path + [_eos(len(chars))])
    return paths


def _dense_features(paths, rng, n_scorers=1):
    """feature_dic over every tuple the paths generate (so that 8 and 9 weights fire on many transitions)."""
    keys = set()
    for words in paths:
        for i in range(1, len(words) - 1):
            keys.update(lo.feature_tuples(None if i == 1 else tuple(words[i - 2]), tuple(words[i - 1]), tuple(words[i])))
    keys = sorted(keys, key=repr)
    out = []
    for s in range(n_scorers):
        chosen = [k for k in keys if rng.random() < 0.95]
        feature_dic = {k: i for i, k in enumerate(chosen)}
        coef = np.array([rng.choice([rng.gauss(0, 1), 1e-17, 3.0, -0.5]) for _ in chosen], dtype=np.float64)
        out.append(pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    return out


@pytest.mark.parametrize('seed', [1000, 1003, 1005])
@pytest.mark.parametrize('program', ['reg', 'reg_trigram', 'all', 'two_trigram'])
def test_arbitrary_paths_against_oracle(seed, program):
    rng = random.Random(seed * 7 + len(program))
    case = _cases.random_case(seed, n_sent=10, prefs=True)
    dictionary, full = _cases.build_objects(case, pkg)
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore()))
    paths = _random_paths(case, probe, rng)
    probe.close()
    reg = next(f for f in full.funcs if isinstance(f, pkg.beam.RegularizationScore))
    prefs = [f for f in full.funcs if isinstance(f, (pkg.beam.MorphemePreferenceScore, pkg.beam.WordPreferenceScore))]
    if program == 'reg':
        funcs = [reg]
    elif program == 'reg_trigram':
        funcs = [reg] + _dense_features(paths, rng)
    elif program == 'all':
        funcs = prefs[:1] + _dense_features(paths, rng) + [reg] + prefs[1:]
    else:
        funcs = _dense_features(paths, rng, 2)
    score_funcs = pkg.beam.BeamScoreFunctions(*funcs)
    tagger = pkg.Tagger(dictionary, score_funcs=score_funcs)
    oracle = lo.ScoreProgram(score_funcs)
    got = tagger.score_paths(paths)
    assert got.tolist() == [_oracle_score(oracle, p) for p in paths]
    assert tagger.score_paths([pkg.beam.beam.Sequence(p, 0.0) for p in paths]).tolist() == got.tolist()
    for scorer in [f for f in funcs if isinstance(f, pkg.beam.SimpleTrigramFeatureScore)]:
        assert tagger.encode_paths(paths, scorer) == [scorer.encoder.encode_sequence(p) for p in paths]
        if scorer is funcs[0] or program != 'two_trigram':
            hits = [len(x) for p in tagger.encode_paths(paths, scorer) for x in p]
            assert max(hits) >= 8


def test_encode_paths_many_to_one_feature_dic():
    rng = random.Random(5)
    case = _cases.random_case(1004, n_sent=10)
    dictionary, _ = _cases.build_objects(case, pkg)
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore()))
    paths = _random_paths(case, probe, rng)
    probe.close()
    scorer = _dense_features(paths, rng)[0]
    fdic = scorer.encoder.feature_dic
    n = max(1, len(fdic) // 3)
    scorer.encoder.feature_dic = {k: i % n for k, i in fdic.items()}
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(), scorer))
    assert tagger.encode_paths(paths) == [scorer.encoder.encode_sequence(p) for p in paths]


# ---- perceptron step -------------------------------------------------------------------------------------

PAIRS = [
    ('너무너무너무 는  아이오아이 의  노래  입니다',
     '너무너무너무/Noun 는/Josa  아이오아이/Noun 의/Josa  노래/Noun  이/Adjective+ㅂ니다/Eomi'),
    ('아이 는  노래 를  했다', '아이/Noun 는/Josa  노래/Noun 를/Josa  하/Verb+았다/Eomi'),
    ('아이오아이 는  공연 을  했다', '아이오아이/Noun 는/Josa  공연/Noun 을/Josa  하/Verb+았다/Eomi'),
    ('우와  노래 이  있다', '우와/Exclamation  노래/Noun 이/Josa  있/Adjective+다/Eomi'),
    ('아이 의  노래 는  공연 입니다', '아이/Noun 의/Josa  노래/Noun 는/Josa  공연/Noun 이/Adjective+ㅂ니다/Eomi'),
    ('노래  아이', '노래/Suffix  아이/Noun'),                        # a gold tag the dictionary lacks
    ('뷁뷁', '뷁뷁/Noun'),                                           # no dictionary edge
    ('노래 \U0001F600', '노래/Noun \U0001F600/Noun'),                # outside the BMP
]


def _reference_epoch(word_morph_pairs, encoder, tagger, coef, beam_size=5):
    """The trainer's epoch as a host loop (the definition the device step must reproduce)."""
    coef = np.asarray(coef, dtype=np.float64).copy()
    scorer = next(f for f in tagger.score_funcs.funcs if isinstance(f, pkg.beam.SimpleTrigramFeatureScore))
    if scorer.encoder is encoder and getattr(tagger, '_trained_features', None) is encoder.feature_dic:
        scorer.coefficients = coef
        tagger.update_weights()
    else:
        scorer.set_encoder(encoder, coef)
        tagger.refresh()
        tagger._trained_features = encoder.feature_dic
    golds, sents = [], []
    for word_text, morph_text in word_morph_pairs:
        try:
            gold = text_to_words(word_text, morph_text)
        except Exception:
            continue
        golds.append(gold)
        sents.append(_surface(word_text))
    update = np.zeros_like(coef)
    loss = 0
    for gold, seq in zip(golds, tagger.tag_batch(sents, beam_size=beam_size, errors='none')):
        if seq is not None and _same_path(seq.sequences, gold):
            continue
        loss += 1
        for idxs in encoder.encode_sequence(gold):
            for idx in idxs:
                update[idx] += 1.0
        if seq is not None:
            for idxs in encoder.encode_sequence(seq.sequences):
                for idx in idxs:
                    update[idx] -= 1.0
    coef += update
    return coef, loss


def _toy_tagger(extra_tags=()):
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    reg = pkg.beam.RegularizationScore(unknown_penalty=-0.1, known_preference=-0.3, syllable_penalty=0.0)
    golds = []
    for w, m in PAIRS:
        golds.append(text_to_words(w, m))
    keys = set()
    for g in golds:
        for idxs in pkg.features.SimpleTrigramEncoder().transform_sequence(g):
            keys.update(idxs)
    keys = sorted(keys, key=repr)
    encoder = pkg.features.SimpleTrigramEncoder({k: i for i, k in enumerate(keys)})
    rng = np.random.default_rng(0)
    coef = rng.choice([-1.0, 0.0, 1.0, 2.0], size=len(keys))
    scorer = pkg.beam.SimpleTrigramFeatureScore(encoder, coef)
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, scorer), extra_tags=extra_tags)
    return tagger, encoder, scorer, reg, dictionary


def test_perceptron_delta_against_host_loop():
    tagger, encoder, scorer, reg, _ = _toy_tagger(extra_tags=['Suffix'])
    pairs = [p for p in PAIRS if all(ord(c) < 0x10000 for c in p[0])]
    golds = [text_to_words(w, m) for w, m in pairs]
    sents = [_surface(w) for w, _ in pairs]
    predicted = tagger.tag_batch(sents, errors='none')
    # a right prediction, and one equal to gold except for Word.len / is_l
    golds[1] = list(predicted[1].sequences)
    g2 = list(predicted[2].sequences)
    g2[1] = g2[1]._replace(len=g2[1].len + 3, is_l=not g2[1].is_l)
    golds[2] = g2
    engine = tagger._engine
    gold = engine.upload_paths([g[1:-1] for g in golds])
    engine.tag_packed(sents, 5)
    delta, differs, n_differ = engine.perceptron_delta(gold, 1)
    gold.close()
    desc_func, desc_fdic = engine.tables.desc_sources()
    got = np.zeros(len(encoder.feature_dic))
    np.add.at(got, desc_fdic[desc_func == 1], delta[desc_func == 1].astype(np.float64))
    want = np.zeros_like(got)
    want_differs = []
    for g, seq in zip(golds, predicted):
        d = seq is None or not _same_path(seq.sequences, g)
        want_differs.append(d)
        if d:
            for idxs in encoder.encode_sequence(g):
                np.add.at(want, idxs, 1.0)
            if seq is not None:
                for idxs in encoder.encode_sequence(seq.sequences):
                    np.add.at(want, idxs, -1.0)
    assert differs.tolist() == want_differs
    assert want_differs[1] is False and want_differs[2] is False and want_differs[5] is True
    assert n_differ == sum(want_differs)
    assert got.tolist() == want.tolist()


def test_train_epoch_matches_reference_epoch():
    tagger, encoder, scorer, reg, dictionary = _toy_tagger()
    ref_tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder)))
    coef_dev = coef_ref = np.zeros(len(encoder.feature_dic))
    for epoch in range(1, 6):
        coef_dev, loss_dev = train_epoch(PAIRS, encoder, tagger, coef_dev, epoch, False)
        coef_ref, loss_ref = _reference_epoch(PAIRS, encoder, ref_tagger, coef_ref)
        assert loss_dev == loss_ref
        assert coef_dev.tolist() == coef_ref.tolist()


def _reference_train(pairs, dictionary, max_epochs):
    """train() as it was with the host epoch: tables without extra tags, host counting."""
    from lattice_based_tagger_b200.features.utils import scan_features
    encoder = pkg.features.SimpleTrigramEncoder()
    reg = pkg.beam.RegularizationScore(unknown_penalty=-0.1, known_preference=-0.3, syllable_penalty=0.0)
    idx_to_feature, feature_to_idx, _ = scan_features(pairs, encoder, min_count=1,
                                                      predefined_features={(6, n): 1 for n in range(1, 9)})
    encoder.feature_dic = feature_to_idx
    scorer = pkg.beam.SimpleTrigramFeatureScore().set_encoder(encoder)
    tagger = pkg.Tagger(dictionary, encoder=encoder, score_funcs=pkg.beam.BeamScoreFunctions(reg, scorer))
    coef = np.zeros(len(feature_to_idx))
    best_loss, best_coef, stale = None, coef, 0
    for epoch in range(1, max_epochs + 1):
        decoded_with = coef
        coef, loss = _reference_epoch(pairs, encoder, tagger, coef)
        if best_loss is None or loss < best_loss:
            best_loss, best_coef, stale = loss, decoded_with, 0
        else:
            stale += 1
        if loss == 0 or stale >= 5:
            break
    tagger.close()
    return {'idx_to_feature': idx_to_feature, 'coefficient': [float(c) for c in best_coef]}


@pytest.mark.parametrize('max_epochs', [1, 2, 5])
def test_train_returns_the_same_parameters(max_epochs):
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    reg = pkg.beam.RegularizationScore(unknown_penalty=-0.1, known_preference=-0.3, syllable_penalty=0.0)
    got = train(PAIRS, dictionary, pkg.features.SimpleTrigramEncoder(), pkg.beam.SimpleTrigramFeatureScore(), reg,
                max_epochs=max_epochs)
    assert got == _reference_train(PAIRS, dictionary, max_epochs)


def test_fit_parameter_on_a_flatten_tagger_uses_the_host_loop():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    tagger, encoder, scorer, reg, _ = _toy_tagger()
    flat = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder)),
                      lookup=pkg.dictionary.lookup.MorphemeLookup(dictionary, flatten=True))
    coef = fit_parameter(PAIRS[:3], encoder, flat, max_epochs=2)
    assert len(coef) == len(encoder.feature_dic)


# ---- malformed input ---------------------------------------------------------------------------------

def test_malformed_paths_raise():
    tagger, encoder, scorer, reg, _ = _toy_tagger()
    good = text_to_words(*PAIRS[0])
    for bad in (['not a path'], [good[1:]], [good[:-1]], [42], [[BOS, 'x', _eos(0)]],
                [[BOS, good[1]._replace(tag0='NoSuchTag'), _eos(6)]],
                [[BOS, good[1]._replace(word='\U0001F600'), _eos(6)]],
                [[BOS, good[1]._replace(len=70000), _eos(6)]]):
        with pytest.raises(ValueError):
            tagger.score_paths(bad)
    with pytest.raises(ValueError):
        tagger.encode_paths([good], scorer=pkg.beam.SimpleTrigramFeatureScore(encoder))
    reg_only = pkg.Tagger(pkg.dictionary.DemoMorphemeDictionary(), score_funcs=pkg.beam.BeamScoreFunctions(reg))
    with pytest.raises(ValueError):
        reg_only.encode_paths([good])


def test_c_abi_rejects_malformed_path_sets():
    tagger, encoder, scorer, reg, _ = _toy_tagger()
    lib, tables, batch = tagger._lib, tagger._tables.handle, tagger._batch
    engine = tagger._engine
    words = text_to_words(*PAIRS[0])[1:-1]
    edges, units, str_off, n_str = engine.pack_words(words)
    off = np.array([0, len(words)], dtype=np.int64)
    out = ctypes.c_void_p()

    def create(edges=edges, off=off, n_paths=1, n_str=n_str):
        return lib.lt_pathset_create(tables, n_paths, _native.ptr(edges), _native.ptr(off), _native.ptr(units),
                                     _native.ptr(str_off), n_str, ctypes.byref(out))

    invalid = 1
    assert create(off=np.array([0, 3, 2], dtype=np.int64), n_paths=2) == invalid
    assert create(off=np.array([1, len(words)], dtype=np.int64)) == invalid
    assert create(n_str=n_str - 3) == invalid
    assert create(n_str=n_str - 1) == invalid
    for field, value in (('tag0', 40), ('tag1', 40), ('flags', 0), ('rule', 99)):
        bad = edges.copy()
        bad[0][field] = value
        assert create(edges=bad) == invalid, field
    assert lib.lt_pathset_create(None, 1, _native.ptr(edges), _native.ptr(off), _native.ptr(units), _native.ptr(str_off),
                                 n_str, ctypes.byref(out)) == invalid
    assert create() == 0
    paths = out
    scores = np.zeros(1)
    feat_off = np.zeros(len(words) + 1, dtype=np.int64)
    feat_idx = np.zeros(9 * len(words), dtype=np.int32)
    assert lib.lt_pathset_eval(batch, paths, 0, _native.ptr(scores), _native.ptr(feat_off), _native.ptr(feat_idx), feat_idx.size) == invalid
    assert lib.lt_pathset_eval(batch, paths, 7, _native.ptr(scores), _native.ptr(feat_off), _native.ptr(feat_idx), feat_idx.size) == invalid
    assert lib.lt_pathset_eval(batch, paths, 1, _native.ptr(scores), _native.ptr(feat_off), _native.ptr(feat_idx), 0) == 3
    assert lib.lt_pathset_eval(batch, paths, 1, _native.ptr(scores), _native.ptr(feat_off), _native.ptr(feat_idx), feat_idx.size) == 0
    delta = np.zeros(max(1, engine.tables.n_desc), dtype=np.int64)
    differs = np.zeros(2, dtype=np.uint8)
    nd = ctypes.c_int64()
    engine.tag_packed([_surface(PAIRS[0][0]), _surface(PAIRS[1][0])], 5)     # two sentences, one gold path
    assert lib.lt_perceptron_delta(batch, paths, 1, _native.ptr(delta), engine.tables.n_desc, _native.ptr(differs), ctypes.byref(nd)) == invalid
    engine.tag_packed([_surface(PAIRS[0][0])], 5)
    assert lib.lt_perceptron_delta(batch, paths, 1, _native.ptr(delta), engine.tables.n_desc + 1, _native.ptr(differs), ctypes.byref(nd)) == invalid
    assert lib.lt_perceptron_delta(batch, paths, 0, _native.ptr(delta), engine.tables.n_desc, _native.ptr(differs), ctypes.byref(nd)) == invalid
    assert lib.lt_perceptron_delta(batch, paths, 1, _native.ptr(delta), engine.tables.n_desc, _native.ptr(differs), ctypes.byref(nd)) == 0
    assert nd.value == int(differs[0])
    lib.lt_pathset_destroy(paths)
