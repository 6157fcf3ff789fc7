"""Mini-batch perceptron training on the device (lt_trainer_*, `DeviceTrainer`, `fit_parameter(batch_size=...)`)
against a host loop that, per mini-batch, decodes with `tag_batch`, compares with `_same_path`, counts with
`encode_sequence`, applies coef += update and u += (t - 1) * update, and loads the weights with `update_weights`.
Weights, averaged weights, step and mistake counts and the per-sentence flags are compared with `==`."""

import ctypes

import numpy as np
import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native, synth
from lattice_based_tagger_b200.dictionary import Word
from lattice_based_tagger_b200.dictionary.text import text_to_words
from lattice_based_tagger_b200.trainer.train import _surface, fit_parameter, train, train_epoch
from tests.test_gpu_path_edges import host_delta
from tests.test_gpu_paths import BOS, PAIRS, _eos

pytestmark = pytest.mark.gpu

REG = pkg.beam.RegularizationScore(unknown_penalty=-0.1, known_preference=-0.3, syllable_penalty=0.0)


class HostLoop:
    """The definition the device trainer reproduces."""

    def __init__(self, tagger, func, coef, n_sent):
        self.tagger, self.scorer = tagger, tagger.score_funcs.funcs[func]
        self.coef = np.asarray(coef, dtype=np.float64).copy()
        self.u = np.zeros_like(self.coef)
        self.t = self.mistakes = 0
        self.differs = [False] * n_sent
        self.last = None

    def load(self, coef):
        self.scorer.coefficients = coef
        self.tagger.update_weights()

    def step(self, sents, golds, first, count, beam):
        self.t += 1
        self.load(self.coef)
        engine = self.tagger._engine
        sl = sents[first:first + count]
        self.last = engine.tag_packed(sl, beam)
        predicted = engine.unpack(sl, self.last, 'none')
        update, differs = host_delta(golds[first:first + count], predicted, self.scorer.encoder)
        update = np.concatenate([update, np.zeros(len(self.coef) - len(update))])
        self.differs[first:first + count] = differs
        self.mistakes += sum(differs)
        self.coef = self.coef + update
        self.u = self.u + (self.t - 1) * update

    def state(self):
        averaged = self.coef - self.u / self.t if self.t else self.coef
        return self.coef, averaged, self.t, self.mistakes, self.differs


def _feat_coef(engine, func):
    desc_func, desc_fdic = engine.tables.desc_sources()
    return np.where(desc_func == func, desc_fdic, -1)


def _train_both(dev, ref, func, sents, golds, coef, batch, epochs, beam=5, check=None):
    """Epochs of consecutive mini-batches on the device and on the host, compared after every epoch."""
    engine = dev._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    trainer = engine.trainer(sents, pathset, func, len(coef), _feat_coef(engine, func), coef)
    host = HostLoop(ref, func, coef, len(sents))
    n = len(sents)
    batch = batch or n
    try:
        for _ in range(epochs):
            for first in range(0, n, batch):
                count = min(batch, n - first)
                trainer.step(first, count, beam)
                host.step(sents, golds, first, count, beam)
                if check:
                    check(trainer, host, first, count)
            got = trainer.fetch()
            want = host.state()
            assert got[0].tolist() == want[0].tolist()
            assert got[1].tolist() == want[1].tolist()
            assert got[2:4] == want[2:4]
            assert got[4].tolist() == want[4]
    finally:
        trainer.close()
        pathset.close()
    return host


def _same_decode(dev, ref, host, sents, beam=5):
    """The tables the trainer left decode `sents` exactly as tables loaded with the host's weights."""
    host.load(host.coef)
    got = dev._engine.tag_packed(sents, beam)
    want = ref._engine.tag_packed(sents, beam)
    for a, b in zip(got, want):
        assert a.tolist() == b.tolist()


# ---- the toy corpus, with sentences the search cannot tag ----------------------------------------------------

def _toy(extra_sents=True):
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    pairs = [p for p in PAIRS if all(ord(c) < 0x10000 for c in p[0])]
    golds = [text_to_words(w, m) for w, m in pairs]
    sents = [_surface(w) for w, _ in pairs]
    if extra_sents:
        long_sent = '가' * 5000                                   # beyond lt_tables_max_sentence_units
        long_gold = [BOS] + [Word('가' * 8, '가' * 8, None, 'Noun', None, 8, b, b + 8, False) for b in range(0, 5000, 8)]
        long_gold[-1] = long_gold[-1]._replace(word='가' * 8, e=5000)
        extra = [('', [BOS, _eos(0)]), ('   ', [BOS, _eos(0)]), (long_sent, long_gold + [_eos(5000)]),
                 ('뷁뷁 노래', [BOS, Word('뷁뷁', '뷁뷁', None, 'Noun', None, 2, 0, 2, False),
                              Word('노래', '노래', None, 'Noun', None, 2, 2, 4, False), _eos(4)])]
        # mixed into the corpus so that mini-batches of every size hold some of them
        for i, (s, g) in enumerate(extra):
            sents.insert(2 + 5 * i, s)
            golds.insert(2 + 5 * i, g)
        sents, golds = sents * 2, golds * 2
    keys = set()
    for g in golds:
        if len(g) < 100:
            for idxs in pkg.features.SimpleTrigramEncoder().transform_sequence(g):
                keys.update(idxs)
    keys = sorted(keys, key=repr)
    feature_dic = {k: i for i, k in enumerate(keys)}
    coef = np.random.default_rng(0).choice([-1.0, 0.0, 1.0, 2.0], size=len(keys))
    return dictionary, sents, golds, feature_dic, coef


def _pair(dictionary, funcs, **kw):
    return pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'], **kw), \
        pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])


@pytest.mark.parametrize('batch', [1, 7, 64, None])
def test_toy_corpus_against_host_loop(batch):
    dictionary, sents, golds, feature_dic, coef = _toy()
    assert len(sents) % 7 != 0                                    # a short last mini-batch

    def funcs():
        return pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    dev, ref = _pair(dictionary, funcs)
    host = _train_both(dev, ref, 1, sents, golds, coef, batch, epochs=3)
    assert host.mistakes > 0 and 0 < host.t
    st = dev._engine.tag_packed(sents, 5)[3]
    assert {0, 1, 3} <= set(st.tolist())                          # tagged, no edge, too long
    _same_decode(dev, ref, host, [_surface(w) for w, _ in PAIRS[:5]] + ['노래 아이', '아이오아이 노래'])


def test_many_to_one_feature_dic():
    dictionary, sents, golds, feature_dic, coef = _toy()
    n = max(1, len(feature_dic) // 3)
    many = {k: i % n for k, i in feature_dic.items()}        # coefficients n .. len - 1 receive nothing

    def funcs():
        return pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(many), coef))
    dev, ref = _pair(dictionary, funcs)
    host = _train_both(dev, ref, 1, sents, golds, coef, 5, epochs=3)
    _same_decode(dev, ref, host, [_surface(w) for w, _ in PAIRS[:5]])


def test_second_trigram_scorer_trains_while_the_first_stays():
    """Scorers [trigram, preference, regulariser, trigram]: scorer 3 trains, scorer 0's weights stay."""
    dictionary, sents, golds, feature_dic, coef = _toy()
    fixed = np.random.default_rng(1).normal(0.0, 1.0, len(feature_dic))
    pref = {'Noun': {'노래': 0.5, '아이': -0.25}, 'Josa': {'는': 0.125}}

    def funcs():
        enc = pkg.features.SimpleTrigramEncoder(feature_dic)
        return pkg.beam.BeamScoreFunctions(pkg.beam.SimpleTrigramFeatureScore(enc, fixed), pkg.beam.MorphemePreferenceScore(pref), REG,
                                           pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    dev, ref = _pair(dictionary, funcs)
    host = _train_both(dev, ref, 3, sents, golds, coef, 5, epochs=3)
    assert host.mistakes > 0
    _same_decode(dev, ref, host, [_surface(w) for w, _ in PAIRS[:5]] + ['노래 는 아이'])


def test_forced_rerun_inside_a_step(monkeypatch):
    dictionary, sents, golds, feature_dic, coef = _toy()

    def funcs():
        return pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    ref = pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])
    monkeypatch.setenv('LT_EDGE_CAP', '16')
    dev = pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])
    monkeypatch.delenv('LT_EDGE_CAP')
    before = dev.info()['reruns']
    host = _train_both(dev, ref, 1, sents, golds, coef, 9, epochs=2)
    assert dev.info()['reruns'] > before
    _same_decode(dev, ref, host, [_surface(w) for w, _ in PAIRS[:5]])


def test_more_sentences_in_a_step_than_the_launch_has_warps():
    dictionary, sents, golds, feature_dic, coef = _toy(extra_sents=False)

    def funcs():
        return pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    dev, ref = _pair(dictionary, funcs)
    n = 2 * dev.info()['sm_count'] * 64 + 7
    reps = -(-n // len(sents))
    sents, golds = (sents * reps)[:n], (golds * reps)[:n]
    _train_both(dev, ref, 1, sents, golds, coef, n - 3, epochs=2)


def test_whole_corpus_step_is_train_epoch():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    pairs = [p for p in PAIRS if all(ord(c) < 0x10000 for c in p[0])]
    _, _, _, feature_dic, coef = _toy(extra_sents=False)
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)

    def tagger():
        return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder, coef)),
                          extra_tags=['Suffix'])
    want, loss = train_epoch(pairs, encoder, tagger(), coef, 1, False)
    dev = tagger()
    engine = dev._engine
    golds = [text_to_words(w, m)[1:-1] for w, m in pairs]
    pathset = engine.upload_paths(golds)
    trainer = engine.trainer([_surface(w) for w, _ in pairs], pathset, 1, len(coef), _feat_coef(engine, 1), coef)
    trainer.step(0, len(pairs), 5)
    got, averaged, steps, mistakes, _ = trainer.fetch()
    trainer.close()
    pathset.close()
    assert got.tolist() == want.tolist()
    assert averaged.tolist() == got.tolist() and steps == 1 and mistakes == loss > 0


# ---- the C2 teacher-student sample --------------------------------------------------------------------------

@pytest.fixture(scope='module')
def c2_annotated():
    """C2 sentences with the best paths of a teacher (the C2 features, other seeded weights) as gold, as
    profiles/tools/train_epoch.py builds them."""
    cfg, dictionary, sents = synth.build_workload('c2', n_sent=300)
    beam = cfg['beam']
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore()))
    ok = [s for s, st in zip(sents, probe.tag_batch_packed(sents, beam)[3]) if st == 0]
    feature_dic, _ = synth.make_features(ok, lambda s: probe.tag_batch(s, beam, errors='none'), probe.lattice_batch,
                                         cfg['n_feat'], list(dictionary.tag_to_morphs), seed=3)
    probe.close()
    other = np.random.default_rng(11).normal(0.0, 1.0, len(feature_dic))
    teacher = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(
        pkg.beam.RegularizationScore(), pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), other)))
    golds = [list(seq.sequences) if seq is not None else [BOS, _eos(0)] for seq in teacher.tag_batch(ok, beam, errors='none')]
    teacher.close()
    return beam, dictionary, feature_dic, ok, golds


@pytest.mark.parametrize('batch', [64, None])
@pytest.mark.parametrize('many_to_one', [False, True])
def test_c2_sample_against_host_loop(c2_annotated, batch, many_to_one):
    beam, dictionary, feature_dic, sents, golds = c2_annotated
    if many_to_one:
        n = max(1, len(feature_dic) // 3)
        feature_dic = {k: i % n for k, i in feature_dic.items()}
    coef = np.zeros(len(feature_dic))

    def funcs():
        return pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(),
                                           pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    dev, ref = pkg.Tagger(dictionary, score_funcs=funcs()), pkg.Tagger(dictionary, score_funcs=funcs())
    host = _train_both(dev, ref, 1, sents, golds, coef, batch, epochs=2, beam=beam)
    assert 0 < host.mistakes
    _same_decode(dev, ref, host, sents[:50], beam)


# ---- the batch and the tables after a step ------------------------------------------------------------------

def _fetch_paths(engine):
    lib, batch = engine._lib, engine.batch
    total = ctypes.c_int64()
    _native.check(lib.lt_paths_size(batch, ctypes.byref(total)))
    return total.value


def test_batch_holds_the_step_and_outlives_the_trainer():
    dictionary, sents, golds, feature_dic, coef = _toy()

    def funcs():
        return pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    dev, ref = _pair(dictionary, funcs)
    engine = dev._engine
    first, count = 5, 8
    sl_sents, sl_golds = sents[first:first + count], golds[first:first + count]
    results = {}

    def check(trainer, host, f, c):
        if f != first:
            return
        # lt_paths_fetch and lt_evaluate on the batch: the mini-batch, decoded with the weights before the step
        packed = _paths(engine, c)
        for a, b in zip(packed, host.last):
            assert a.tolist() == b.tolist()
        # lt_evaluate scores gold images with the tables as they are now (after the update): the same state on the host
        # is the host's decode of the slice (with the weights before) followed by loading the weights after
        host.load(host.coef)
        got, want = (_evaluate(e, sl_golds) for e in (engine, ref._engine))
        for a, b in zip(got, want):
            assert np.array_equal(a, b, equal_nan=True)
        assert sorted(set(got[0].tolist())) == [0, 1, 2]                # correct, failed and unreachable sentences
        results['packed'] = packed

    pathset = engine.upload_paths([g[1:-1] for g in golds])
    trainer = engine.trainer(sents, pathset, 1, len(coef), _feat_coef(engine, 1), coef)
    host = HostLoop(ref, 1, coef, len(sents))
    trainer.step(first, count, 5)
    host.step(sents, golds, first, count, 5)
    check(trainer, host, first, count)
    trainer.close()
    pathset.close()
    for a, b in zip(_paths(engine, count), results['packed']):
        assert a.tolist() == b.tolist()


def _evaluate(engine, golds):
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    try:
        return engine.evaluate(pathset)
    finally:
        pathset.close()


def _paths(engine, n):
    total = _fetch_paths(engine)
    path_off = np.zeros(n + 1, dtype=np.int32)
    edges = np.empty(max(1, total), dtype=_native.EDGE_DTYPE)
    scores = np.zeros(n, dtype=np.float64)
    status = np.zeros(n, dtype=np.int32)
    _native.check(engine._lib.lt_paths_fetch(engine.batch, _native.ptr(path_off), _native.ptr(edges), edges.size,
                                             _native.ptr(scores), _native.ptr(status)))
    return path_off, edges[:total], scores, status


def test_update_weights_after_steps_rewrites_the_dense_blocks():
    """The trainer writes dense weights on the device only; lt_tables_update_weights rewrites every weight that
    has a feature, so the tables then decode as freshly compiled ones."""
    dictionary, sents, golds, feature_dic, coef = _toy()
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
    dev = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder, coef)),
                     extra_tags=['Suffix'])
    engine = dev._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    trainer = engine.trainer(sents, pathset, 1, len(coef), _feat_coef(engine, 1), coef)
    for first in range(0, len(sents), 4):
        trainer.step(first, min(4, len(sents) - first), 5)
    trained = trainer.fetch()[0]
    trainer.close()
    pathset.close()
    assert not np.array_equal(trained, coef)
    other = np.random.default_rng(5).normal(0.0, 1.0, len(coef))
    dev.score_funcs.funcs[1].coefficients = other
    dev.update_weights()
    fresh = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder, other)),
                       extra_tags=['Suffix'])
    probe = [_surface(w) for w, _ in PAIRS[:5]] + sents[:12]
    for a, b in zip(dev._engine.tag_packed(probe, 5), fresh._engine.tag_packed(probe, 5)):
        assert a.tolist() == b.tolist()


# ---- Python: fit_parameter / train with batch_size ---------------------------------------------------------

def _host_fit(pairs, dictionary, feature_dic, batch, max_epochs, averaged, patience=5):
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
    ref = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder)),
                     extra_tags=['Suffix'])
    golds = [text_to_words(w, m) for w, m in pairs]
    sents = [_surface(w) for w, _ in pairs]
    host = HostLoop(ref, 1, np.zeros(len(feature_dic)), len(sents))
    best, stale, seen = None, 0, 0
    for _ in range(max_epochs):
        for first in range(0, len(sents), batch):
            host.step(sents, golds, first, min(batch, len(sents) - first), 5)
        loss, seen = host.mistakes - seen, host.mistakes
        if best is None or loss < best:
            best, stale = loss, 0
        else:
            stale += 1
        if loss == 0 or stale >= patience:
            break
    coef, mean = host.state()[:2]
    return (mean if averaged else coef), host.t


@pytest.mark.parametrize('averaged', [False, True])
def test_fit_parameter_with_batch_size(averaged):
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    _, _, _, feature_dic, _ = _toy(extra_sents=False)
    pairs = list(PAIRS)                                          # the last pair is outside the BMP: left out
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder)),
                        extra_tags=['Suffix'])
    got = fit_parameter(pairs, encoder, tagger, max_epochs=4, batch_size=3, averaged=averaged)
    want, steps = _host_fit(pairs[:-1], dictionary, feature_dic, 3, 4, averaged)
    assert steps > 3
    assert got.tolist() == want.tolist()
    scorer = tagger.score_funcs.funcs[1]
    assert np.asarray(scorer.coefficients).tolist() == want.tolist()
    probe = [_surface(w) for w, _ in PAIRS[:7]]
    fresh = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder, want)),
                       extra_tags=['Suffix'])
    for a, b in zip(tagger._engine.tag_packed(probe, 5), fresh._engine.tag_packed(probe, 5)):
        assert a.tolist() == b.tolist()


def test_train_with_batch_size_and_errors():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    params = train(PAIRS, dictionary, pkg.features.SimpleTrigramEncoder(), pkg.beam.SimpleTrigramFeatureScore(), REG,
                   max_epochs=3, batch_size=2, averaged=True)
    assert len(params['coefficient']) == len(params['idx_to_feature']) > 0
    _, _, _, feature_dic, coef = _toy(extra_sents=False)
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
    funcs = pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder))
    flat = pkg.Tagger(dictionary, score_funcs=funcs, lookup=pkg.dictionary.lookup.MorphemeLookup(dictionary, flatten=True))
    with pytest.raises(ValueError):
        fit_parameter(PAIRS[:3], encoder, flat, max_epochs=1, batch_size=2)
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder)))
    for bad in (0, -1, 1.5):
        with pytest.raises(ValueError):
            fit_parameter(PAIRS[:3], encoder, tagger, max_epochs=1, batch_size=bad)
    engine = tagger._engine
    golds = [text_to_words(w, m)[1:-1] for w, m in PAIRS[:3]]
    pathset = engine.upload_paths(golds)
    sents = [_surface(w) for w, _ in PAIRS[:3]]
    with pytest.raises(ValueError):
        engine.trainer(sents, pathset, 1, len(coef), _feat_coef(engine, 1), coef[:-1])
    with pytest.raises(ValueError):
        engine.trainer(sents, pathset, 1, len(coef), _feat_coef(engine, 1)[:-1], coef)
    trainer = engine.trainer(sents, pathset, 1, len(coef), _feat_coef(engine, 1), coef)
    for first, count, beam in ((0, 0, 5), (2, 2, 5), (-1, 1, 5), (0, 1, 0), (0, 1, 65)):
        with pytest.raises(_native.NativeLibraryError):
            trainer.step(first, count, beam)
    trainer.close()
    pathset.close()


# ---- C ABI errors ---------------------------------------------------------------------------------------------

def test_c_abi_rejects_invalid_trainers():
    dictionary, sents, golds, feature_dic, coef = _toy(extra_sents=False)

    def funcs():
        enc = pkg.features.SimpleTrigramEncoder(feature_dic)
        return pkg.beam.BeamScoreFunctions(pkg.beam.SimpleTrigramFeatureScore(enc, coef), REG,
                                           pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    tagger = pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])
    other = pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])
    engine, lib = tagger._engine, tagger._engine._lib
    text, offsets = pkg.engine.pack_sentences(sents)
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    foreign = other._engine.upload_paths([g[1:-1] for g in golds])
    short = engine.upload_paths([g[1:-1] for g in golds[:-1]])
    fc = _feat_coef(engine, 2)
    n = len(sents)
    out = ctypes.c_void_p()
    invalid = 1

    def create(func=2, offsets=offsets, gold=pathset, fc=fc, n_coef=len(coef)):
        return lib.lt_trainer_create(engine.tables.handle, func, _native.ptr(text), _native.ptr(offsets), n, gold.handle, n_coef,
                                     _native.ptr(fc), _native.ptr(coef), ctypes.byref(out))
    assert create(func=1) == invalid                               # the regulariser
    assert create(func=5) == invalid
    assert create(gold=foreign) == invalid
    assert create(gold=short) == invalid
    assert create(offsets=offsets + 1) == invalid                  # sent_off[0] != 0
    dec = offsets.copy()
    dec[3] = dec[2] - 1
    assert create(offsets=dec) == invalid
    for bad_value in (-2, len(coef)):
        bad = fc.copy()
        bad[np.flatnonzero(fc >= 0)[0]] = bad_value
        assert create(fc=bad) == invalid
    bad = fc.copy()
    bad[np.flatnonzero(fc < 0)[0]] = 0                            # a feature of scorer 0
    assert create(fc=bad) == invalid
    assert 'scorer' in lib.lt_last_error().decode()
    assert create() == 0
    trainer = out
    for first, count, beam in ((0, 0, 5), (0, -1, 5), (n - 1, 2, 5), (-1, 2, 5), (0, 1, 0), (0, 1, 65)):
        assert lib.lt_trainer_step(trainer, engine.batch, first, count, beam) == invalid, (first, count, beam)
    assert lib.lt_trainer_step(trainer, other._engine.batch, 0, 1, 5) == invalid
    assert lib.lt_trainer_step(trainer, engine.batch, n - 1, 1, 64) == 0
    steps = ctypes.c_int64()
    assert lib.lt_trainer_fetch(trainer, None, None, ctypes.byref(steps), None, None) == 0
    assert steps.value == 1
    lib.lt_trainer_destroy(trainer)
    for p in (pathset, foreign, short):
        p.close()
