"""Early and max-violation perceptron updates on the device (lt_trainer_set_update, `DeviceTrainer(update=...)`,
`fit_parameter(update=...)`) against a host reference that does not share the device's inductive rank sets: per
mini-batch it decodes with `tag_packed`, reruns the oracle's beam search (oracle/lattice_oracle.py:beam_search)
keeping every end position's survivors on the slice's `lattice_batch` lattices, decides "gold prefix in the beam"
by comparing whole hypotheses with the gold prefix, takes B from the survivors' scores and G from
`ScoreProgram.increment`, and counts features with `encode_sequence` on the two prefixes.  Weights, averaged weights,
steps, mistakes, differs flags, prefix words and violations are compared with `==` after every epoch."""

import ctypes
import math

import numpy as np
import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native
from lattice_based_tagger_b200.dictionary import Word
from lattice_based_tagger_b200.dictionary.text import text_to_words
from lattice_based_tagger_b200.trainer.train import _same_path, _surface, fit_parameter, train
from oracle import lattice_oracle as lo
from tests.test_gpu_minibatch_train import REG, HostLoop, _feat_coef, _pair, _toy, c2_annotated  # noqa: F401
from tests.test_gpu_paths import BOS, PAIRS, _eos

pytestmark = pytest.mark.gpu

MODES = ('early', 'max_violation')
NAN = float('nan')


def _key(w):
    return (w[lo.B], w[lo.E], w[lo.MORPH0], w[lo.MORPH1], w[lo.TAG0], w[lo.TAG1])


def position_beams(bindex, chars, program, beam_size):
    """The oracle's `beam_search` loop, returning the survivors of every end position (beams[e], best first)."""
    length = len(chars)
    bos = (lo.BOS, lo.BOS, None, lo.BOS, None, 0, 0, 0, False)
    beams = [[lo.Hypothesis([bos], 0)]]
    for e in range(1, length + 1):
        grown = []
        b_min = max(0, e - lo.WINDOW)
        for b in range(b_min, e):
            expansions = [edge for edge in bindex[b] if edge[lo.E] == e]
            if not expansions:
                sub = chars[b:e]
                expansions = [(sub, sub, None, lo.UNK, None, e - b, b, e, False)]
            for hyp in beams[b]:
                for edge in expansions:
                    if hyp.num_unk > 0 and edge[lo.TAG0] == lo.UNK and b_min < b:
                        continue
                    word_i = None if len(hyp.words) == 1 else hyp.words[-2]
                    grown.append(hyp.extended(edge, program.increment(word_i, hyp.words[-1], edge)))
        beams.append(sorted(grown, key=lambda h: -h.score)[:beam_size])
    return beams


def _tiles(words, length):
    end = 0
    for w in words:
        if w.b != end or w.e <= w.b:
            return False
        end = w.e
    return bool(words) and end == length


class ViolationRef(HostLoop):
    """HostLoop with the update on the prefix m* the mode picks."""

    def __init__(self, tagger, func, coef, n_sent, mode):
        super().__init__(tagger, func, coef, n_sent)
        self.mode = mode
        self.prefix = [0] * n_sent
        self.violation = [NAN] * n_sent
        self.search_errors = []         # (G_W, B_W, m*, violation) of the sentences whose gold outscores the best path
        self.shared = 0                 # boundaries where more than one kept hypothesis equals the gold prefix

    def step(self, sents, golds, first, count, beam):
        self.t += 1
        self.load(self.coef)
        engine = self.tagger._engine
        sl = sents[first:first + count]
        self.last = engine.tag_packed(sl, beam)
        predicted = engine.unpack(sl, self.last, 'none')
        program = lo.ScoreProgram(self.tagger.score_funcs)
        encoder = self.scorer.encoder
        update = np.zeros(len(self.coef))

        def add(words, sign):       # words [BOS, w_1 .. w_n, <ignored>]
            for idxs in encoder.encode_sequence(words):
                np.add.at(update, idxs, sign)
        ok = [i for i, seq in enumerate(predicted) if seq is not None]
        distinct = sorted({sl[i] for i in ok})
        lattices = dict(zip(distinct, self.tagger.lattice_batch(distinct)))
        differs, cache = [], {}        # (the survivors of a sentence repeated in the slice are computed once)
        for i, seq in enumerate(predicted):
            s, gold = first + i, golds[first + i]
            d = seq is None or not _same_path(seq.sequences, gold)
            differs.append(d)
            words = gold[1:-1]
            self.prefix[s], self.violation[s] = (len(words) if d else 0), NAN
            if not d:
                continue
            chars = sl[i].replace(' ', '')
            if seq is None or not _tiles(words, len(chars)):
                add(gold, 1.0)
                if seq is not None:
                    add(seq.sequences, -1.0)
                continue
            if sl[i] not in cache:
                cache[sl[i]] = position_beams(lattices[sl[i]][1], chars, program, beam)
            beams = cache[sl[i]]
            best = beams[len(chars)][0]
            assert [tuple(w) for w in best.words] + [tuple(seq.sequences[-1])] == [tuple(w) for w in seq.sequences]
            assert best.score == seq.score
            G, score, path = [0], 0, [tuple(w) for w in gold]
            for m in range(1, len(words) + 1):
                score = score + program.increment(None if m == 1 else path[m - 2], path[m - 1], path[m])
                G.append(score)
            in_beam = [None] + [[r for r, h in enumerate(beams[words[m - 1].e])
                                 if [_key(w) for w in h.words[1:]] == [_key(w) for w in words[:m]]]
                                for m in range(1, len(words) + 1)]
            self.shared += sum(len(r) > 1 for r in in_beam[1:])
            W = len(words)
            if self.mode == 'early':
                mstar = next((m for m in range(1, W + 1) if not in_beam[m]), W)
            else:
                mstar = max((beams[words[m - 1].e][0].score - G[m], m) for m in range(1, W + 1) if 0 not in in_beam[m])[1]
            hyp = beams[words[mstar - 1].e][0]
            self.prefix[s], self.violation[s] = mstar, hyp.score - G[mstar]
            if G[W] > best.score:
                self.search_errors.append((G[W], best.score, mstar, self.violation[s]))
            add([BOS] + words[:mstar] + [None], 1.0)
            add([Word(*w) for w in hyp.words] + [None], -1.0)
        self.differs[first:first + count] = differs
        self.mistakes += sum(differs)
        self.coef = self.coef + update
        self.u = self.u + (self.t - 1) * update


def _check_same(trainer, host):
    got, want = trainer.fetch(), host.state()
    assert got[0].tolist() == want[0].tolist()
    assert got[1].tolist() == want[1].tolist()
    assert got[2:4] == want[2:4]
    assert got[4].tolist() == want[4]
    prefix, violation = trainer.update_info()
    assert prefix.tolist() == host.prefix
    assert np.array_equal(violation, np.array(host.violation), equal_nan=True)


def train_modes(dev, ref, func, sents, golds, coef, batch, epochs, mode, beam=5):
    """Epochs of consecutive mini-batches in `mode` on the device and in ViolationRef, compared after every epoch."""
    engine = dev._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    trainer = engine.trainer(sents, pathset, func, len(coef), _feat_coef(engine, func), coef, update=mode)
    host = ViolationRef(ref, func, coef, len(sents), mode)
    n = len(sents)
    batch = batch or n
    try:
        for _ in range(epochs):
            for first in range(0, n, batch):
                count = min(batch, n - first)
                trainer.step(first, count, beam)
                host.step(sents, golds, first, count, beam)
            _check_same(trainer, host)
    finally:
        trainer.close()
        pathset.close()
    return host


def _toy_funcs(feature_dic, coef):
    def funcs():
        return pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    return funcs


def _noun(text, b):
    return Word(text, text, None, 'Noun', None, len(text), b, b + len(text), False)


def _unk(text, b):
    return Word(text, text, None, 'Unknown', None, len(text), b, b + len(text), False)


def _unreachable():
    """Sentences whose gold path lt_evaluate reports unreachable, one per reason."""
    nine = '가나다라마바사아자'
    return [
        ('노래 노래', [BOS, _noun('노래', 0), Word('노래', '노래', None, 'Josa', None, 2, 2, 4, False), _eos(4)]),  # not in the lattice
        (nine + ' 노래', [BOS, _noun(nine, 0), _noun('노래', 9), _eos(11)]),                                    # beyond the window
        ('뷁뷁뷁 노래', [BOS, _unk('뷁', 0), _unk('뷁뷁', 1), _noun('노래', 3), _eos(5)]),                         # unknown after unknown
        ('노래 아이', [BOS, _noun('노래', 0), _noun('이', 3), _eos(4)]),                                         # breaks the tiling
    ]


def _corpus():
    dictionary, sents, golds, feature_dic, coef = _toy()
    for i, (s, g) in enumerate(_unreachable()):
        sents.insert(3 + 4 * i, s)
        golds.insert(3 + 4 * i, g)
    return dictionary, sents, golds, feature_dic, coef


# ---- the toy corpus, every batch size, both modes ---------------------------------------------------------------

@pytest.mark.parametrize('batch', [1, 7, 64, None])
@pytest.mark.parametrize('mode', MODES)
def test_toy_corpus_against_host_reference(mode, batch):
    dictionary, sents, golds, feature_dic, coef = _corpus()
    dev, ref = _pair(dictionary, _toy_funcs(feature_dic, coef))
    host = train_modes(dev, ref, 1, sents, golds, coef, batch, 3, mode)
    assert host.mistakes > 0
    assert any(0 < p < len(g) - 2 for p, g in zip(host.prefix, golds))          # some update on a proper prefix
    gap = [i for i, g in enumerate(golds) if any(w.b != v.e for v, w in zip(g[1:-2], g[2:-1]))]
    assert gap and all(host.prefix[i] == len(golds[i]) - 2 and math.isnan(host.violation[i]) for i in gap)


def test_unreachable_gold_paths_are_the_intended_ones():
    dictionary, _, _, feature_dic, coef = _toy()
    tagger = pkg.Tagger(dictionary, score_funcs=_toy_funcs(feature_dic, coef)(), extra_tags=['Suffix'])
    engine = tagger._engine
    cases = _unreachable()
    engine.tag_packed([s for s, _ in cases], 5)
    pathset = engine.upload_paths([g[1:-1] for _, g in cases])
    try:
        sent_class, _, _, reason = engine.evaluate(pathset)
    finally:
        pathset.close()
    assert set(sent_class.tolist()) == {_native.LT_EVAL_UNREACHABLE}
    assert {_native.LT_GOLD_NOT_IN_LATTICE, _native.LT_GOLD_BEYOND_WINDOW, _native.LT_GOLD_UNK_AFTER_UNK,
            _native.LT_GOLD_BREAKS_TILING} <= set(reason.tolist())


@pytest.mark.parametrize('beam', [1, 64])
@pytest.mark.parametrize('mode', MODES)
def test_beam_1_and_64(mode, beam):
    dictionary, sents, golds, feature_dic, coef = _corpus()
    dev, ref = _pair(dictionary, _toy_funcs(feature_dic, coef))
    train_modes(dev, ref, 1, sents, golds, coef, 7, 2, mode, beam=beam)


@pytest.mark.parametrize('mode', MODES)
def test_c2_sample_against_host_reference(c2_annotated, mode):  # noqa: F811
    beam, dictionary, feature_dic, sents, golds = c2_annotated
    coef = np.zeros(len(feature_dic))

    def funcs():
        return pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(),
                                           pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    dev, ref = pkg.Tagger(dictionary, score_funcs=funcs()), pkg.Tagger(dictionary, score_funcs=funcs())
    host = train_modes(dev, ref, 1, sents, golds, coef, 64, 2, mode, beam=beam)
    assert host.mistakes > 0


# ---- long gold paths, the grid stride, reruns, stale back-pointers ------------------------------------------------

def _long_corpus(tagger, edits=(31, 32, 33, 63, 64)):
    """70-word sentences; gold = the tagger's own best path with word k given another tag."""
    sents = [' '.join(['노래', '아이'] * 35), ' '.join(['아이', '노래', '는'] * 24)]
    base = [list(seq.sequences) for seq in tagger.tag_batch(sents, 5)]
    out_s, out_g = [], []
    for n, k in enumerate(edits):
        g = list(base[n % 2])
        assert len(g) - 2 > 64
        w = g[k + 1]
        g[k + 1] = w._replace(tag0='Verb' if w.tag0 != 'Verb' else 'Noun')
        out_s.append(sents[n % 2])
        out_g.append(g)
    return out_s, out_g


def _duplicate_dictionary():
    """The demo dictionary with a second rule for the one-syllable key '했'.  The lattice emits each analysis of a
    one-syllable key once per rule of the key (R x R, as the reference does), so '했다' holds 하/Verb+았다/Eomi twice:
    two equal edges in one bucket, with equal scores."""
    demo = pkg.dictionary.DemoMorphemeDictionary()
    tag_to_morphs = {t: set(m) for t, m in demo.tag_to_morphs.items()}
    tag_to_morphs['Eomi'] |= {'였다'}
    rules = dict(demo.rules)
    rules['했'] = (('하', '았'), ('하', '였'))
    return pkg.dictionary.MorphemeDictionary(tag_to_morphs, rules)


DUPLICATE_PAIRS = [
    ('노래 를  했다', '노래/Noun 를/Josa  하/Verb+았다/Eomi'),
    ('아이 는  노래 를  했다', '아이/Noun 는/Josa  노래/Noun 를/Josa  하/Verb+았다/Eomi'),
    ('했다  노래', '하/Verb+았다/Eomi  노래/Noun'),
    ('노래 를  했다  아이 는  노래', '노래/Noun 를/Josa  하/Verb+았다/Eomi  아이/Noun 는/Josa  노래/Noun'),
    ('했다  아이 는', '하/Verb+았다/Eomi  아이/Josa 는/Noun'),                     # wrong tags after the duplicate
    ('아이 는  했다  노래 를', '아이/Noun 는/Josa  하/Verb+였다/Eomi  노래/Josa 를/Noun'),
]


@pytest.mark.parametrize('beam', [3, 5])
@pytest.mark.parametrize('mode', MODES)
def test_equal_duplicate_edges_both_in_the_beam(mode, beam):
    """A gold word with two equal edges in its bucket, both kept: the rank set follows either copy."""
    dictionary = _duplicate_dictionary()
    golds = [text_to_words(w, m) for w, m in DUPLICATE_PAIRS]
    sents = [_surface(w) for w, _ in DUPLICATE_PAIRS] * 3
    golds = golds * 3
    keys = sorted({k for g in golds for idxs in pkg.features.SimpleTrigramEncoder().transform_sequence(g) for k in idxs}, key=repr)
    feature_dic = {k: i for i, k in enumerate(keys)}
    coef = np.random.default_rng(4).choice([-1.0, 0.0, 1.0, 2.0], size=len(keys))
    dev, ref = _pair(dictionary, _toy_funcs(feature_dic, coef))
    words, _ = ref.lattice_batch(['했다'])[0]
    assert sum(tuple(w)[1:5] == ('하', '았다', 'Verb', 'Eomi') for w in words) == 2
    host = train_modes(dev, ref, 1, sents, golds, coef, 4, 3, mode, beam=beam)
    assert host.shared > 0 and host.mistakes > 0


@pytest.mark.parametrize('mode', MODES)
def test_gold_paths_of_more_than_64_words(mode):
    dictionary, sents, golds, feature_dic, coef = _toy(extra_sents=False)
    dev, ref = _pair(dictionary, _toy_funcs(feature_dic, coef))
    long_s, long_g = _long_corpus(ref)
    host = train_modes(dev, ref, 1, long_s + sents, long_g + golds, coef, 3, 2, mode)
    assert any(p > 32 for p in host.prefix)


@pytest.mark.parametrize('mode', MODES)
def test_short_step_after_long_step(mode):
    """Step 1 fills the trail far into the buffer, step 2's shorter sentences leave most of it: stale entries must
    not read as survivors."""
    dictionary, sents, golds, feature_dic, coef = _toy(extra_sents=False)
    dev, ref = _pair(dictionary, _toy_funcs(feature_dic, coef))
    long_s, long_g = _long_corpus(ref)
    unk = [('뷁뷁 노래 아이', [BOS, _unk('뷁뷁', 0), _noun('노래', 2), _noun('아이', 4), _eos(6)]),
           ('노래 뷁 아이', [BOS, _noun('노래', 0), _unk('뷁', 2), _noun('아이', 3), _eos(5)])]
    short_s = [s for s, _ in unk] + sents
    short_g = [g for _, g in unk] + golds
    train_modes(dev, ref, 1, long_s + short_s, long_g + short_g, coef, len(long_s), 3, mode, beam=64)


@pytest.mark.parametrize('mode', MODES)
def test_forced_rerun_inside_a_step(monkeypatch, mode):
    dictionary, sents, golds, feature_dic, coef = _corpus()
    funcs = _toy_funcs(feature_dic, coef)
    ref = pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])
    monkeypatch.setenv('LT_EDGE_CAP', '16')
    dev = pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])
    monkeypatch.delenv('LT_EDGE_CAP')
    before = dev.info()['reruns']
    train_modes(dev, ref, 1, sents, golds, coef, 9, 2, mode)
    assert dev.info()['reruns'] > before


def test_more_sentences_in_a_step_than_the_launch_has_warps():
    dictionary, sents, golds, feature_dic, coef = _toy(extra_sents=False)
    dev, ref = _pair(dictionary, _toy_funcs(feature_dic, coef))
    n = 2 * dev.info()['sm_count'] * 64 + 7
    reps = -(-n // len(sents))
    sents, golds = (sents * reps)[:n], (golds * reps)[:n]
    train_modes(dev, ref, 1, sents, golds, coef, n - 3, 1, 'max_violation')


# ---- properties --------------------------------------------------------------------------------------------

def _trainers(engine, sents, golds, coef, modes):
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    return pathset, [engine.trainer(sents, pathset, 1, len(coef), _feat_coef(engine, 1), coef, update=m) for m in modes]


def test_full_through_set_update_is_the_default():
    dictionary, sents, golds, feature_dic, coef = _corpus()
    tagger = pkg.Tagger(dictionary, score_funcs=_toy_funcs(feature_dic, coef)(), extra_tags=['Suffix'])
    engine = tagger._engine
    pathset, (plain, switched) = _trainers(engine, sents, golds, coef, ['full', 'max_violation'])
    switched.set_update('full')
    results = []
    for trainer in (plain, switched):
        for first in range(0, len(sents), 7):
            trainer.step(first, min(7, len(sents) - first), 5)
        results.append((trainer.fetch(), trainer.update_info()))
        # the two trainers share the tables: the second starts again from w_0
        tagger.score_funcs.funcs[1].coefficients = coef
        tagger.update_weights()
    (a, ua), (b, ub) = results
    assert a[0].tolist() == b[0].tolist() and a[1].tolist() == b[1].tolist() and a[2:4] == b[2:4]
    assert a[4].tolist() == b[4].tolist()
    assert ua[0].tolist() == ub[0].tolist() and np.array_equal(ua[1], ub[1], equal_nan=True)
    words = [len(g) - 2 for g in golds]
    assert ua[0].tolist() == [w if d else 0 for w, d in zip(words, a[4])]
    assert np.isnan(ua[1]).all()
    for t in (plain, switched):
        t.close()
    pathset.close()


def test_first_step_decodes_alike_and_violations_hold(c2_annotated):  # noqa: F811
    """From the same w_0 the first step decodes identically in every mode; search errors are no violation at W and
    MAX_VIOLATION updates where there is one; every reachable gold path gets a violation >= 0."""
    beam, dictionary, feature_dic, sents, golds = c2_annotated
    coef = np.random.default_rng(11).normal(0.0, 1.0, len(feature_dic))        # c2_annotated's teacher weights (same draw)
    beam = 2

    def fresh():
        return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(
            pkg.beam.RegularizationScore(), pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef)))
    tagger = fresh()
    engine = tagger._engine
    engine.tag_packed(sents, beam)
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    sent_class, _, gold_scores, _ = engine.evaluate(pathset)
    scores = engine.tag_packed(sents, beam)[2]
    pathset.close()
    tagger.close()
    out = {}
    for mode in ('full',) + MODES:
        tagger = fresh()
        pathset, (trainer,) = _trainers(tagger._engine, sents, golds, coef, [mode])
        trainer.step(0, len(sents), beam)
        out[mode] = trainer.fetch(), trainer.update_info()
        trainer.close()
        pathset.close()
        tagger.close()
    full = out['full'][0]
    for mode in MODES:
        got = out[mode][0]
        assert got[3] == full[3] and got[4].tolist() == full[4].tolist()
    W = np.array([len(g) - 2 for g in golds])
    search = sent_class == _native.LT_EVAL_SEARCH_ERROR
    assert search.sum() > 0
    prefix, violation = out['max_violation'][1]
    assert (gold_scores[search] > scores[search]).all()
    assert (prefix[search] < W[search]).all() and (violation[search] >= 0).all()
    reachable = search | (sent_class == _native.LT_EVAL_MODEL_ERROR)
    for mode in MODES:
        assert (out[mode][1][1][reachable] >= 0).all()


def test_early_equals_full_where_gold_stays_in_the_beam():
    """One step over exactly the sentences whose gold prefix never left the beam (EARLY took all W words) or that
    need no update: EARLY and FULL give the same weights."""
    dictionary, sents, golds, feature_dic, coef = _corpus()
    funcs = _toy_funcs(feature_dic, coef)

    def step(mode, sl, gl):
        tagger = pkg.Tagger(dictionary, score_funcs=funcs(), extra_tags=['Suffix'])
        pathset, (trainer,) = _trainers(tagger._engine, sl, gl, coef, [mode])
        trainer.step(0, len(sl), 5)
        out = trainer.fetch()[0], trainer.update_info()
        trainer.close()
        pathset.close()
        tagger.close()
        return out
    _, (prefix, violation) = step('early', sents, golds)
    W = [len(g) - 2 for g in golds]
    keep = [i for i in range(len(sents)) if prefix[i] in (0, W[i])]
    assert len(keep) < len(sents)
    assert any(prefix[i] == W[i] and not math.isnan(violation[i]) for i in keep)      # a full update read from the trail
    sub_s, sub_g = [sents[i] for i in keep], [golds[i] for i in keep]
    w_full, w_early = step('full', sub_s, sub_g)[0], step('early', sub_s, sub_g)[0]
    assert w_full.tolist() == w_early.tolist() and w_full.tolist() != coef.tolist()


# ---- Python and C ABI -----------------------------------------------------------------------------------------

def test_fit_parameter_and_train_take_update():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    _, _, _, feature_dic, _ = _toy(extra_sents=False)
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)

    def tagger(**kw):
        return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder)),
                          extra_tags=['Suffix'], **kw)
    pairs = PAIRS[:-1]
    sents = [_surface(w) for w, _ in pairs]
    golds = [text_to_words(w, m) for w, m in pairs]
    for mode in MODES:
        t = tagger()
        got = fit_parameter(pairs, encoder, t, max_epochs=1, batch_size=3, update=mode)
        ref = tagger()
        host = ViolationRef(ref, 1, np.zeros(len(feature_dic)), len(sents), mode)
        for first in range(0, len(sents), 3):
            host.step(sents, golds, first, min(3, len(sents) - first), 5)
        assert got.tolist() == host.coef.tolist()
    params = train(PAIRS, dictionary, pkg.features.SimpleTrigramEncoder(), pkg.beam.SimpleTrigramFeatureScore(), REG,
                               max_epochs=2, batch_size=2, update='max_violation')
    assert len(params['coefficient']) == len(params['idx_to_feature']) > 0
    t = tagger()
    with pytest.raises(ValueError, match='batch_size'):
        fit_parameter(pairs, encoder, t, max_epochs=1, update='early')
    with pytest.raises(ValueError, match='batch_size'):
        train(PAIRS, dictionary, pkg.features.SimpleTrigramEncoder(), pkg.beam.SimpleTrigramFeatureScore(), REG,
                          max_epochs=1, update='max_violation')
    for bad in ('Early', 'violation', None):
        with pytest.raises(ValueError):
            fit_parameter(pairs, encoder, t, max_epochs=1, batch_size=2, update=bad)
    flat = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(REG, pkg.beam.SimpleTrigramFeatureScore(encoder)),
                      lookup=pkg.dictionary.lookup.MorphemeLookup(dictionary, flatten=True))
    with pytest.raises(ValueError):
        fit_parameter(pairs[:3], encoder, flat, max_epochs=1, batch_size=2, update='early')
    engine = t._engine
    _, _, _, _, coef = _toy(extra_sents=False)
    pathset = engine.upload_paths([g[1:-1] for g in golds[:3]])
    with pytest.raises(ValueError):
        engine.trainer(sents[:3], pathset, 1, len(coef), _feat_coef(engine, 1), coef, update='nope')
    trainer = engine.trainer(sents[:3], pathset, 1, len(coef), _feat_coef(engine, 1), coef)
    with pytest.raises(ValueError):
        trainer.set_update('max-violation')
    lib = engine._lib
    for mode in (-1, 3, 100):
        assert lib.lt_trainer_set_update(trainer.handle, mode) == 1
    assert lib.lt_trainer_set_update(None, 1) == 1
    assert lib.lt_trainer_fetch_update(None, None, None) == 1
    for mode in range(3):
        assert lib.lt_trainer_set_update(trainer.handle, mode) == 0
    trainer.step(0, 3, 5)
    prefix = np.zeros(3, dtype=np.int32)
    assert lib.lt_trainer_fetch_update(trainer.handle, _native.ptr(prefix), None) == 0
    assert lib.lt_trainer_fetch_update(trainer.handle, None, ctypes.c_void_p()) == 0
    trainer.close()
    pathset.close()
