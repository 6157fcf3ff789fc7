"""GPU parity: the CUDA path (through the C ABI) against the oracle and the golden fixtures."""

import pytest

import lattice_based_tagger_b200 as pkg
from oracle import lattice_oracle as lo
from tests import _cases, _checks, _golden

pytestmark = pytest.mark.gpu


def _lattice_key(edges):
    """reference order -> the order the device emits: stable by (end, begin)"""
    return sorted(edges, key=lambda w: (w[7], w[6]))


@pytest.mark.parametrize('name', _golden.names())
def test_golden_fixtures(name):
    payload = _golden.load(name)
    case = payload['case']
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs, k3_first=payload['k3_first'])
    sents = case['sentences']
    # lattice
    for sent, entry, (words, bindex) in zip(sents, payload['expected'], tagger.lattice_batch(sents)):
        want = _lattice_key([_golden.edge(w) for w in entry['lattice']])
        assert [tuple(w) for w in words[1:-1]] == want, sent
    # best path for every recorded beam size
    beams = sorted({int(k) for entry in payload['expected'] for k in entry['beams']})
    for k in beams:
        got = tagger.tag_batch(sents, beam_size=k, errors='none')
        for sent, entry, seq in zip(sents, payload['expected'], got):
            want = _golden.expected_survivors(entry, k)
            if want is None:
                assert seq is None, sent
                continue
            words, score, num_unk = want[0]
            assert [tuple(w) for w in seq.sequences] == words, (sent, k)
            assert seq.score == score, (sent, k)
            assert seq.num_unk == num_unk


@pytest.mark.parametrize('seed', range(2000, 2030))
def test_random_cases_against_oracle(seed):
    case = _cases.random_case(seed, n_sent=24, features=True, prefs=(seed % 2 == 0), max_sent_len=60)
    _cases.add_features(case, _cases.observed_features(case, lo, seed=seed), seed)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    sents = case['sentences']
    lat_counters = lo.Counters()
    for sent, (words, bindex) in zip(sents, tagger.lattice_batch(sents)):
        assert [tuple(w) for w in words[1:-1]] == _lattice_key(oracle.lattice(sent, lat_counters)), sent
    for k in (1, 2, 5, 10, 33, 64):
        got = tagger.tag_batch(sents, beam_size=k, errors='none')
        counters = lo.Counters()
        for sent, seq in zip(sents, got):
            try:
                want = oracle.tag(sent, k, counters)
            except IndexError:
                assert seq is None, sent
                continue
            assert [tuple(w) for w in seq.sequences] == want.words, (sent, k)
            assert seq.score == want.score, (sent, k)
        dev = tagger.counters()
        # the device counts the work of the reference's control flow (SURVEY §8d)
        for name in ('T', 'F', 'Bk', 'W'):
            assert dev[name] == getattr(counters, name), (name, k)
        assert dev['E'] == lat_counters.E and dev['P'] == lat_counters.P


def test_error_behaviour():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore())
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    with pytest.raises(IndexError):
        tagger.tag('가나다라')                      # no dictionary hit at all
    empty = tagger.tag('')
    assert [w.word for w in empty.sequences] == ['BOS', 'EOS'] and empty.score == 0
    assert tagger.tag_batch([]) == []
    assert [len(s.sequences) for s in tagger.tag_batch(['', ' ', ''])] == [2, 2, 2]
    assert tagger.lattice_batch([]) == []
    with pytest.raises(ValueError):
        tagger.tag('노래\t입니다')
    with pytest.raises(ValueError):
        pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(object()))


def test_demo_known_answer():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(unknown_penalty=-.1, known_preference=0.5))
    best = pkg.Tagger(dictionary, score_funcs=funcs).tag('너무너무너무는 아이오아이의 노래 입니다')
    assert best.score == 15.5
    assert [(w.word, w.tag0, w.len) for w in best.sequences[1:-1]] == [
        ('너무너무너무', 'Noun', 7), ('는', 'Josa', 7), ('아이오아이', 'Noun', 6), ('의', 'Josa', 6),
        ('노래', 'Noun', 2), ('입니다', 'Adjective', 3)]


def test_buffers_grow_and_rerun(monkeypatch):
    """Tiny initial staging / edge capacities force the overflow flags, the host enlarges the
    buffers and reruns on the device; results must not change."""
    case = _cases.random_case(4242, n_sent=40, features=True, max_sent_len=60)
    _cases.add_features(case, _cases.observed_features(case, lo, seed=1), 1)
    dictionary, funcs = _cases.build_objects(case, pkg)
    sents = [s for s in case['sentences']]
    oracle = lo.OracleTagger(dictionary, funcs)
    monkeypatch.setenv('LT_HIT_CAP', '8')
    monkeypatch.setenv('LT_EDGE_CAP', '16')
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    for sent, (words, bindex) in zip(sents, tagger.lattice_batch(sents)):
        assert [tuple(w) for w in words[1:-1]] == _lattice_key(oracle.lattice(sent)), sent
    got = tagger.tag_batch(sents, beam_size=5, errors='none')
    for sent, seq in zip(sents, got):
        try:
            want = oracle.tag(sent, 5)
        except IndexError:
            assert seq is None
            continue
        assert [tuple(w) for w in seq.sequences] == want.words
        assert seq.score == want.score


def test_trained_weight_format_end_to_end():
    """Tagged corpus -> scan_features -> trainer weight format -> load_params -> GPU tagger, against
    the oracle fed with the same objects (SURVEY §8f row f1)."""
    from lattice_based_tagger_b200.features import scan_features
    from lattice_based_tagger_b200.trainer import load_params
    pairs = [('너무너무너무 는  아이오아이 의  노래  입니다',
              '너무너무너무/Noun 는/Josa  아이오아이/Noun 의/Josa  노래/Noun  이/Adjective+ㅂ니다/Eomi'),
             ('아이오아이 는  공연 을  했다', '아이오아이/Noun 는/Josa  공연/Noun 을/Josa  하/Verb+았다/Eomi')]
    idx_to_feature, _, counts = scan_features(pairs, pkg.features.SimpleTrigramEncoder(),
                                              predefined_features={(6, n): 1 for n in range(1, 9)})
    params = {'idx_to_feature': idx_to_feature, 'coefficient': [0.1 * c for c in counts]}
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(), load_params(params))
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    for sent in ('너무너무너무는 아이오아이의 노래 입니다', '아이오아이는 공연을 했다', '노래를 했다 우와'):
        got, want = tagger.tag(sent), oracle.tag(sent, 5)
        assert [tuple(w) for w in got.sequences] == want.words
        assert got.score == want.score


def test_edge_cases_against_oracle():
    """Inputs the reference treats specially: blank sentences, repeated / leading / trailing spaces,
    a dictionary entry longer than the beam window, a dictionary without stand-alone tags
    (MorphemeLookup.max_len = 0 -> the sub-word scan is unbounded, lookup.py:229-230), single
    syllables, and a long sentence."""
    tag_to_morphs = {
        'Josa': {'는', '을', '가'}, 'Noun': {'가나다라마바사아자차', '가', '나다', '라마'},
        'Eomi': {'다', 'ㄴ다', '았다'}, 'Verb': {'하', '가'}, 'Adjective': {'나'},
    }
    rules = {'한': (('하', 'ㄴ'),), '갔': (('가', '았'),), '했다': (('하', '았다'),)}
    dictionary = pkg.dictionary.MorphemeDictionary(tag_to_morphs, rules)
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(-0.3, 0.4, -0.1))
    sents = ['', ' ', '   ', '가', ' 가 ', '가  나다', '가나다라마바사아자차', '가나다라마바사아자차는 갔다', '한다 했다 갔다',
             '나다라마가는' * 40, '가 ' * 100, 'x가나다라마y']
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    for k in (1, 5, 40):
        got = tagger.tag_batch(sents, beam_size=k, errors='none')
        for sent, seq in zip(sents, got):
            try:
                want = oracle.tag(sent, k)
            except IndexError:
                assert seq is None, repr(sent)
                continue
            assert [tuple(w) for w in seq.sequences] == want.words, (repr(sent), k)
            assert seq.score == want.score
    # no stand-alone tag, no predicate tag: max_len = 0
    only = pkg.dictionary.MorphemeDictionary({'Josa': {'는', '가'}, 'Eomi': {'다'}, 'Pronoun': {'나', '너는'}}, {})
    tagger2 = pkg.Tagger(only, score_funcs=funcs)
    oracle2 = lo.OracleTagger(only, funcs)
    assert tagger2.eojeol_lookup.max_len == 0
    for sent in ['나는 너는', '가나는다', '너는나']:
        words, _ = tagger2.lattice_batch([sent])[0]
        assert [tuple(w) for w in words[1:-1]] == _lattice_key(oracle2.lattice(sent))
        try:
            want = oracle2.tag(sent)
        except IndexError:
            with pytest.raises(IndexError):
                tagger2.tag(sent)
            continue
        assert [tuple(w) for w in tagger2.tag(sent).sequences] == want.words


def test_rejected_inputs():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore())
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    with pytest.raises(ValueError):
        tagger.tag('노래 \U0001F600')                       # outside the BMP
    with pytest.raises(ValueError):
        tagger.tag_batch(['노래'], beam_size=65)
    with pytest.raises(TypeError):
        pkg.Tagger(dictionary, score_funcs=None).tag('노래')
    import numpy as np
    enc = pkg.features.SimpleTrigramEncoder({(4, 1): 0})
    with pytest.raises(ValueError):
        pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(
            pkg.beam.SimpleTrigramFeatureScore(enc, np.zeros(1, dtype=np.float32))))

    class Custom(pkg.beam.BeamScoreFunction):
        pass
    with pytest.raises(ValueError):
        pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(Custom()))
    with pytest.raises(ValueError):
        pkg.Tagger(object(), score_funcs=funcs)              # not a morpheme dictionary


def _check_against_oracle(tagger, oracle, sents, beams):
    for sent, (words, bindex) in zip(sents, tagger.lattice_batch(sents)):
        assert [tuple(w) for w in words[1:-1]] == _lattice_key(oracle.lattice(sent)), sent
    for k in beams:
        got = tagger.tag_batch(sents, beam_size=k, errors='none')
        for sent, seq in zip(sents, got):
            try:
                want = oracle.tag(sent, k)
            except IndexError:
                assert seq is None, sent
                continue
            assert [tuple(w) for w in seq.sequences] == want.words, (sent, k)
            assert seq.score == want.score, (sent, k)


@pytest.mark.parametrize('seed,syllables', [(7, 14), (8, 14), (9, 22)])
def test_buckets_beyond_the_edge_cache(seed, syllables):
    """Buckets beyond the 64 edges the beam kernel caches per end position: the 14-syllable cases sit around that
    size (one second prep pass, a handful of edges scored on the fly), the 22-syllable one far beyond it."""
    _checks.check_dense_case(seed, syllables, (1, 5, 10, 20, 32, 40), min_bucket=90 if syllables > 14 else 41)


def test_trail_in_hbm_and_generic_array_sizes(monkeypatch):
    """Long sentences (sentence arrays beyond the templated 64 / 128 elements) and the HBM
    back-pointer trail forced for short ones."""
    case = _cases.random_case(5151, n_sent=16, features=True, prefs=True, max_sent_len=180)
    _cases.add_features(case, _cases.observed_features(case, lo, seed=5), 5)
    dictionary, funcs = _cases.build_objects(case, pkg)
    oracle = lo.OracleTagger(dictionary, funcs)
    sents = case['sentences']
    assert max(len(s) for s in sents) > 128
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    _check_against_oracle(tagger, oracle, sents, (5, 10, 12))
    short = [s for s in sents if len(s) <= 40]
    _check_against_oracle(tagger, oracle, short, (5, 10))              # 64-element arrays (beam 10: trail never in shared memory)
    monkeypatch.setenv('LT_TRAIL_SMEM', '0')
    _check_against_oracle(tagger, oracle, short, (5, 10, 12))          # same kernels, trail in HBM


def test_dictionary_mutation_and_refresh():
    """SURVEY §8f row f4: `add` / `remove_words` on the host dictionary (reference
    `dictionary.py:244-262`) + `Tagger.refresh()` recompiles the device tables; results follow the
    oracle on the mutated dictionary, including the stale `verbs/adjectives/eomis` views the
    reference keeps after `remove_words`."""
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(unknown_penalty=-.1, known_preference=0.5))
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    sents = ['트와이스의 노래 입니다', '아이오아이는 노래를 했다', '노래 입니다']
    first = tagger.tag_batch(sents, errors='none')
    assert [w.tag0 for w in first[0].sequences[1:3]] == ['Unknown', 'Josa'] or first[0].sequences[1].tag0 == 'Unknown'
    dictionary.add({'트와이스'}, 'Noun')
    dictionary.add('짱', 'Suffix', force=True)
    dictionary.remove_words({'입니다', '이'}, 'Adjective')
    with pytest.raises(ValueError):
        dictionary.add('x', 'NoSuchTag')
    tagger.refresh()
    _check_against_oracle(tagger, lo.OracleTagger(dictionary, funcs), sents + ['트와이스짱'], (1, 5))
    assert tagger.tag(sents[0]).sequences[1].tag0 == 'Noun'


def test_retry_pass_and_adaptive_staging(monkeypatch):
    """A staging area far too small for most eojeols: the sentences go through the retry pass, the
    main pass's capacity adapts over successive batches (>= 64 sentences), results never change."""
    case = _cases.random_case(777, n_sent=90, features=True, max_sent_len=50)
    _cases.add_features(case, _cases.observed_features(case, lo, seed=2), 2)
    dictionary, funcs = _cases.build_objects(case, pkg)
    sents = list(case['sentences'])
    oracle = lo.OracleTagger(dictionary, funcs)
    monkeypatch.setenv('LT_HIT_CAP', '8')
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    for _ in range(4):                       # capacities are sticky per tagger: 8 -> 16 -> 32 ...
        _check_against_oracle(tagger, oracle, sents, (5,))


@pytest.mark.parametrize('hit_cap', ['64', '32'])
def test_rank_by_sorting(monkeypatch, hit_cap):
    """Large eojeols are ranked by an in-place sort (lattice.cuh: rank_staged); LT_SORT_MIN=1 sends every eojeol
    through it: same lattices (edge order included), same paths, same scores."""
    case = _cases.random_case(778, n_sent=90, features=True, max_sent_len=50)
    _cases.add_features(case, _cases.observed_features(case, lo, seed=2), 2)
    dictionary, funcs = _cases.build_objects(case, pkg)
    monkeypatch.setenv('LT_SORT_MIN', '1')
    if hit_cap:
        monkeypatch.setenv('LT_HIT_CAP', hit_cap)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    _check_against_oracle(tagger, lo.OracleTagger(dictionary, funcs), list(case['sentences']), (5,))


# ---- round 2: all survivors, lookup modes, host-level API, per-sentence statuses, larger configurations ----

@pytest.mark.parametrize('name', ['demo_morph', 'random_1003', 'random_1011'])
def test_golden_all_survivors(name):
    """`beam_search` returns every survivor (beam.py:59-61): the fixtures hold all of them for k = 5
    (demo_morph: for every recorded k), as the reference returned them."""
    payload = _golden.load(name)
    case = payload['case']
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs, k3_first=payload['k3_first'])
    sents = case['sentences']
    for k in sorted({int(k) for entry in payload['expected'] for k in entry['beams']}):
        got = tagger.tag_batch_kbest(sents, beam_size=k, errors='none')
        for sent, entry, seqs in zip(sents, payload['expected'], got):
            want = _golden.expected_survivors(entry, k)
            if want is None:
                assert seqs is None, sent
                continue
            if len(want) == 1 and k > 1:
                seqs = seqs[:1]                  # the fixture kept matures[0] only for this k
            assert len(seqs) == len(want), (sent, k)
            for seq, (words, score, num_unk) in zip(seqs, want):
                assert [tuple(w) for w in seq.sequences] == words and seq.score == score and seq.num_unk == num_unk


@pytest.mark.parametrize('seed', [3001, 3011, 3012])
def test_kbest_against_oracle(seed):
    case = _checks.make_case(seed, n_sent=24, max_sent_len=50)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    _checks.check_kbest(tagger, lo.OracleTagger(dictionary, funcs), case['sentences'], (1, 3, 5, 10, 12, 32, 40, 64))


@pytest.mark.parametrize('seed', [3002, 3021, 3022, 3023])
def test_lookup_modes_and_flatten(seed):
    _checks.check_lookup_modes(_checks.make_case(seed, n_sent=16, max_sent_len=30), beams=(1, 5, 33))


@pytest.mark.parametrize('seed', [3003, 3031])
def test_host_level_api(seed):
    _checks.check_host_api(_checks.make_case(seed, n_sent=16, max_sent_len=30))


def test_reference_docstring_examples():
    """The reference's docstring examples that still reproduce against its own code (SURVEY §4)."""
    d = pkg.dictionary.DemoMorphemeDictionary()
    assert pkg.dictionary.analyze_morphology('파랬다', {}, {'파랗'}, {'았다'}, {'랬': (('랗', '았'),)}) == [
        (('파랗', 'Adjective'), ('았다', 'Eomi'))]                                        # lemmatizer.py:34-40
    assert d.lemmatize('있다') == [(('있', 'Adjective'), ('다', 'Eomi')), (('이', 'Adjective'), ('ㅆ다', 'Eomi'))]   # dictionary.py:283-291
    assert [str(w) for w in d.lookup('있다', b=3)] == ['Word(있다, 있/Adjective + 다/Eomi, len=2, b=3, e=5)',
                                                       'Word(있다, 이/Adjective + ㅆ다/Eomi, len=2, b=3, e=5)']
    assert [str(w) for w in d.lookup('아이오아이', 5)] == ['Word(아이오아이, 아이오아이/Noun, len=5, b=5, e=10)']
    lr = pkg.dictionary.LRLookup(d)
    assert [str(w) for w in lr('아이오아이', 2)] == ['Word(아이오아이, 아이오아이/Noun, len=5, b=2, e=7, L)']     # lookup.py:176-185
    lr_all = pkg.dictionary.LRLookup(d, prefer_exact_match=False)
    assert sorted(str(w) for w in lr_all('아이오아이')) == sorted([
        'Word(아이오아이, 아이오아이/Noun, len=5, b=0, e=5, L)', 'Word(아이오, 아이오/Noun, len=3, b=0, e=3, L)',
        'Word(아이, 아이/Noun, len=2, b=3, e=5)'])
    # lr_lookup's Noun + Josa special case: both words carry len = n (SURVEY App. A Q4)
    assert [(w.word, w.tag0, w.len) for w in lr_all('아이오아이의')] == [('아이오아이', 'Noun', 6), ('의', 'Josa', 6)]


def test_per_sentence_statuses():
    """One bad sentence does not fail its batch (ADVICE r1): too long for the kernels' shared memory,
    characters outside the BMP, foreign whitespace, no dictionary word — each gets its own status."""
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore())
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    limit = tagger.info()['unit_limit']
    assert 1000 <= limit <= 4088
    sents = ['노래 입니다', '노래 ' * (limit // 3 + 2), '노래 \U0001F600', '노래\t입니다', '가나다라', '']
    got = tagger.tag_batch(sents, errors='none')
    assert [s is not None for s in got] == [True, False, False, False, False, True]
    assert got[0].score == oracle.tag(sents[0]).score
    assert list(got.status) == [0, 3, 4, 2, 1, 0]
    long_ok = '노래 ' * ((limit - 8) // 3)
    want = oracle.tag(long_ok)
    seq = tagger.tag(long_ok)
    assert [tuple(w) for w in seq.sequences] == want.words and seq.score == want.score


def test_tag_debug_trace(capsys):
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore(unknown_penalty=-.1, known_preference=0.5))
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    sent = '노래 입니다'
    best = tagger.tag(sent, beam_size=3, debug=True)
    out = capsys.readouterr().out
    assert out.count('End point = ') == 5 and best.score == oracle.tag(sent, 3).score
    # the survivors printed for the last position are the search result itself
    assert str(round(best.score, 6)) in out or repr(best.score) in out


_CONFIG_SAMPLES = {'c3': (600, (10,)), 'c4': (24, (32,)), 'c5': (400, (1, 8, 10, 64))}


@pytest.mark.parametrize('name', ['c3', 'c4', 'c5'])
def test_config_samples(name):
    """BASELINE configs[2-4] at their full dictionary sizes (1 M / 100 k entries; C5's feature table is cut to
    2 M weights here — the 10 M table is built by bench.py), sentence samples against the oracle."""
    from lattice_based_tagger_b200 import synth
    n_sent, beams = _CONFIG_SAMPLES[name]
    cfg = dict(synth.CONFIGS[name])
    cfg['n_feat'] = min(cfg['n_feat'], 2_000_000)
    cfg, dictionary, sents = synth.build_workload(cfg, n_sent=max(n_sent, 256))
    reg = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore())
    reg_tagger = pkg.Tagger(dictionary, score_funcs=reg)
    vocab = None
    if cfg['n_feat'] > 1_000_000:
        vocab = [(m, t) for t, ms in dictionary.tag_to_morphs.items() for m in sorted(ms)]
    feature_dic, coef = synth.make_features(
        sents[:256], lambda s: reg_tagger.tag_batch(s, cfg['beam'], errors='none'), reg_tagger.lattice_batch,
        cfg['n_feat'], list(dictionary.tag_to_morphs), seed=3, vocab=vocab)
    reg_tagger.close()
    funcs = pkg.beam.BeamScoreFunctions(
        pkg.beam.RegularizationScore(),
        pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    sample = sents[:n_sent]
    for k in beams:
        got = tagger.tag_batch(sample, beam_size=k, errors='none')
        for sent, seq in zip(sample, got):
            try:
                want = oracle.tag(sent, k)
            except IndexError:
                assert seq is None
                continue
            assert [tuple(w) for w in seq.sequences] == want.words, (name, k, sent)
            assert seq.score == want.score
    # the lattice itself on a part of the sample, and a batch large enough to go through the adaptive staging
    for sent, (words, bindex) in zip(sample[:50], tagger.lattice_batch(sample[:50])):
        assert [tuple(w) for w in words[1:-1]] == _checks.lattice_key(oracle.lattice(sent)), sent
    info = tagger.info()
    assert info['reruns'] >= 0 and info['launches'] > 0


def test_update_weights_in_place():
    """`Tagger.update_weights()` (lt_tables_update_weights): new coefficients for the same features, written
    into the device tables without a rebuild — results follow the oracle with the new weights, hashed and
    dense (templates 3 / 4 / 6) features alike."""
    import numpy as np
    case = _checks.make_case(3041, n_sent=20, max_sent_len=40, prefs=True)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    tri = next(f for f in funcs.funcs if type(f).__name__ == 'SimpleTrigramFeatureScore')
    rng = np.random.default_rng(4)
    for _ in range(2):
        tri.coefficients = rng.standard_normal(len(tri.coefficients))
        tagger.update_weights()
        _checks.check_against_oracle(tagger, lo.OracleTagger(dictionary, funcs), case['sentences'], (1, 5, 33))
