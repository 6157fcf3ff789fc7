"""The CUDA kernel SOURCES, compiled for the host against the SIMT emulator (tests/simt), checked
against the oracle on the CPU — test infrastructure: it exercises the kernels' logic (enumeration
order, tie-breaking, fp64 association, overflow / retry paths, lookup modes, k-best, imported
lattices) where no GPU exists, and the emulator aborts on warp-divergent collectives.  The product
never loads this build; the `-m gpu` tests run the same checks through `liblt_b200.so`.
"""

import pytest

import lattice_based_tagger_b200 as pkg
from oracle import lattice_oracle as lo
from tests import _cases, _checks, _emu, _golden


@pytest.fixture(autouse=True)
def emulated():
    with _emu.emulated():
        yield


@pytest.mark.parametrize('seed', [2001, 2016])
def test_random_cases(seed):
    case = _checks.make_case(seed, n_sent=10, max_sent_len=40)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    _checks.check_against_oracle(tagger, oracle, case['sentences'], (1, 5, 10, 33), counters=True)


def test_golden_demo_fixture():
    payload = _golden.load('demo_morph')
    case = payload['case']
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs, k3_first=payload['k3_first'])
    sents = case['sentences']
    for sent, entry, (words, bindex) in zip(sents, payload['expected'], tagger.lattice_batch(sents)):
        assert [tuple(w) for w in words[1:-1]] == _checks.lattice_key([_golden.edge(w) for w in entry['lattice']]), sent
    for k in (1, 3, 5, 32):
        got = tagger.tag_batch_kbest(sents, beam_size=k, errors='none')
        for sent, entry, seqs in zip(sents, payload['expected'], got):
            want = _golden.expected_survivors(entry, k)
            if want is None:
                assert seqs is None, sent
                continue
            assert len(seqs) == len(want)
            for seq, (words, score, num_unk) in zip(seqs, want):       # every survivor the reference returned
                assert [tuple(w) for w in seq.sequences] == words and seq.score == score and seq.num_unk == num_unk


@pytest.mark.parametrize('block_order', ['forward', 'reverse'])
def test_many_sentences_across_ctas(monkeypatch, block_order):
    """A batch large enough for the multi-CTA kernels around the two big ones (work-order prologue, path
    offsets + packing), with the emulator running the CTAs first-to-last and last-to-first: a result that
    depends on which CTA writes last is a race on the GPU."""
    monkeypatch.setenv('LT_SIMT_BLOCK_ORDER', block_order)
    monkeypatch.setenv('LT_SIMT_SMS', '64')          # grids as wide as on the device: several CTAs per kernel
    case = _checks.make_case(2001, n_sent=12, max_sent_len=14)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    sents = [case['sentences'][i % 12] for i in range(4200)]
    want = {}
    for sent in set(sents):
        try:
            want[sent] = oracle.tag(sent, 5)
        except IndexError:
            want[sent] = None
    got = tagger.tag_batch(sents, beam_size=5, errors='none')
    for sent, seq in zip(sents, got):
        if want[sent] is None:
            assert seq is None
        else:
            assert [tuple(w) for w in seq.sequences] == want[sent].words and seq.score == want[sent].score


@pytest.mark.parametrize('hit_cap', ['64', '32'])
def test_rank_by_sorting(monkeypatch, hit_cap):
    """The lattice kernel ranks the hits of large eojeols with an in-place sort instead of the counting loop;
    LT_SORT_MIN=1 sends every eojeol through it (staging areas other than the default one: the instantiation for
    short sentences with the default area carries no sort; small areas add flushes, retries and the fallback for
    eojeols whose padding does not fit)."""
    monkeypatch.setenv('LT_SORT_MIN', '1')
    if hit_cap:
        monkeypatch.setenv('LT_HIT_CAP', hit_cap)
    case = _checks.make_case(2016, n_sent=14, max_sent_len=48)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    _checks.check_against_oracle(tagger, oracle, case['sentences'], (5,), counters=True)


@pytest.mark.parametrize('seed,syllables', [(7, 14), (9, 22)])
def test_buckets_beyond_the_edge_cache(seed, syllables):
    """The beam kernel's any-sentence copy of the position loop: buckets of more edges than the edge cache holds
    (a second prep pass up to 64 edges, edges beyond prepared on the fly), spans beyond the window."""
    _checks.check_dense_case(seed, syllables, (5, 10, 33), min_bucket=90 if syllables > 14 else 41)


def test_kbest_survivors():
    case = _checks.make_case(3001, n_sent=10, max_sent_len=24)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    _checks.check_kbest(tagger, lo.OracleTagger(dictionary, funcs), case['sentences'], (1, 3, 5, 12, 40))


def test_lookup_modes_and_flatten():
    _checks.check_lookup_modes(_checks.make_case(3002, n_sent=8, max_sent_len=14))


def test_host_level_api():
    _checks.check_host_api(_checks.make_case(3003, n_sent=10, max_sent_len=20))


def test_overflow_rerun_and_retry_pass(monkeypatch):
    case = _checks.make_case(2001, n_sent=18, prefs=False, max_sent_len=60)
    dictionary, funcs = _cases.build_objects(case, pkg)
    oracle = lo.OracleTagger(dictionary, funcs)
    monkeypatch.setenv('LT_HIT_CAP', '8')
    monkeypatch.setenv('LT_EDGE_CAP', '16')
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    _checks.check_against_oracle(tagger, oracle, case['sentences'], (5,))
    info = tagger.info()
    assert info['reruns'] > 0 and info['retry_hcap'] > 0


def test_per_sentence_statuses():
    """One bad sentence does not fail its batch: too long for the kernels' shared memory, characters
    outside the BMP, foreign whitespace, no dictionary word — each gets its own status."""
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    funcs = pkg.beam.BeamScoreFunctions(pkg.beam.RegularizationScore())
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    limit = tagger.info()['unit_limit']
    assert 1000 <= limit <= 4088
    sents = ['노래 입니다', '노래 ' * (limit // 3 + 2), '노래 \U0001F600', '노래\t입니다', '가나다라', '']
    got = tagger.tag_batch(sents, errors='none')
    assert [s is not None for s in got] == [True, False, False, False, False, True]
    assert got[0].score == lo.OracleTagger(dictionary, funcs).tag(sents[0]).score
    assert list(got.status) == [0, 3, 4, 2, 1, 0]
    for i, exc in ((1, ValueError), (2, ValueError), (3, ValueError), (4, IndexError)):
        with pytest.raises(exc):
            tagger.tag(sents[i])
    assert [w is None for w in tagger.eojeol_lookup.lookup_batch(sents, errors='none')] == [False, True, True, True, False, False]
    long_ok = '노래 ' * ((limit - 8) // 3)
    assert tagger.tag(long_ok).score == lo.OracleTagger(dictionary, funcs).tag(long_ok).score


def test_update_weights_and_trainer():
    import numpy as np
    import tests.test_trainer as trainer_tests
    trainer_tests.test_perceptron_fits_the_toy_corpus()          # the perceptron over the (emulated) decoder
    case = _checks.make_case(3001, n_sent=8, max_sent_len=24)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    tri = next(f for f in funcs.funcs if type(f).__name__ == 'SimpleTrigramFeatureScore')
    tri.coefficients = np.random.default_rng(0).standard_normal(len(tri.coefficients))
    tagger.update_weights()
    _checks.check_against_oracle(tagger, lo.OracleTagger(dictionary, funcs), case['sentences'], (1, 5))


@pytest.mark.parametrize('block_order', ['forward', 'reverse'])
def test_path_kernels(monkeypatch, block_order):
    """The given-path kernels (tests/test_gpu_path_edges.py) on an emulated device of 2 SMs, whose launches are
    small enough that the path and perceptron grids take their stride: paths across chunk boundaries, the
    perceptron on long sentences, after each kind of search and through a sequence of batches."""
    import tests.test_gpu_path_edges as path_edges
    monkeypatch.setenv('LT_SIMT_BLOCK_ORDER', block_order)
    monkeypatch.setenv('LT_SIMT_SMS', '2')
    path_edges.check_chunk_boundaries(21, 'all', per_length=3)
    path_edges.check_path_grid_stride(23, per_length=2)
    path_edges.check_long_sentences(31, n_long=2)
    for search in ('tag', 'kbest', 'imported'):
        path_edges.check_after_search(search)
    path_edges.check_batch_sequence(n_big=60)
    monkeypatch.setenv('LT_HIT_CAP', '8')
    monkeypatch.setenv('LT_EDGE_CAP', '16')
    path_edges.check_after_search('rerun')


@pytest.mark.parametrize('block_order', ['forward', 'reverse'])
def test_constrained_search_across_ctas(monkeypatch, block_order):
    """The constrained search over a few hundred sentences of mixed statuses on an emulated device of 2 SMs: the
    constraint preparation and the beam grids take their stride, with the CTAs run in both orders."""
    import random
    from lattice_based_tagger_b200 import _native
    from tests import _constrained_oracle as co
    from tests.test_gpu_constraint_edges import PATTERNS, pattern_constraints
    from tests.test_gpu_constraints import _as_items
    monkeypatch.setenv('LT_SIMT_BLOCK_ORDER', block_order)
    monkeypatch.setenv('LT_SIMT_SMS', '2')
    case = _checks.make_case(5400, n_sent=14, max_sent_len=60)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    bad = ['\U0001F600가', '가\t나', 'x' * (tagger.info()['unit_limit'] + 1)]
    pool = case['sentences'] + bad
    sents = [pool[i % len(pool)] for i in range(320)]
    memo, cons = {}, []
    for i, sent in enumerate(sents):
        key = (sent, PATTERNS[i % len(PATTERNS)])
        if key not in memo:
            memo[key] = pattern_constraints(key[1], random.Random(i), sent, oracle.lattice(sent), case['tags'])
        cons.append(memo[key])
    got = tagger.tag_batch_kbest(sents, 5, errors='none', constraints=[_as_items(c) for c in cons])
    status = tagger.tag_batch_packed(sents, 5, constraints=[_as_items(c) for c in cons])[3]
    assert {_native.LT_SENT_UNSUPPORTED_CHAR, _native.LT_SENT_BAD_SPACE, _native.LT_SENT_TOO_LONG,
            _native.LT_SENT_NO_EDGES} <= set(status.tolist())
    want = {}
    for sent, c, seqs in zip(sents, cons, got):
        if sent in bad:
            assert seqs is None
            continue
        key = (sent, tuple(c))
        if key not in want:
            try:
                want[key] = [(h.words, h.score) for h in co.survivors(oracle, sent, 5, c)]
            except IndexError:
                want[key] = None
        if want[key] is None:
            assert seqs is None, sent
        else:
            assert [([tuple(w) for w in s.sequences], s.score) for s in seqs] == want[key], (sent, c)


def test_memcheck_self_test(tmp_path):
    """LT_SIMT_MEMCHECK=1 places device buffers and a launch's dynamic shared memory against guard pages: the
    emulator's own check that an access one element past either is caught (and that a clean kernel is not)."""
    import os
    import subprocess
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'simt')
    exe = str(tmp_path / 'selftest_memcheck')
    subprocess.run(['g++', '-std=c++17', '-O1', '-DLT_SIMT_EMU', '-I', here, '-o', exe,
                    os.path.join(here, 'selftest_memcheck.cpp'), os.path.join(here, 'simt.cpp')], check=True)
    env = dict(os.environ, LT_SIMT_MEMCHECK='1')
    clean = subprocess.run([exe, 'ok'], env=env, capture_output=True, text=True)
    assert clean.returncode == 0 and 'clean' in clean.stdout
    for what in ('global', 'shared'):
        out = subprocess.run([exe, what], env=env, capture_output=True, text=True)
        assert out.returncode != 0 and 'memcheck: invalid access' in out.stderr, (what, out.stderr)
    assert subprocess.run([exe, 'global'], capture_output=True).returncode == 0      # off without the switch


def test_kernels_under_memcheck():
    """The kernels over random cases with every device buffer and the shared memory of every launch ending at a
    guard page (a fresh process: the switch is read once), small staging areas included — the retry pass and the
    grow-and-rerun path index the buffers closest to their ends."""
    import os
    import subprocess
    import sys
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'fuzz_emulated.py')
    for extra in ({}, {'LT_HIT_CAP': '8', 'LT_EDGE_CAP': '16'}):
        env = dict(os.environ, LT_SIMT_MEMCHECK='1', **extra)
        out = subprocess.run([sys.executable, script, '2001', '2004'], env=env, capture_output=True, text=True)
        assert out.returncode == 0 and '0 failures' in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
