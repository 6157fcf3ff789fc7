"""The constrained search (`lt_batch_set_constraints`) at the shapes where its kernels have logic of their own:
sentences of 60-200 syllables and one near the unit limit (end positions past a warp's 32 lanes in
constraint_prep_kernel, is_l words past the first), constrained spans in a bucket past the beam kernel's 64-edge
cache, the trail in HBM, edge cases of the C ABI, and the C2 / C4 workloads at full size.  The device is compared
with the host oracle (tests/_constrained_oracle.py) with `==` on words, fp64 scores and every survivor.

The `full_size` tests build the C2 / C4 workloads; a run through the SIMT emulator leaves them out by name."""

import random

import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native, synth
from lattice_based_tagger_b200.tagset import Unk
from oracle import lattice_oracle as lo
from tests import _cases, _checks
from tests import _constrained_oracle as co
from tests.test_gpu_constraints import _as_items, _c_constraints, _check_satisfied, _objects, check_parity, random_constraints

pytestmark = pytest.mark.gpu

# the running top-K changes its mode between 16 and 17 and between 32 and 33
BEAMS = (1, 5, 16, 17, 32, 33, 64)
PATTERNS = ('random', 'back_to_back', 'eight', 'gaps', 'dozens', 'forced_is_l')


# ---- constraint patterns ------------------------------------------------------------------------------------------
def _pick_tag(rng, tags, have):
    """A tag the span has, a tag it lacks (a forced word) or None (any word)."""
    r = rng.random()
    if have and r < 0.4:
        return rng.choice(sorted(have))
    lacking = [t for t in tags if t not in have]
    if lacking and r < 0.7:
        return rng.choice(lacking)
    return None


def _tiling(rng, tags, spans_with, b, end, lengths, gaps=(0,)):
    """Constraints from b up to `end`, each of a length from `lengths`, separated by a gap from `gaps`."""
    out = []
    while b < end:
        e = min(end, b + rng.choice(lengths))
        out.append((b, e, _pick_tag(rng, tags, spans_with.get((b, e), set()))))
        b = e + rng.choice(gaps)
    return out


def pattern_constraints(kind, rng, sent, edges, tags, survivor=None):
    """One sentence's constraints of pattern `kind` (PATTERNS)."""
    n_syl = len(sent.replace(' ', ''))
    if n_syl == 0:
        return []
    spans_with = {}
    for w in edges:
        spans_with.setdefault((w[6], w[7]), set()).add(w[3])
    if kind == 'random':
        return random_constraints(rng, sent, edges, tags, survivor)
    if kind == 'back_to_back':
        # every position ends a constraint
        return _tiling(rng, tags, spans_with, 0, n_syl, range(1, 9))
    if kind == 'eight':
        # most positions are strictly inside a constraint and keep no hypothesis
        return _tiling(rng, tags, spans_with, 0, n_syl, (8,))
    if kind == 'gaps':
        return _tiling(rng, tags, spans_with, rng.randint(0, 1), n_syl, range(1, 5), gaps=(1,))
    if kind == 'dozens':
        return _tiling(rng, tags, spans_with, 0, n_syl, (1, 2, 3), gaps=(0, 0, 1, 2))
    assert kind == 'forced_is_l'
    # the first syllable of an eojeol past syllable 32 begins a span with a tag it lacks: a forced word with is_l
    is_l = co.is_l_of(sent)
    out, free = [], 0
    for b in range(n_syl):
        if b >= 32 and b >= free and is_l[b]:
            e = min(n_syl, b + rng.randint(1, 4))
            lacking = [t for t in tags if t not in spans_with.get((b, e), set())]
            if lacking:
                out.append((b, e, rng.choice(lacking)))
                free = e
    return out


def check_forced_flags(tagger, sents, cons, beam):
    """Independent of the oracle: the word of a tagged constraint is the forced word (LT_EDGE_FORCED, the
    constraint's tag, is_l of its begin) exactly when no lattice edge of the span has that tag."""
    items = [None if c is None else _as_items(c) for c in cons]
    off, edges, _, status = tagger.tag_batch_packed(sents, beam, constraints=items)
    tag_ids = tagger._engine.tables.tag_ids
    checked = 0
    for i, (sent, (words, _)) in enumerate(zip(sents, tagger.lattice_batch(sents))):
        if status[i] != _native.LT_SENT_OK or not cons[i]:
            continue
        have = {(w.b, w.e, w.tag0) for w in words[1:-1]}
        is_l = co.is_l_of(sent)
        path = {(int(x['b']), int(x['e'])): x for x in edges[off[i]:off[i + 1]]}
        for b, e, tag in cons[i]:
            x = path[(b, e)]
            forced = bool(x['flags'] & _native.LT_EDGE_FORCED)
            assert forced == (tag is not None and (b, e, tag) not in have), (sent, (b, e, tag))
            if tag is not None:
                assert x['tag0'] == tag_ids[tag]
            if forced:
                assert bool(x['flags'] & _native.LT_EDGE_IS_L) == is_l[b], (sent, (b, e, tag))
                checked += 1
    return checked


# ---- fixtures -----------------------------------------------------------------------------------------------------
@pytest.fixture(params=['plan', 'hbm'])
def trail(request, monkeypatch, capfd):
    """'plan': the trail where the launch plan puts it; 'hbm': LT_TRAIL_SMEM=0, and after the test the LT_DEBUG
    trace must show every constrained beam launch with its trail in HBM.  Set before the tagger is built (its batch
    object reads both switches)."""
    if request.param == 'plan':
        yield request.param
        return
    monkeypatch.setenv('LT_TRAIL_SMEM', '0')
    monkeypatch.setenv('LT_DEBUG', '1')
    yield request.param
    lines = [ln for ln in capfd.readouterr().err.splitlines() if 'beam kernel' in ln and 'constrained' in ln]
    assert lines and all('trail in HBM' in ln for ln in lines), lines[:4]


def _long_sentences(seed):
    """A random case whose sentences run to 200 syllables; the ones of 60 syllables and more with a lattice."""
    case = _checks.make_case(seed, n_sent=16, prefs=seed % 2 == 0, max_sent_len=200)
    tagger, oracle = _objects(case)
    sents = [s for s in case['sentences'] if 60 <= len(s.replace(' ', '')) <= 200 and oracle.lattice(s)]
    assert len(sents) >= 4
    return case, tagger, oracle, sents


# ---- 1 + 3. long sentences, trail where the plan puts it and in HBM -----------------------------------------------
@pytest.mark.parametrize('kind', PATTERNS)
def test_long_sentences(kind, trail):
    seed = 5100 + PATTERNS.index(kind)
    case, tagger, oracle, sents = _long_sentences(seed)
    rng = random.Random(seed)
    cons = []
    for sent in sents:
        edges = oracle.lattice(sent)
        surv = rng.choice(co.survivors(oracle, sent, 5, [])).words[1:-1]
        cons.append(pattern_constraints(kind, rng, sent, edges, case['tags'], surv))
    lengths = [len(s.replace(' ', '')) for s in sents]
    if kind in ('back_to_back', 'eight', 'gaps', 'dozens'):
        assert all(c[-1][1] >= n - 2 for c, n in zip(cons, lengths))        # constraints reach the last positions
    if kind == 'dozens':
        assert min(len(c) for c in cons) >= 16 and max(len(c) for c in cons) >= 40
    if kind == 'forced_is_l':
        assert sum(len(c) for c in cons) >= 8
    check_parity(tagger, oracle, sents, cons, BEAMS)
    forced = check_forced_flags(tagger, sents, cons, 5)
    if kind == 'forced_is_l':
        assert forced >= 8


def test_sentence_near_the_unit_limit(trail):
    """One sentence a few units short of `unit_limit` with its last syllables constrained back to back (the last
    constraint ends at its last syllable), forced words at eojeol starts among them."""
    case, tagger, oracle, sents = _long_sentences(5200)
    limit = tagger._engine.unit_limit
    text = ''
    while len(text) < limit:
        text += random.Random(len(text)).choice(sents) + ' '
    sent = text[:limit - 3].strip()
    n_syl = len(sent.replace(' ', ''))
    assert n_syl > 32 * 32 and len(sent) <= limit
    rng = random.Random(52)
    edges = oracle.lattice(sent)
    spans_with = {}
    for w in edges:
        spans_with.setdefault((w[6], w[7]), set()).add(w[3])
    cons = _tiling(rng, case['tags'], spans_with, n_syl - 48, n_syl, range(1, 9))
    is_l = co.is_l_of(sent)
    for i, (b, e, tag) in enumerate(cons):
        lacking = [t for t in case['tags'] if t not in spans_with.get((b, e), set())]
        if is_l[b] and lacking:
            cons[i] = (b, e, lacking[0])
    assert cons[-1][1] == n_syl and any(is_l[b] for b, _, _ in cons)
    batch = [sents[0], sent, sents[1]]
    check_parity(tagger, oracle, batch, [[], cons, None], BEAMS)
    assert tagger.tag_batch_packed(batch, 5, constraints=[[], _as_items(cons), None])[3].tolist() == [0, 0, 0]
    check_forced_flags(tagger, [sent], [cons], 5)


# ---- 2 + 3. constrained spans in a bucket past the edge cache ------------------------------------------------------
CACHED = 64          # kBucketCached (beam.cuh): edges of a bucket the beam kernel prepares ahead


def _dense(seed, syllables):
    case = _checks.dense_case(seed, syllables)
    _cases.add_features(case, _cases.observed_features(case, lo, seed=seed), seed)
    tagger, oracle = _objects(case)
    return case, tagger, oracle, case['sentences']


@pytest.mark.parametrize('seed,syllables', [(7, 14), (9, 22)])
def test_dense_buckets(seed, syllables, trail):
    """In-window spans of the biggest bucket of each sentence, constrained with a tag of the span's edges (at bucket
    index >= 64 where the bucket is that large), with a tag no edge of the span has (a forced word) and with any
    word, alone and two at a time."""
    case, tagger, oracle, sents = _dense(seed, syllables)
    rng = random.Random(seed)
    cons_by_kind = {'present': [], 'absent': [], 'any': [], 'two': []}
    beyond = 0
    for sent, (words, _) in zip(sents, tagger.lattice_batch(sents)):
        inner = words[1:-1]
        big_e = max({w.e for w in inner}, key=lambda e: sum(w.e == e for w in inner))
        bucket = [w for w in inner if w.e == big_e]             # the device's CSR order: begin ascending
        spans = sorted({(w.b, w.e) for w in bucket if w.e - w.b <= _native.LT_WINDOW})
        index = {}
        for k, w in enumerate(bucket):
            index.setdefault((w.b, w.e, w.tag0), []).append(k)
        # the in-window span and tag whose edges sit furthest into the bucket
        b, e, tag = max((k for k in index if k[1] - k[0] <= _native.LT_WINDOW), key=lambda k: min(index[k]))
        if min(index[(b, e, tag)]) >= CACHED:
            beyond += 1
        lacking = [t for t in case['tags'] if (b, e, t) not in index]
        b0 = spans[0][0]
        cons_by_kind['present'].append([(b, e, tag)])
        cons_by_kind['absent'].append([(b, e, rng.choice(lacking))])
        cons_by_kind['any'].append([(b, e, None)])
        cons_by_kind['two'].append([(b0, b, rng.choice(case['tags'] + [None])), (b, e, tag)] if b0 < b else [(b, e, tag)])
    # (the 14-syllable case's biggest buckets hold up to 67 edges: their in-window spans begin below index 64)
    assert beyond >= (2 if syllables > 14 else 0)
    for kind, cons in cons_by_kind.items():
        check_parity(tagger, oracle, sents, cons, BEAMS)
        check_forced_flags(tagger, sents, cons, 5)


# ---- 4. edge cases through the C ABI ------------------------------------------------------------------------------
def _bound(tagger, per_sent, call):
    rc, handle = _c_constraints(tagger, per_sent)
    assert rc == _native.LT_OK
    try:
        _native.check(tagger._lib.lt_batch_set_constraints(tagger._batch, handle))
        return call()
    finally:
        _native.check(tagger._lib.lt_batch_set_constraints(tagger._batch, None))
        tagger._lib.lt_constraints_destroy(handle)


def test_empty_batch_with_a_bound_set():
    tagger, _ = _objects(_checks.make_case(5300, n_sent=6, max_sent_len=24))
    engine = tagger._engine
    path_off, edges, _, status = _bound(tagger, [], lambda: engine.tag_packed([], 5))
    assert path_off.tolist() == [0] and len(edges) == 0 and len(status) == 0
    n_best, path_off, edges, _, status = _bound(tagger, [], lambda: engine.kbest_packed([], 33))
    assert path_off.tolist() == [0] and len(n_best) == len(edges) == len(status) == 0
    assert engine.unpack_kbest([], (n_best, path_off, edges, _, status), 33, 'none') == []


def test_c_abi_edge_cases():
    """An empty sentence with a constraint; a constraint ending at the last syllable beside the same sentence with
    one ending past it; sentences whose lattice status is not OK keep it whatever their constraints."""
    case = _checks.make_case(5301, n_sent=10, max_sent_len=40)
    tagger, oracle = _objects(case)
    engine = tagger._engine
    tags = engine.tables.tag_ids
    base = [s for s in case['sentences'] if len(s.replace(' ', '')) >= 4 and oracle.lattice(s)][:2]
    n = [len(s.replace(' ', '')) for s in base]
    tag = case['tags'][0]
    sents = ['', base[0], base[0], base[1], base[1],
             'x' * (engine.unit_limit + 1), '\U0001F600' + base[0], 'a\tb', case['sentences'][-1]]
    per = [[(0, 1, _native.LT_NO_TAG)],
           [(0, 1, _native.LT_NO_TAG), (n[0] - 2, n[0], tags[tag])],
           [(0, 1, _native.LT_NO_TAG), (n[0] - 2, n[0] + 1, tags[tag])],
           [(n[1] - 1, n[1], _native.LT_NO_TAG)],
           [(n[1], n[1] + 1, _native.LT_NO_TAG)],
           [(0, 1, tags[tag]), (engine.unit_limit, engine.unit_limit + 1, _native.LT_NO_TAG)],
           [(0, 8, _native.LT_NO_TAG), (n[0] + 1, n[0] + 9, _native.LT_NO_TAG)],
           [(0, 1, tags[tag]), (2, 3, _native.LT_NO_TAG), (4, 5, _native.LT_NO_TAG)],
           [(0, 3, _native.LT_NO_TAG), (3, 9, _native.LT_NO_TAG)]]
    want_status = [_native.LT_SENT_BAD_CONSTRAINT, 0, _native.LT_SENT_BAD_CONSTRAINT, 0, _native.LT_SENT_BAD_CONSTRAINT,
                   _native.LT_SENT_TOO_LONG, _native.LT_SENT_UNSUPPORTED_CHAR, _native.LT_SENT_BAD_SPACE,
                   _native.LT_SENT_NO_EDGES]
    for k in (1, 5, 17, 33):
        packed = _bound(tagger, per, lambda: engine.tag_packed(sents, k))
        assert packed[3].tolist() == want_status
        kbest = _bound(tagger, per, lambda: engine.kbest_packed(sents, k))
        n_best, kstatus = kbest[0], kbest[4]
        assert kstatus.tolist() == want_status
        got = engine.unpack_kbest(sents, kbest, k, 'none')
        for i, st in enumerate(want_status):
            if st != 0:
                assert n_best[i] == 0 and got[i] is None and packed[0][i + 1] == packed[0][i], i
                continue
            cons = [(c[0], c[1], None if c[2] == _native.LT_NO_TAG else tag) for c in per[i]]
            want = co.survivors(oracle, sents[i], k, cons)
            assert n_best[i] == len(want)
            for seq, hyp in zip(got[i], want):
                assert [tuple(w) for w in seq.sequences] == hyp.words and seq.score == hyp.score, (i, k)
            assert packed[2][i] == want[0].score


# ---- 5. the C2 and C4 workloads at full size ------------------------------------------------------------------------
_FULL = {'c2': dict(n_sent=None, oracle=300), 'c4': dict(n_sent=256, oracle=24)}


@pytest.fixture(scope='module')
def full_size_workload():
    cache = {}

    def get(name):
        if name not in cache:
            cfg, dictionary, sents = synth.build_workload(name, n_sent=_FULL[name]['n_sent'])
            beam = cfg['beam']
            reg = pkg.beam.RegularizationScore()
            probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
            ok = [s for s, st in zip(sents, probe.tag_batch_packed(sents, beam)[3]) if st == 0]
            feature_dic, coef = synth.make_features(ok[:1000], lambda s: probe.tag_batch(s, beam, errors='none'),
                                                    probe.lattice_batch, cfg['n_feat'], list(dictionary.tag_to_morphs), seed=3)
            probe.close()
            funcs = pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
            cache[name] = (beam, dictionary, funcs, sents, pkg.Tagger(dictionary, score_funcs=funcs))
        return cache[name]
    yield get
    for entry in cache.values():
        entry[-1].close()


def _from_best_paths(tagger, sents, best, setting, tags, seed):
    """Per sentence constraints drawn from its unconstrained best path: two of its words, or every word (Unknown
    words as untagged spans); about one tagged constraint in eight gets a tag its span lacks."""
    rng = random.Random(seed)
    cons = []
    for seq in best:
        if seq is None:
            cons.append(None)
            continue
        items = [(w.b, w.e, None if w.tag0 == Unk else w.tag0) for w in seq.sequences[1:-1] if w.e - w.b <= _native.LT_WINDOW]
        cons.append(items if setting == 'every_word' else sorted(rng.sample(items, min(2, len(items)))))
    swap = [i for i, c in enumerate(cons) if c and rng.random() < 0.25]
    for i, (words, _) in zip(swap, tagger.lattice_batch([sents[i] for i in swap])):
        have = {(w.b, w.e, w.tag0) for w in words[1:-1]}
        for k, (b, e, tag) in enumerate(cons[i]):
            lacking = [t for t in tags if (b, e, t) not in have]
            if tag is not None and lacking and rng.random() < 0.5:
                cons[i][k] = (b, e, rng.choice(lacking))
    return cons


@pytest.mark.parametrize('name', ['c2', 'c4'])
@pytest.mark.parametrize('setting', ['two_per_sentence', 'every_word'])
def test_full_size_workloads(full_size_workload, name, setting):
    """Every OK sentence gets a path that keeps its constraints, every survivor's score is what the given-path
    kernel (`Tagger.score_paths`, the reference's arithmetic) computes for its words, and a sample matches the
    oracle survivor for survivor."""
    beam, dictionary, funcs, sents, tagger = full_size_workload(name)
    tags = list(dictionary.tag_to_morphs)
    best = tagger.tag_batch(sents, beam, errors='none', lazy=False)
    cons = _from_best_paths(tagger, sents, best, setting, tags, seed=len(sents))
    assert sum(1 for c in cons if c) > 0.9 * len(sents)
    items = [None if c is None else _as_items(c) for c in cons]
    got = tagger.tag_batch_kbest(sents, beam, errors='none', constraints=items)
    paths = []
    for seq0, c, seqs in zip(best, cons, got):
        if seq0 is None:
            continue
        assert seqs, c
        for seq in seqs:
            _check_satisfied(seq.sequences, c)
        paths += seqs
    scores = tagger.score_paths(paths)
    assert scores.tolist() == [seq.score for seq in paths]
    oracle = lo.OracleTagger(dictionary, funcs)
    for i in random.Random(5).sample(range(len(sents)), _FULL[name]['oracle']):
        if best[i] is None:
            continue
        want = co.survivors(oracle, sents[i], beam, cons[i])
        assert len(got[i]) == len(want), i
        for seq, hyp in zip(got[i], want):
            assert [tuple(w) for w in seq.sequences] == hyp.words and seq.score == hyp.score, i
