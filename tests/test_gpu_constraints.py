"""Constrained search (`constraints=` of `Tagger.tag_batch`, `lt_batch_set_constraints`): the oracle against brute
force on the host, then the device against the oracle (tests/_constrained_oracle.py) with `==` on words and fp64
scores, best path and every survivor."""

import ctypes
import random

import numpy as np
import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native
from oracle import lattice_oracle as lo
from tests import _cases, _checks, _golden
from tests import _constrained_oracle as co

BEAMS = (1, 2, 5, 10, 16, 32, 33, 64)
CONTEXTUAL = ('Noun', 'Verb', 'Adjective', 'Adverb')
LT_ERR_INVALID = 1


# ---- fixtures ----------------------------------------------------------------------------------------------------
def _case(seed, prefs, reg_tri=False, n_sent=16, max_sent_len=24):
    case = _checks.make_case(seed, n_sent=n_sent, prefs=prefs, max_sent_len=max_sent_len)
    if reg_tri:
        # the (RegularizationScore, SimpleTrigramFeatureScore) program, the other family of instantiations
        case['funcs'] = [f for f in case['funcs'] if f['kind'] == 'reg'] + [f for f in case['funcs'] if f['kind'] == 'trigram']
    return case


def _objects(case, **kw):
    dictionary, funcs = _cases.build_objects(case, pkg)
    return pkg.Tagger(dictionary, score_funcs=funcs, **kw), lo.OracleTagger(dictionary, funcs)


def _word_tags(case):
    return [t for t in case['tags']]


def _free_spans(rng, n_syl, taken, lo_len=1, hi_len=8):
    """A random span of lo_len..hi_len syllables that overlaps none of `taken`, or None."""
    for _ in range(20):
        length = rng.randint(lo_len, min(hi_len, n_syl)) if n_syl >= lo_len else 0
        if length == 0:
            return None
        b = rng.randint(0, n_syl - length)
        if all(b + length <= tb or te <= b for tb, te in taken):
            return b, b + length
    return None


def random_constraints(rng, sent, edges, tags, survivor=None):
    """One sentence's constraints, drawn from one of several kinds (see the module's tests)."""
    chars = sent.replace(' ', '')
    n_syl = len(chars)
    if n_syl == 0:
        return []
    spans_with = {}
    for w in edges:
        spans_with.setdefault((w[6], w[7]), set()).add(w[3])
    kind = rng.choice(['survivor', 'survivor_any', 'lacking', 'eight', 'whole', 'adjacent', 'unk_chain', 'edges'])
    out = []
    if kind in ('survivor', 'survivor_any') and survivor:
        for w in survivor:
            if rng.random() < 0.5 and w[7] - w[6] <= lo.WINDOW:
                tag = w[3] if (kind == 'survivor' and w[3] not in (lo.UNK,)) else None
                out.append((w[6], w[7], tag))
        return out
    if kind == 'whole':
        return [(0, min(n_syl, 8), rng.choice(tags + [None]))]
    if kind == 'eight':
        span = _free_spans(rng, n_syl, [], 8, 8) if n_syl >= 8 else (0, n_syl)
        return [span + (rng.choice(tags + [None]),)]
    if kind == 'adjacent':
        b = rng.randint(0, n_syl - 1)
        while b < n_syl and len(out) < 4:
            e = min(n_syl, b + rng.randint(1, 3))
            out.append((b, e, rng.choice(tags + [None])))
            b = e
        return out
    if kind == 'unk_chain':
        # spans without any lattice edge, one after the other, any word: unknown words after unknown words
        b = 0
        while b < n_syl:
            e = b + 1
            while e <= n_syl and (b, e) in spans_with:
                e += 1
            if e <= n_syl and e - b <= 2 and rng.random() < 0.7:
                out.append((b, e, None))
            b = e
        return out
    taken = []
    for _ in range(rng.randint(1, 3)):
        if kind == 'edges' and spans_with and rng.random() < 0.7:
            b, e = rng.choice(sorted(spans_with))
            if e - b > 8 or any(not (e <= tb or te <= b) for tb, te in taken):
                continue
        else:
            span = _free_spans(rng, n_syl, taken)
            if span is None:
                continue
            b, e = span
        lacking = [t for t in tags if t not in spans_with.get((b, e), set())]
        tag = rng.choice(lacking) if (lacking and rng.random() < 0.6) else rng.choice(tags + [None])
        taken.append((b, e))
        out.append((b, e, tag))
    return sorted(out)


def _first_last(n_syl, rng, tags):
    """Constraints on the first and the last syllable."""
    if n_syl < 2:
        return [(0, n_syl, None)] if n_syl else []
    return [(0, 1, rng.choice(tags + [None])), (n_syl - 1, n_syl, rng.choice(tags + [None]))]


def _as_items(cons):
    return [(b, e) if tag is None else (b, e, tag) for b, e, tag in cons]


def _constraints_for(case, oracle, sents, seed, beam=5):
    rng = random.Random(seed)
    tags = _word_tags(case)
    out = []
    for i, sent in enumerate(sents):
        edges = oracle.lattice(sent)
        try:
            surv = oracle.survivors(sent, beam)
            words = rng.choice(surv).words[1:-1]
        except IndexError:
            out.append(None)
            continue
        if i % 5 == 4:
            out.append(_first_last(len(sent.replace(' ', '')), rng, tags))
        else:
            out.append(random_constraints(rng, sent, edges, tags, words))
    return out


def _check_satisfied(words, cons):
    """Independent of the oracle: a word exactly on every constrained span, with its tag, none crossing one."""
    spans = {(w[6], w[7]): w for w in words[1:-1]}
    for b, e, tag in cons or ():
        assert (b, e) in spans, ((b, e), words)
        if tag is not None:
            assert spans[(b, e)][3] == tag, ((b, e, tag), spans[(b, e)])
    for w in words[1:-1]:
        for b, e, _ in cons or ():
            assert not (w[6] < e and b < w[7]) or (w[6], w[7]) == (b, e), (w, (b, e))


def check_parity(tagger, oracle, sents, cons, beams, imported=None):
    items = [None if c is None else _as_items(c) for c in cons]
    for k in beams:
        if imported is None:
            got = tagger.tag_batch_kbest(sents, beam_size=k, errors='none', constraints=items)
            best = tagger.tag_batch(sents, beam_size=k, errors='none', constraints=items)
        else:
            engine = tagger._engine
            packed = engine.kbest_packed(sents, k, imported=imported, constraints=items)
            got = engine.unpack_kbest(sents, packed, k, 'none', engine._imported_words)
            best = [None if g is None else g[0] for g in got]
        for sent, c, seqs, top in zip(sents, cons, got, best):
            try:
                want = co.survivors(oracle, sent, k, c if c is not None else [])
            except IndexError:
                assert seqs is None and top is None, sent
                continue
            assert seqs is not None and len(seqs) == len(want), (sent, c, k)
            assert len(want) >= 1, (sent, c)
            for seq, hyp in zip(seqs, want):
                assert [tuple(w) for w in seq.sequences] == hyp.words, (sent, c, k)
                assert seq.score == hyp.score, (sent, c, k)
                _check_satisfied(hyp.words, c)
            assert top == seqs[0]


# ---- the oracle against brute force (host only) -------------------------------------------------------------------
@pytest.mark.parametrize('seed', range(6))
def test_oracle_matches_brute_force(seed):
    case = _case(3000 + seed, prefs=seed % 2 == 0, n_sent=4, max_sent_len=8)
    dictionary, funcs = _cases.build_objects(case, pkg)
    oracle = lo.OracleTagger(dictionary, funcs)
    rng = random.Random(seed)
    tags = _word_tags(case)
    checked = 0
    alphabet = sorted({ch for s in case['sentences'] for ch in s if ch != ' '})
    for trial in range(30):
        sent = ''.join(rng.choice(alphabet + [' ']) for _ in range(rng.randint(1, 8))).strip() or alphabet[0]
        chars = sent.replace(' ', '')
        if len(chars) > 7:
            continue
        edges = oracle.lattice(sent)
        if not edges:
            continue
        bindex = lo.begin_index(sent, edges)
        is_l = co.is_l_of(sent)
        cons = random_constraints(rng, sent, edges, tags) if trial % 4 else _first_last(len(chars), rng, tags)
        paths = co.brute_force(bindex, chars, oracle.program, cons, is_l)
        # a beam larger than any position's hypotheses: the search is exhaustive
        got = co.beam_search(bindex, chars, oracle.program, 10 ** 6, constraints=cons, is_l=is_l)
        assert paths and got, (sent, cons)
        assert got[0].score == max(s for _, s in paths), (sent, cons)
        assert sorted(repr((h.words[1:-1], h.score)) for h in got) == sorted(repr((p, s)) for p, s in paths)
        for h in got:
            _check_satisfied(h.words, cons)
        checked += 1
    assert checked >= 10


@pytest.mark.parametrize('name', ['demo_morph', 'random_1000', 'random_1003', 'random_1010'])
def test_oracle_without_constraints_is_the_oracle(name):
    payload = _golden.load(name)
    case = payload['case']
    dictionary, funcs = _cases.build_objects(case, pkg)
    oracle = lo.OracleTagger(dictionary, funcs, k3_first=payload.get('k3_first'))
    for sent in case['sentences']:
        chars = sent.replace(' ', '')
        edges = oracle.lattice(sent)
        bindex = lo.begin_index(sent, edges)
        try:
            want = lo.beam_search(bindex, chars, oracle.program, 5)
        except IndexError:
            for cons in (None, []):
                with pytest.raises(IndexError):
                    co.beam_search(bindex, chars, oracle.program, 5, constraints=cons, is_l=co.is_l_of(sent))
            continue
        for cons in (None, []):
            got = co.beam_search(bindex, chars, oracle.program, 5, constraints=cons, is_l=co.is_l_of(sent))
            assert [(h.words, h.score) for h in got] == [(h.words, h.score) for h in want]


# ---- device against oracle --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('seed,prefs,reg_tri', [(3100, False, True), (3101, True, False), (3102, False, False)])
def test_parity_every_beam(seed, prefs, reg_tri):
    case = _case(seed, prefs, reg_tri)
    tagger, oracle = _objects(case)
    sents = case['sentences']
    cons = _constraints_for(case, oracle, sents, seed)
    check_parity(tagger, oracle, sents, cons, BEAMS)


@pytest.mark.gpu
@pytest.mark.parametrize('seed', [3200, 3201])
def test_forced_words_fire_features(seed):
    """Forced words score like any word: a WPREF entry on (tag, surface), template 5 with is_l, template 8 with
    contextual tags."""
    case = _case(seed, prefs=True)
    dictionary, funcs = _cases.build_objects(case, pkg)
    oracle = lo.OracleTagger(dictionary, funcs)
    rng = random.Random(seed)
    sents = [s for s in case['sentences'] if len(s.replace(' ', '')) >= 3 and oracle.lattice(s)]
    cons = []
    for sent in sents:
        chars = sent.replace(' ', '')
        edges = oracle.lattice(sent)
        have = {(w[6], w[7], w[3]) for w in edges}
        b = rng.randint(0, len(chars) - 2)
        e = min(len(chars), b + rng.randint(1, 3))
        tag = rng.choice([t for t in CONTEXTUAL if t in case['tags'] and (b, e, t) not in have] or [None])
        c2 = [(b, e, tag)]
        if e + 1 <= len(chars):
            tag2 = rng.choice([t for t in CONTEXTUAL if t in case['tags'] and (e, e + 1, t) not in have] or [None])
            c2.append((e, e + 1, tag2))
        cons.append(c2)
    # features and preferences keyed on the forced words
    wp = next(f for f in case['funcs'] if f['kind'] == 'wpref')['table']
    for sent, c in zip(sents, cons):
        chars = sent.replace(' ', '')
        is_l = co.is_l_of(sent)
        for b, e, tag in c:
            if tag is None:
                continue
            surface = chars[b:e]
            wp.setdefault(tag, {})[surface] = 1.75
            case['feature_keys'].append((5, surface, tag, is_l[b]))
            case['coefficients'].append(0.625)
            for b0 in range(max(0, b - 8), b):
                case['feature_keys'].append((8, chars[b0:b], surface))
                case['coefficients'].append(0.375)
        if len(c) == 2 and c[0][2] is not None and c[1][2] is not None:
            case['feature_keys'].append((8, chars[c[0][0]:c[0][1]], chars[c[1][0]:c[1][1]]))
            case['coefficients'].append(1.125)
    keys, coef = [], []
    for k, w in zip(case['feature_keys'], case['coefficients']):
        if tuple(k) not in {tuple(x) for x in keys}:
            keys.append(k)
            coef.append(w)
    case['feature_keys'], case['coefficients'] = keys, coef
    tagger, oracle = _objects(case)
    check_parity(tagger, oracle, sents, cons, (1, 5, 33))
    got = tagger.tag_batch(sents, beam_size=5, errors='none', constraints=[_as_items(c) for c in cons])
    forced = [w for seq in got if seq is not None for w in seq.sequences
              if w.tag0 in wp and w.word in wp[w.tag0] and w.tag0 in CONTEXTUAL and w.len == w.e - w.b]
    assert forced, 'no forced word on a best path'
    packed = tagger.tag_batch_packed(sents, 5, constraints=[_as_items(c) for c in cons])
    assert (packed[1]['flags'] & _native.LT_EDGE_FORCED).any()


@pytest.mark.gpu
def test_unknown_after_unknown_from_the_first_open_begin():
    """`None` spans without an edge, one right after the other: the reference's rule would leave the beam empty."""
    case = _case(3300, prefs=False)
    tagger, oracle = _objects(case)
    sents, cons = [], []
    for sent in case['sentences']:
        chars = sent.replace(' ', '')
        edges = oracle.lattice(sent)
        if len(chars) < 4 or not edges:
            continue
        spans = {(w[6], w[7]) for w in edges}
        free = [b for b in range(len(chars) - 1) if (b, b + 1) not in spans and (b + 1, b + 2) not in spans]
        if free:
            b = free[0]
            sents.append(sent)
            cons.append([(b, b + 1, None), (b + 1, b + 2, None)])
    assert sents
    check_parity(tagger, oracle, sents, cons, (1, 5))
    for seq, c in zip(tagger.tag_batch(sents, beam_size=5, constraints=[_as_items(x) for x in cons]), cons):
        assert seq is not None
        _check_satisfied([tuple(w) for w in seq.sequences], c)


@pytest.mark.gpu
def test_empty_constraints_are_no_constraints(monkeypatch, capfd):
    case = _case(3400, prefs=True)
    monkeypatch.setenv('LT_DEBUG', '1')
    tagger, _ = _objects(case)
    sents = case['sentences']
    for k in (1, 5, 20, 40):
        capfd.readouterr()
        plain = tagger.tag_batch_packed(sents, k)
        trace = capfd.readouterr().err
        assert 'beam kernel' in trace and 'constrained' not in trace
        empty = tagger.tag_batch_packed(sents, k, constraints=[[]] * len(sents))
        trace = capfd.readouterr().err
        assert 'constrained' in trace
        none = tagger.tag_batch_packed(sents, k, constraints=[None] * len(sents))
        for got in (empty, none):
            for a, b in zip(plain, got):
                assert a.tobytes() == b.tobytes()
        kb_plain = tagger.tag_batch_kbest(sents, k, errors='none')
        kb_empty = tagger.tag_batch_kbest(sents, k, errors='none', constraints=[[]] * len(sents))
        assert kb_plain == kb_empty


@pytest.mark.gpu
def test_mixed_batch_statuses():
    case = _case(3500, prefs=False)
    tagger, oracle = _objects(case)
    base = [s for s in case['sentences'] if oracle.lattice(s)][:6]
    nb = len(base)
    sents = base + ['\U0001F600abc', 'a\tb', 'x' * (tagger._engine.unit_limit + 1), case['sentences'][-1]] + base
    cons = _constraints_for(case, oracle, base, 35) + [None] * 4 + _constraints_for(case, oracle, base, 36)
    items = [None if c is None else _as_items(c) for c in cons]
    packed = tagger.tag_batch_packed(sents, 5, constraints=items)
    status = packed[3].tolist()
    assert status[nb:nb + 4] == [_native.LT_SENT_UNSUPPORTED_CHAR, _native.LT_SENT_BAD_SPACE, _native.LT_SENT_TOO_LONG,
                                 _native.LT_SENT_NO_EDGES]
    seqs = tagger.tag_batch(sents, 5, errors='none', constraints=items)
    for i in list(range(nb)) + list(range(nb + 4, 2 * nb + 4)):
        want = co.survivors(oracle, sents[i], 5, cons[i] or [])[0]
        assert [tuple(w) for w in seqs[i].sequences] == want.words and seqs[i].score == want.score


def _c_constraints(tagger, per_sent):
    rec = [(b, e, tag, (0, 0, 0)) for cons in per_sent for b, e, tag in cons]
    arr = np.array(rec, dtype=_native.CONSTRAINT_DTYPE) if rec else np.zeros(1, dtype=_native.CONSTRAINT_DTYPE)
    off = np.zeros(len(per_sent) + 1, dtype=np.int64)
    np.cumsum([len(c) for c in per_sent], out=off[1:])
    handle = ctypes.c_void_p()
    rc = tagger._lib.lt_constraints_create(tagger._tables.handle, len(per_sent), _native.ptr(arr), _native.ptr(off), ctypes.byref(handle))
    return rc, handle


@pytest.mark.gpu
def test_bad_constraint_status_through_the_c_abi():
    case = _case(3600, prefs=False)
    tagger, oracle = _objects(case)
    sents = [s for s in case['sentences'] if oracle.lattice(s)][:5]
    lens = [len(s.replace(' ', '')) for s in sents]
    per = [[] for _ in sents]
    per[1] = [(0, 1, _native.LT_NO_TAG), (lens[1] - 1, lens[1] + 1, _native.LT_NO_TAG)]
    rc, handle = _c_constraints(tagger, per)
    assert rc == _native.LT_OK
    try:
        _native.check(tagger._lib.lt_batch_set_constraints(tagger._batch, handle))
        packed = tagger._engine.tag_packed(sents, 5)
        _native.check(tagger._lib.lt_batch_set_constraints(tagger._batch, None))
    finally:
        tagger._lib.lt_constraints_destroy(handle)
    assert packed[3].tolist() == [0, _native.LT_SENT_BAD_CONSTRAINT, 0, 0, 0]
    assert packed[0][2] == packed[0][1]
    for i in (0, 2, 3, 4):
        want = oracle.tag(sents[i], 5)
        got = tagger._engine.unpack([sents[i]], (np.array([0, packed[0][i + 1] - packed[0][i]], dtype=np.int32),
                                                 packed[1][packed[0][i]:packed[0][i + 1]], packed[2][i:i + 1], packed[3][i:i + 1]))[0]
        assert [tuple(w) for w in got.sequences] == want.words and got.score == want.score


@pytest.mark.gpu
def test_big_batch_matches_sub_batches():
    case = _case(3700, prefs=False, n_sent=40)
    tagger, oracle = _objects(case)
    rng = random.Random(37)
    pool = [s for s in case['sentences'] if oracle.lattice(s)]
    n = 65_600
    sents = [pool[i % len(pool)] for i in range(n)]
    tags = _word_tags(case)
    memo = {}
    cons = []
    for i, s in enumerate(sents):
        if i % 3:
            cons.append(None)
            continue
        key = (s, i % 7)
        if key not in memo:
            memo[key] = random_constraints(random.Random(hash(key) & 0xFFFF), s, oracle.lattice(s), tags)
        cons.append(memo[key])
    items = [None if c is None else _as_items(c) for c in cons]
    whole = tagger.tag_batch(sents, 5, errors='none', lazy=False, constraints=items)
    for lo_, hi_ in ((0, 30_000), (30_000, 65_600)):
        part = tagger.tag_batch(sents[lo_:hi_], 5, errors='none', lazy=False, constraints=items[lo_:hi_])
        assert part == whole[lo_:hi_]
    for i in list(range(0, 40)) + list(range(65_500, 65_600)) + [rng.randrange(n) for _ in range(40)]:
        want = co.survivors(oracle, sents[i], 5, cons[i] or [])[0]
        assert [tuple(w) for w in whole[i].sequences] == want.words and whole[i].score == want.score, i


@pytest.mark.gpu
@pytest.mark.parametrize('env', [{'LT_EDGE_CAP': '16'}, {'LT_HIT_CAP': '8'}])
def test_grow_and_rerun(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    case = _case(3800, prefs=True)
    tagger, oracle = _objects(case)
    sents = case['sentences']
    cons = _constraints_for(case, oracle, sents, 38)
    check_parity(tagger, oracle, sents, cons, (5, 33))


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['lr', 'word'])
def test_lookup_modes(name):
    case = _case(3900, prefs=False)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, lookup=_checks.LOOKUPS[name](dictionary), score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs, lookup=name)
    sents = case['sentences']
    cons = _constraints_for(case, oracle, sents, 39)
    check_parity(tagger, oracle, sents, cons, (1, 5, 20))


@pytest.mark.gpu
def test_imported_lattice():
    case = _case(4000, prefs=True)
    tagger, oracle = _objects(case)
    sents = [s for s in case['sentences'] if oracle.lattice(s)]
    lattices = [[pkg.dictionary.Word(*w) for w in oracle.lattice(s)] for s in sents]
    cons = _constraints_for(case, oracle, sents, 40)
    check_parity(tagger, oracle, sents, cons, (5, 40), imported=lattices)


# ---- state --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_state_after_a_constrained_search():
    case = _case(4100, prefs=True)
    tagger, oracle = _objects(case)
    fresh, _ = _objects(case)
    sents = case['sentences']
    cons = [None if c is None else _as_items(c) for c in _constraints_for(case, oracle, sents, 41)]
    tagger.tag_batch(sents, 5, errors='none', constraints=cons)
    tagger.tag_batch_kbest(sents, 5, errors='none', constraints=cons)
    for k in (5, 33):
        assert tagger.tag_batch_packed(sents, k)[3].tolist() == fresh.tag_batch_packed(sents, k)[3].tolist()
        assert tagger.tag_batch(sents, k, errors='none', lazy=False) == fresh.tag_batch(sents, k, errors='none', lazy=False)
        assert tagger.tag_batch_kbest(sents, k, errors='none') == fresh.tag_batch_kbest(sents, k, errors='none')


@pytest.mark.gpu
def test_unconstrained_space_calls_refuse_a_constrained_search():
    case = _case(4200, prefs=False)
    tagger, oracle = _objects(case)
    engine = tagger._engine
    sents = [s for s in case['sentences'] if oracle.lattice(s)]
    golds = [oracle.tag(s, 5).words[1:-1] for s in sents]
    gold = engine.upload_paths([[pkg.dictionary.Word(*w) for w in g] for g in golds])
    cons = [[(0, 1)]] * len(sents)
    tagger.tag_batch_packed(sents, 5, constraints=cons)
    func = [type(f).__name__ for f in tagger.score_funcs.funcs].index('SimpleTrigramFeatureScore')
    with pytest.raises(_native.NativeLibraryError, match='constrained'):
        engine.evaluate(gold)
    with pytest.raises(_native.NativeLibraryError, match='constrained'):
        engine.perceptron_delta(gold, func)
    tagger.tag_batch_packed(sents, 5)
    engine.evaluate(gold)                       # an unconstrained search again: fine
    trainer = engine.trainer(sents, gold, func, 0, -np.ones(engine.tables.n_desc, dtype=np.int64), np.zeros(0))
    rc, handle = _c_constraints(tagger, [[] for _ in sents])
    assert rc == _native.LT_OK
    try:
        _native.check(tagger._lib.lt_batch_set_constraints(tagger._batch, handle))
        with pytest.raises(_native.NativeLibraryError, match='constraints bound'):
            trainer.step(0, len(sents), 5)
        # n_sent of the search differs from the bound set's
        with pytest.raises(_native.NativeLibraryError, match='constraint set has'):
            engine.tag_packed(sents[:-1], 5)
        _native.check(tagger._lib.lt_batch_set_constraints(tagger._batch, None))
    finally:
        tagger._lib.lt_constraints_destroy(handle)
        trainer.close()
        gold.close()


# ---- validation -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('items,match', [
    ([(2, 3), (0, 1)], 'sorted'),
    ([(0, 2), (1, 3)], 'overlaps'),
    ([(2, 2)], 'b < e'),
    ([(3, 1)], 'b < e'),
    ([(0, 9)], 'window'),
    ([(0, 99)], 'window'),
    ([(4, 11)], 'beyond'),
    ([(-1, 1)], 'b < e'),
    ([(0, 1, 'BOS')], 'not a tag'),
    ([(0, 1, 'EOS')], 'not a tag'),
    ([(0, 1, 'Unknown')], 'not a tag'),
    ([(0, 1, 'NoSuchTag')], 'unknown'),
    ([(0,)], 'not \\(b, e\\)'),
    ([(0.0, 1)], 'integers'),
])
def test_python_validation(items, match):
    case = _case(4300, prefs=False)
    tagger, _ = _objects(case)
    sent = 'ab cdefghij'            # 10 syllables
    launches = tagger.info()['launches']
    for call in (lambda: tagger.tag(sent, constraints=items), lambda: tagger.tag_batch([sent], constraints=[items]),
                 lambda: tagger.tag_batch_kbest([sent], constraints=[items]), lambda: tagger.tag_batch_packed([sent], constraints=[items])):
        with pytest.raises(ValueError, match=match):
            call()
    assert tagger.info()['launches'] == launches
    with pytest.raises(ValueError, match='constraint lists'):
        tagger.tag_batch([sent, sent], constraints=[[]])
    with pytest.raises(ValueError, match='debug'):
        tagger.tag(sent, debug=True, constraints=[])


@pytest.mark.gpu
def test_flatten_refuses_constraints():
    case = _case(4400, prefs=False)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, lookup=_checks.LOOKUPS['morpheme'](dictionary, flatten=True), score_funcs=funcs)
    for call in (lambda: tagger.tag_batch(['ab'], constraints=[[]]), lambda: tagger.tag_batch_kbest(['ab'], constraints=[[]]),
                 lambda: tagger.tag_batch_packed(['ab'], constraints=[[]])):
        with pytest.raises(ValueError, match='flatten'):
            call()


@pytest.mark.gpu
@pytest.mark.parametrize('per,match', [
    ([[(2, 3, 0xFF), (0, 1, 0xFF)]], 'sorted'),
    ([[(0, 2, 0xFF), (1, 3, 0xFF)]], 'sorted'),
    ([[(2, 2, 0xFF)]], 'syllables'),
    ([[(3, 1, 0xFF)]], 'syllables'),
    ([[(0, 9, 0xFF)]], 'syllables'),
    ([[(0, 1, 10)]], 'word tag'),
    ([[(0, 1, 11)]], 'word tag'),
    ([[(0, 1, 12)]], 'word tag'),
    ([[(0, 1, 40)]], 'word tag'),
])
def test_c_abi_validation(per, match):
    case = _case(4300, prefs=False)
    tagger, _ = _objects(case)
    rc, handle = _c_constraints(tagger, [[]] + per)
    assert rc == LT_ERR_INVALID and not handle.value
    message = tagger._lib.lt_last_error().decode()
    assert match in message and 'sentence 1, constraint' in message
    off = np.array([0, 1, 0], dtype=np.int64)
    arr = np.zeros(1, dtype=_native.CONSTRAINT_DTYPE)
    out = ctypes.c_void_p()
    assert tagger._lib.lt_constraints_create(tagger._tables.handle, 2, _native.ptr(arr), _native.ptr(off), ctypes.byref(out)) == LT_ERR_INVALID
    assert 'monotone' in tagger._lib.lt_last_error().decode()
