"""`lt_evaluate` (csrc/evaluate.cuh), `Tagger.evaluate` and `trainer.evaluate` against a host reference written
here: predictions from the search itself (`tag_batch` / the k-best and imported-lattice searches), lattices from
`lookup_batch` (= `lattice_batch`) or the imported words, the window and unknown-word rules of the oracle's
`beam_search`, and image scores from the oracle's `ScoreProgram.increment`.  Every per-sentence output is
compared with ==.

The `check_*` functions take their sizes as arguments so that they can run through the SIMT emulator as well."""

import math
import random
from collections import Counter

import numpy as np
import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native, synth
from lattice_based_tagger_b200.dictionary import Word
from lattice_based_tagger_b200.dictionary.text import text_to_words
from lattice_based_tagger_b200.tagger.evaluation import ordered
from lattice_based_tagger_b200.trainer.train import _surface
from oracle import lattice_oracle as lo
from tests import _cases, _golden
from tests.test_gpu_path_edges import _mixed_batch, _tags, _trained_tagger, change_field
from tests.test_gpu_paths import BOS, PAIRS, _dense_features, _eos, _oracle_score

pytestmark = pytest.mark.gpu

N = _native
CORRECT, FAILED, UNREACHABLE, SEARCH, MODEL = (N.LT_EVAL_CORRECT, N.LT_EVAL_FAILED, N.LT_EVAL_UNREACHABLE,
                                               N.LT_EVAL_SEARCH_ERROR, N.LT_EVAL_MODEL_ERROR)
OK, TILING, WINDOW, NOT_IN, UNK_UNK, UNCHECKED = (N.LT_GOLD_OK, N.LT_GOLD_BREAKS_TILING, N.LT_GOLD_BEYOND_WINDOW,
                                                 N.LT_GOLD_NOT_IN_LATTICE, N.LT_GOLD_UNK_AFTER_UNK, N.LT_GOLD_UNCHECKED)
UNK = 'Unknown'


def _full(w):
    return (w.b, w.e, w.tag0, w.tag1, w.morph0, w.morph1)


def _units(words):
    return sum(1 + (w.tag1 is not None) for w in words)


def reference(program, sents, golds, predicted, lattices):
    """Per sentence (class, 8 counts, image score or None, reason codes) by the definitions of lt_evaluate.
    `predicted[i]`: the search's best path (None when its status is not OK); `lattices[i]`: the lattice's words
    in lattice order (grouped by end, then begin, a span's edges in their order)."""
    out = []
    for sent, gold, pred, lattice in zip(sents, golds, predicted, lattices):
        chars = sent.replace(' ', '')
        n = len(chars)
        G = list(gold[1:-1])
        ok = pred is not None
        P = list(pred.sequences[1:-1]) if ok else []
        by_b = {g.b: g for g in G}
        seg = tag = full = unit = 0
        for p in P:
            g = by_b.get(p.b)
            if g is None or g.e != p.e:
                continue
            seg += 1
            same_tags = (p.tag0, p.tag1) == (g.tag0, g.tag1)
            tag += same_tags
            full += same_tags and (p.morph0, p.morph1) == (g.morph0, g.morph1)
            unit += (p.morph0, p.tag0) == (g.morph0, g.tag0)
            unit += p.tag1 is not None and (p.morph1, p.tag1) == (g.morph1, g.tag1)
        counts = [len(G), len(P), seg, tag, full, _units(G), _units(P), unit]
        reasons, image = [], []
        if ok:
            spans = {}
            for w in lattice or ():
                spans.setdefault((w.b, w.e), []).append(w)
            for j, g in enumerate(G):
                prev_e = G[j - 1].e if j else 0
                if g.b != prev_e or g.e > n or (j == len(G) - 1 and g.e != n):
                    reasons.append(TILING)
                    continue
                if g.e - g.b > lo.WINDOW:
                    reasons.append(WINDOW)
                    continue
                cands = spans.get((g.b, g.e), [])
                hit = next((w for w in cands if _full(w) == _full(g)), None)
                sub = chars[g.b:g.e]
                if hit is None and not cands and (g.tag0, g.tag1, g.morph0, g.morph1) == (UNK, None, sub, None):
                    hit = Word(sub, sub, None, UNK, None, g.e - g.b, g.b, g.e, False)       # beam.py:36-38
                r = OK if hit is not None else NOT_IN
                if r == OK and g.tag0 == UNK and j and G[j - 1].tag0 == UNK and g.b != max(0, g.e - lo.WINDOW):
                    r = UNK_UNK                                                            # beam.py:44-45
                reasons.append(r)
                image.append(hit)
            reach = all(r == OK for r in reasons) and (len(G) > 0 or n == 0)
        else:
            reasons = [UNCHECKED] * len(G)
            reach = False
        score = _oracle_score(program, [BOS] + image + [_eos(n)]) if reach else None
        exact = ok and len(P) == len(G) and full == len(G)
        if not ok:
            cls = FAILED
        elif exact:
            cls = CORRECT
        elif not reach:
            cls = UNREACHABLE
        else:
            cls = SEARCH if score > pred.score else MODEL
        out.append((cls, counts, score, reasons))
    return out


def _nan_none(xs):
    return [None if math.isnan(x) else x for x in xs]


def assert_equal(got, want):
    """got: (sent_class, counts, gold_scores, word_reason as one array per sentence) from the device."""
    sent_class, counts, gold_scores, reasons = got
    assert sent_class.tolist() == [w[0] for w in want]
    assert counts.tolist() == [w[1] for w in want]
    assert _nan_none(gold_scores.tolist()) == [w[2] for w in want]
    assert [r.tolist() for r in reasons] == [w[3] for w in want]


def _search(tagger, batch, beam_size, search, imported=None):
    """One kind of search on the batch; -> its best path per sentence (Sequence or None)."""
    engine = tagger._engine
    if search in ('tag', 'rerun'):
        return engine.unpack(batch, engine.tag_packed(batch, beam_size), 'none')
    packed = engine.kbest_packed(batch, beam_size, imported=imported)
    kept = engine.unpack_kbest(batch, packed, beam_size, 'none', engine._imported_words if imported is not None else None)
    return [seqs[0] if seqs else None for seqs in kept]


def check(tagger, batch, golds, beam_size, search='evaluate', imported=None):
    """The device's evaluation of `golds` after one search against the host reference; -> the reference."""
    engine = tagger._engine
    program = lo.ScoreProgram(tagger.score_funcs)
    lattices = imported if imported is not None else tagger.eojeol_lookup.lookup_batch(batch, errors='none')
    if search == 'evaluate':
        predicted = list(tagger.tag_batch(batch, beam_size, errors='none'))
        ev = tagger.evaluate(batch, golds, beam_size)
        got = (ev.sent_class, ev.counts, ev.gold_scores, ev.word_reason)
        assert _nan_none(ev.predicted_scores.tolist()) == [None if p is None else p.score for p in predicted]
    else:
        pathset = engine.upload_paths([g[1:-1] for g in golds])
        predicted = _search(tagger, batch, beam_size, search, imported)
        sent_class, counts, gold_scores, word_reason = engine.evaluate(pathset)
        off = pathset.path_off.tolist()
        got = (sent_class, counts, gold_scores, [word_reason[off[i]:off[i + 1]] for i in range(len(batch))])
        pathset.close()
    if imported is not None:
        # the lattice order of an import: by end, then begin, then the order given (Engine.import_lattice)
        lattices = [sorted((w for w in ws if 0 <= w.b < w.e), key=lambda w: (w.e, w.b)) for ws in imported]
    want = reference(program, batch, golds, predicted, lattices)
    assert_equal(got, want)
    return want


def classes(want):
    return {w[0] for w in want}


def reasons(want):
    return {r for w in want for r in w[3]}


# ---- the search's own best paths: every sentence correct ------------------------------------------------------

@pytest.mark.parametrize('name', ['demo_morph', 'base_c1', 'random_1000', 'random_1003', 'random_1007'])
def test_own_best_paths_are_correct(name):
    payload = _golden.load(name)
    case = payload['case']
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs, k3_first=payload['k3_first'])
    pairs = [(s, q) for s, q in zip(case['sentences'], tagger.tag_batch(case['sentences'], 5, errors='none')) if q is not None]
    sents, golds = [s for s, _ in pairs], [list(q.sequences) for _, q in pairs]
    want = check(tagger, sents, golds, 5)
    assert classes(want) == {CORRECT}
    assert all(w[2] == q.score for w, (_, q) in zip(want, pairs))
    ev = tagger.evaluate(sents, golds, 5)
    assert ev.class_counts['correct'] == len(sents) and ev.exact.all()
    for level in ('seg', 'tag', 'full', 'morph'):
        assert ev.precision(level) == ev.recall(level) == ev.f1(level) == 1.0
    assert ev.missing_words() == Counter()


@pytest.fixture(scope='module')
def c2_sample():
    cfg, dictionary, sents = synth.build_workload('c2', n_sent=300)
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


def test_c2_own_paths_and_perceptron_agree(c2_sample):
    """Gold = the search's own best paths on a C2 sample: every tagged sentence correct, image score = search
    score; then gold = k-best survivors and near misses, where `exact` is the negation of lt_perceptron_delta's
    `differs` on the same batch."""
    cfg, dictionary, funcs, sents = c2_sample
    beam = cfg['beam']
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    best = list(tagger.tag_batch(sents, beam, errors='none'))
    ok = [(s, q) for s, q in zip(sents, best) if q is not None]
    want = check(tagger, [s for s, _ in ok], [list(q.sequences) for _, q in ok], beam)
    assert classes(want) == {CORRECT}
    assert [w[2] for w in want] == [q.score for _, q in ok]
    rng = random.Random(7)
    kept = tagger.tag_batch_kbest(sents, beam, errors='none')
    golds = []
    for sent, seqs in zip(sents, kept):
        if not seqs:
            golds.append([BOS, _eos(len(sent.replace(' ', '')))])
        elif rng.random() < 0.5:
            golds.append(list(seqs[rng.randrange(len(seqs))].sequences))
        else:
            words = seqs[0].sequences
            n = len(words) - 2
            golds.append(change_field(words, rng.randrange(n), rng.choice(['tag0', 'morph0', 'morph1', 'len']), _tags(tagger))
                         if n > 1 else list(words))
    engine = tagger._engine
    pathset = engine.upload_paths([g[1:-1] for g in golds])
    engine.tag_packed(sents, beam)
    _, differs, _ = engine.perceptron_delta(pathset, 1)
    sent_class, _, _, _ = engine.evaluate(pathset)
    pathset.close()
    assert (sent_class == CORRECT).tolist() == (~differs).tolist()
    want = check(tagger, sents, golds, beam)
    assert {CORRECT, MODEL, UNREACHABLE} <= classes(want)


def test_lower_survivors_are_model_errors(c2_sample):
    cfg, dictionary, funcs, sents = c2_sample
    beam = cfg['beam']
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    batch, golds = [], []
    for sent, seqs in zip(sents, tagger.tag_batch_kbest(sents, beam, errors='none')):
        for seq in (seqs or [])[1:]:
            if seq.sequences != seqs[0].sequences:
                batch.append(sent)
                golds.append(list(seq.sequences))
    want = check(tagger, batch, golds, beam)
    assert MODEL in classes(want) and classes(want) <= {MODEL, CORRECT}


def test_beam_one_against_beam_64_finds_search_errors(c2_sample):
    cfg, dictionary, funcs, sents = c2_sample
    wide = pkg.Tagger(dictionary, score_funcs=funcs)
    best = list(wide.tag_batch(sents, 64, errors='none'))
    wide.close()
    ok = [(s, q) for s, q in zip(sents, best) if q is not None]
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    want = check(tagger, [s for s, _ in ok], [list(q.sequences) for _, q in ok], 1)
    assert SEARCH in classes(want) and CORRECT in classes(want)
    ev = tagger.evaluate([s for s, _ in ok], [q.sequences for _, q in ok], 1)
    searched = ev.sent_class == SEARCH
    assert (ev.gold_scores[searched] > ev.predicted_scores[searched]).all()


# ---- one edit per reason code -----------------------------------------------------------------------------

LONG_NOUN = '가나다라마바사아자차'          # 10 syllables: a dictionary word beyond the window
OUTSIDE = '뷁쀍뷁쀍뷁쀍뷁쀍뷁쀍뷁쀍'         # syllables without any dictionary edge


def _edit_tagger():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    dictionary.tag_to_morphs['Noun'] = set(dictionary.tag_to_morphs['Noun']) | {LONG_NOUN}
    reg = pkg.beam.RegularizationScore(unknown_penalty=-0.1, known_preference=0.5, syllable_penalty=-0.2)
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    return dictionary, reg, probe


def _unk(chars, b, e):
    return Word(chars[b:e], chars[b:e], None, UNK, None, e - b, b, e, False)


def edit_workload(tagger, rng):
    """(sentences, gold paths): the prediction itself, then one edit per reason code, and gold unknown words at
    spans without any edge (reachable) next to ones the window or the unknown-after-unknown rule excludes."""
    sents = [_surface(w) for w, _ in PAIRS[:5]]
    predicted = tagger.tag_batch(sents, 5)
    tags = _tags(tagger)
    batch, golds = [], []
    for sent, seq in zip(sents, predicted):
        words = list(seq.sequences)
        n = len(words) - 2
        lemma = [i for i, w in enumerate(words[1:-1]) if w.tag1 is not None]
        edits = [words,
                 words[:2] + words[3:] if n > 2 else words,                      # a gap: breaks the tiling
                 words[:-2] + [words[-2]._replace(e=words[-2].e + 1), words[-1]],  # beyond the last syllable
                 change_field(words, rng.randrange(n), 'tag0', tags)]
        if lemma:
            edits.append(change_field(words, lemma[0], 'morph1', tags))          # morph1 alone differs
            edits.append(change_field(words, lemma[0], 'morph0', tags))
        batch += [sent] * len(edits)
        golds += edits
    # a dictionary word of 10 syllables (the lattice has it) and the unknown-word rules
    long_sent = LONG_NOUN + '는 노래'
    chars = long_sent.replace(' ', '')
    batch.append(long_sent)
    golds.append([BOS, Word(LONG_NOUN, LONG_NOUN, None, 'Noun', None, 10, 0, 10, False),
                  Word('는', '는', None, 'Josa', None, 1, 10, 11, False), Word('노래', '노래', None, 'Noun', None, 2, 11, 13, False),
                  _eos(13)])
    song = '노래 ' + OUTSIDE
    chars = song.replace(' ', '')
    noun = Word('노래', '노래', None, 'Noun', None, 2, 0, 2, False)
    m = len(chars)
    for cut in ([2, 6, m], [2, 4, 6, m], [2, 7, m], [2, 5, m], [2, m], [2, 10]):
        # [2, 6, m]: an unknown word of 8 right after an unknown word, from the window's earliest begin
        words = [noun] + [_unk(chars, b, e) for b, e in zip(cut, cut[1:])]
        if cut[-1] != m:
            words.append(_unk(chars, cut[-1], m))
        batch.append(song)
        golds.append([BOS] + words + [_eos(m)])
    batch.append(song)
    golds.append([BOS, _unk(chars, 0, 2), _unk(chars, 2, 10), _unk(chars, 10, m), _eos(m)])     # an Unk where edges exist
    return batch, golds


def test_each_reason_code():
    dictionary, reg, probe = _edit_tagger()
    rng = random.Random(3)
    batch, golds = edit_workload(probe, rng)
    paths = golds + [list(q.sequences) for q in probe.tag_batch(batch, 5)]
    probe.close()
    funcs = [reg] + _dense_features(paths, rng)
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(*funcs))
    assert any(w.b == 0 and w.e == 10 for w in tagger.eojeol_lookup.lookup_batch([LONG_NOUN + '는 노래'])[0])
    want = check(tagger, batch, golds, 5)
    assert reasons(want) >= {OK, TILING, WINDOW, NOT_IN, UNK_UNK}
    assert {CORRECT, UNREACHABLE} <= classes(want)
    song = [w for w, s in zip(want, batch) if s == '노래 ' + OUTSIDE]
    assert [w[3] for w in song] == [[OK] * 3, [OK, OK, UNK_UNK, OK], [OK, OK, UNK_UNK], [OK, OK, WINDOW], [OK, WINDOW],
                                    [OK, OK, UNK_UNK], [NOT_IN, OK, UNK_UNK]]
    assert song[0][0] != UNREACHABLE
    want = check(tagger, batch, golds, 5, search='tag')
    ev = tagger.evaluate(batch, golds, 5)
    missing = Counter()
    for gold, w in zip(golds, want):
        for g, r in zip(gold[1:-1], w[3]):
            if r == NOT_IN:
                missing[g.morph0, g.tag0, g.morph1, g.tag1] += 1
    assert ev.missing_words() == missing and len(missing) >= 3


# ---- long paths, sentences the search does not tag, the launch's warps -------------------------------------

def long_edits(words, tags, rng, positions=(0, 31, 32, 33, 63, 64)):
    """One edit of each kind at each position and at the last word: a field, a gap, two words merged, a
    boundary moved."""
    n = len(words) - 2
    out = []
    for pos in sorted({p for p in positions if p < n} | {n - 1}):
        i = pos + 1
        out.append(change_field(words, pos, rng.choice(['tag0', 'tag1', 'morph0', 'morph1']), tags))
        out.append(words[:i] + words[i + 1:])
        if i + 1 < len(words) - 1:
            x, y = words[i], words[i + 1]
            out.append(words[:i] + [_unk_merge(x, y)] + words[i + 2:])
        if n > 1:
            out.append(change_field(words, pos, 'boundary', tags))
    return out


def _unk_merge(x, y):
    s = x.word + y.word
    return Word(s, s, None, UNK, None, y.e - x.b, x.b, y.e, False)


def check_long_paths(seed, n_long=2, min_syllables=200, beam_size=5):
    tagger, funcs, case, sents, rng = _trained_tagger(seed, n_long, min_syllables)
    predicted = tagger.tag_batch(sents, beam_size, errors='none')
    assert max(len(s.sequences) for s in predicted) > 66
    tags = _tags(tagger)
    batch, golds = [], []
    for sent, seq in zip(sents, predicted):
        edits = [list(seq.sequences)] + [e for e in long_edits(list(seq.sequences), tags, rng) if ordered([e[1:-1]])]
        batch += [sent] * len(edits)
        golds += edits
    want = check(tagger, batch, golds, beam_size)
    assert {CORRECT, UNREACHABLE} <= classes(want)
    assert {OK, TILING, NOT_IN} <= reasons(want)


@pytest.mark.parametrize('seed', [31, 32])
def test_long_paths_across_chunks(seed):
    check_long_paths(seed)


def check_after_search(search, n_long=2, min_syllables=150, beam_size=4, reps=1):
    """The mixed batch of tests/test_gpu_path_edges.py (long sentences with their prediction, a near miss and a
    tiling; too long, empty, spaces only, no dictionary edge) after each kind of search."""
    tagger, funcs, case, sents, rng = _trained_tagger(41, n_long, min_syllables, two_trigrams=True)
    batch, golds = _mixed_batch(tagger, case, sents, rng, beam_size, too_long=search != 'rerun')
    batch, golds = batch * reps, golds * reps
    imported = None
    if search == 'imported':
        # every edge twice, the copy with another Word.len (another score): the image takes the first
        imported = [(ws or []) + [w._replace(len=w.len + 1) for w in ws or []]
                    for ws in tagger.eojeol_lookup.lookup_batch(batch, errors='none')]
    want = check(tagger, batch, golds, beam_size, search if search != 'public' else 'evaluate', imported)
    if search == 'rerun':
        assert tagger.info()['reruns'] > 0
    assert {CORRECT, FAILED, UNREACHABLE} <= classes(want)
    assert {OK, UNCHECKED, TILING} <= reasons(want)
    empty = [w for s, w in zip(batch, want) if not s.strip()]
    assert {w[0] for w in empty} == {CORRECT, UNREACHABLE}
    return tagger, want


@pytest.mark.parametrize('search', ['public', 'tag', 'kbest', 'imported', 'rerun'])
def test_after_each_search(monkeypatch, search):
    if search == 'rerun':
        monkeypatch.setenv('LT_HIT_CAP', '8')
        monkeypatch.setenv('LT_EDGE_CAP', '16')
    check_after_search(search)


def test_more_sentences_than_warps():
    tagger, _ = check_after_search('tag', n_long=1, min_syllables=70)
    sm = tagger.info()['sm_count']
    check_after_search('tag', n_long=1, min_syllables=70, reps=-(-2 * sm * 64 // 12) + 1)


# ---- the trainer's corpus, errors ----------------------------------------------------------------------------

def test_trainer_evaluate():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    reg = pkg.beam.RegularizationScore(unknown_penalty=-0.1, known_preference=-0.3, syllable_penalty=0.0)
    pairs = list(PAIRS) + [('노래  아이', 'malformed')]
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    ev = pkg.trainer.evaluate(pairs, tagger)
    # PAIRS[5] names a tag the tables lack, PAIRS[7] is outside the BMP, the last pair does not parse
    assert ev.not_evaluated == [5, 7, 8]
    assert ev.indices == [0, 1, 2, 3, 4, 6]
    sents = [_surface(PAIRS[i][0]) for i in ev.indices]
    golds = [text_to_words(*PAIRS[i]) for i in ev.indices]
    want = check(tagger, sents, golds, 5)
    assert [w[0] for w in want] == ev.sent_class.tolist()
    assert FAILED in classes(want) and len(ev) == 6
    assert ev.missing_words() == Counter({(g.morph0, g.tag0, g.morph1, g.tag1): 1 for gold, w in zip(golds, want)
                                          for g, r in zip(gold[1:-1], w[3]) if r == NOT_IN})
    gold, predicted, matched = ev.totals('full')
    assert ev.precision('full') == matched / predicted and ev.recall('full') == matched / gold
    assert ev.f1('full') == 2 * matched / (gold + predicted)
    wide = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg), extra_tags=['Suffix'])
    assert pkg.trainer.evaluate(pairs, wide).not_evaluated == [7, 8]
    flat = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg),
                      lookup=pkg.dictionary.lookup.MorphemeLookup(dictionary, flatten=True))
    with pytest.raises(ValueError):
        pkg.trainer.evaluate(pairs, flat)
    with pytest.raises(ValueError):
        flat.evaluate(sents, golds)


def test_malformed_input():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    reg = pkg.beam.RegularizationScore()
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    gold = text_to_words(*PAIRS[1])
    sent = _surface(PAIRS[1][0])
    for bad in ([gold[:1] + [gold[2], gold[1]] + gold[3:]], [gold[:1] + [gold[1]._replace(e=gold[1].b)] + gold[2:]]):
        with pytest.raises(ValueError):
            tagger.evaluate([sent], bad)
    with pytest.raises(ValueError):
        tagger.evaluate([sent, sent], [gold])
    with pytest.raises(ValueError):
        tagger.evaluate(['노래 \U0001F600'], [[BOS, _eos(2)]])


def test_c_abi_rejects_bad_calls():
    dictionary = pkg.dictionary.DemoMorphemeDictionary()
    reg = pkg.beam.RegularizationScore()
    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    other = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    lib, batch, engine = tagger._lib, tagger._batch, tagger._engine
    golds = [text_to_words(*PAIRS[i]) for i in range(2)]
    sents = [_surface(PAIRS[i][0]) for i in range(2)]
    cls = np.zeros(2, dtype=np.uint8)
    counts = np.zeros((2, 8), dtype=np.int32)
    scores = np.zeros(2)
    reason = np.zeros(64, dtype=np.uint8)

    def call(pathset, cls=cls):
        return lib.lt_evaluate(batch, pathset.handle, _native.ptr(cls), _native.ptr(counts), _native.ptr(scores), _native.ptr(reason))
    invalid = 1
    good = engine.upload_paths([g[1:-1] for g in golds])
    assert call(good) == invalid                                    # no search yet
    engine.tag_packed(sents, 5)
    assert lib.lt_evaluate(batch, good.handle, None, None, None, None) == invalid
    assert call(other._engine.upload_paths([g[1:-1] for g in golds])) == invalid
    assert call(engine.upload_paths([golds[0][1:-1]])) == invalid
    swapped = [golds[0][1:-1], [golds[1][2], golds[1][1]] + golds[1][3:-1]]
    assert call(engine.upload_paths(swapped)) == invalid
    empty_word = [golds[0][1:-1], [golds[1][1]._replace(e=golds[1][1].b)] + golds[1][2:-1]]
    assert call(engine.upload_paths(empty_word)) == invalid
    assert call(good) == 0
    full = cls.copy()
    assert lib.lt_evaluate(batch, good.handle, _native.ptr(cls), None, None, None) == 0
    assert cls.tolist() == full.tolist() == tagger.evaluate(sents, golds).sent_class.tolist()
