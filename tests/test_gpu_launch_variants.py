"""The host's launch choices, covered on purpose (csrc/lt_b200.cu: launch_beam, beam_plan, lattice_plan).

A. Batches past the single-launch limits: path offsets by the fused `pack_paths_scan` up to 64 K sentences, by the
   tiled three-kernel scan (`scan_u32`) and `pack_paths` beyond, k-best offsets by `scan_small` up to 64 K entries
   and by the tiled scan beyond, with a second 256-tile chunk in `scan_sums` past 524 288 entries.  Each big batch
   equals the same sentences tagged in sub-batches that take the small paths, and the oracle on the sentences
   around every tile and sub-batch boundary; `lt_perceptron_delta` and `lt_evaluate`, which read the packed paths
   on the device, agree with their sub-batch results.
B. Every beam size 1..64, best path and all survivors, on a tie-heavy case and on the (reg, trigram) program.
C. The planner's table: every kernel instantiation (and trail placement) that `beam_plan` / `lattice_plan` can
   pick, reached by an input built for it, read back from the `LT_DEBUG=1` launch trace and compared with the oracle.
"""

import random
import re

import numpy as np
import pytest

import lattice_based_tagger_b200 as pkg
from lattice_based_tagger_b200 import _native
from lattice_based_tagger_b200.engine import PackedSequences
from oracle import lattice_oracle as lo
from tests import _cases, _checks

pytestmark = pytest.mark.gpu

SCAN_TILE = 2048                    # scan.cuh: kScanTile, the entries one CTA of the tiled scan covers
SCAN_CHUNK = 256 * SCAN_TILE        # scan_sums scans the tile sums 256 at a time
SINGLE_LAUNCH_MAX = 64 * 1024       # scan.cuh: kPackScanMax (sentences), kScanSmallMax (scan entries)
SUB = 8192                          # best-path sub-batches: always the fused pack_paths_scan
KBEST_SUB = 1000                    # k-best sub-batches: at most 64 001 scan entries, always scan_small


# ---- A. batches past the single-launch limits ----------------------------------------------------------------

def _exact(pool, n):
    """A sentence of exactly `n` raw code units (spaces included) made of the pool's sentences."""
    out = ''
    i = 0
    while len(out) < n:
        out += pool[i % len(pool)] + ' '
        i += 1
    return out[:n]


@pytest.fixture(scope='module')
def big():
    case = _checks.make_case(4242, n_sent=400, prefs=False, max_sent_len=14)
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    pool = [s for s in case['sentences'] if s.strip()]
    no_hit = case['sentences'][-1]
    too_long = _exact(pool, tagger._engine.unit_limit + 1)
    func = [spec['kind'] for spec in case['funcs']].index('trigram')
    yield dictionary, funcs, tagger, pool, no_hit, too_long, func
    tagger.close()


def _big_batch(big, n, stride=1, seed=0):
    """`n` sentences of varied lengths (so that path offsets are no arithmetic progression).  Failures with no
    words — '', all spaces, no dictionary word — sit on both sides of every third `SCAN_TILE` boundary of the scan
    over `n * stride + 1` entries (stride = beam size for k-best offsets), one too-long sentence in the middle."""
    _, _, _, pool, no_hit, too_long, _ = big
    rng = random.Random(seed)
    sents = [pool[rng.randrange(len(pool))] for _ in range(n)]
    fails = ['', '   ', no_hit]
    j = 0
    for b in range(SCAN_TILE, n * stride + 1, SCAN_TILE):
        if (b // SCAN_TILE) % 3 == 0:
            for i in ((b - 1) // stride, b // stride):
                if i < n:
                    sents[i] = fails[j % len(fails)]
                    j += 1
    sents[n // 2 + 1] = too_long
    return sents


def _probes(n, stride, sub, seed):
    """Sentences within 2 of every tile and sub-batch boundary, the last one and 200 random ones."""
    idx = {n - 1}
    for b in range(SCAN_TILE, n * stride + 1, SCAN_TILE):
        idx.update(range(b // stride - 2, b // stride + 3))
    for b in range(sub, n, sub):
        idx.update(range(b - 2, b + 3))
    rng = random.Random(seed)
    idx.update(rng.randrange(n) for _ in range(200))
    return sorted(i for i in idx if 0 <= i < n)


def _bounds(n, sub):
    return [(lo_, min(n, lo_ + sub)) for lo_ in range(0, n, sub)]


def _same_bits(a, b):
    return np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


def _assert_best_concatenates(whole, parts, bounds):
    path_off, edges, scores, status = whole
    for (a, b), part in zip(bounds, parts):
        assert np.array_equal(path_off[a:b + 1] - path_off[a], part[0]), (a, b)
    assert path_off[0] == 0 and path_off[-1] == len(edges)
    assert _same_bits(edges, np.concatenate([p[1] for p in parts]))
    assert _same_bits(scores, np.concatenate([p[2] for p in parts]))
    assert np.array_equal(status, np.concatenate([p[3] for p in parts]))


def _check_best_with_oracle(engine, oracle, sents, packed, beam, idx):
    view = PackedSequences(engine, sents, packed, 'none')
    status = packed[3]
    for i in idx:
        if len(sents[i]) > engine.unit_limit:
            assert status[i] == _native.LT_SENT_TOO_LONG, i
            continue
        try:
            want = oracle.tag(sents[i], beam)
        except IndexError:
            assert status[i] == _native.LT_SENT_NO_EDGES, i
            continue
        seq = view[i]
        assert status[i] == _native.LT_SENT_OK and [tuple(w) for w in seq.sequences] == want.words, i
        assert seq.score == want.score, i


def _check_kbest_with_oracle(engine, oracle, sents, packed, beam, idx):
    n_best, off, edges, scores, status = packed
    for i in idx:
        sent = sents[i]
        if len(sent) > engine.unit_limit:
            assert status[i] == _native.LT_SENT_TOO_LONG and n_best[i] == 0, i
            continue
        try:
            want = oracle.survivors(sent, beam)
        except IndexError:
            assert status[i] == _native.LT_SENT_NO_EDGES and n_best[i] == 0, i
            continue
        assert status[i] == _native.LT_SENT_OK and n_best[i] == len(want), i
        for r in range(beam):
            j = i * beam + r
            if r >= len(want):
                assert off[j + 1] == off[j], (i, r)
                continue
            seq = engine._sequence(sent, edges[off[j]:off[j + 1]].tolist(), float(scores[j]))
            assert [tuple(w) for w in seq.sequences] == want[r].words, (i, r)
            assert seq.score == want[r].score, (i, r)


BEST_CASES = {'n65536': SINGLE_LAUNCH_MAX,             # fused pack_paths_scan at its limit
              'n65537': SINGLE_LAUNCH_MAX + 1,         # scan_u32: 33 tiles, the last one partial; pack_paths
              'n528484': SCAN_CHUNK + 2 * SCAN_TILE + 100}   # scan_sums: sentences in its second 256-tile chunk


@pytest.mark.parametrize('name', list(BEST_CASES))
def test_big_batch_best_paths(big, name):
    n = BEST_CASES[name]
    dictionary, funcs, tagger, *_ = big
    engine = tagger._engine
    sents = _big_batch(big, n, seed=n)
    beam = 5
    whole = engine.tag_packed(sents, beam)
    bounds = _bounds(n, SUB)
    parts = [engine.tag_packed(sents[a:b], beam) for a, b in bounds]
    _assert_best_concatenates(whole, parts, bounds)
    status = whole[3]
    assert {0, 1, 3} <= set(status.tolist()) and (np.diff(whole[0]) == 0).sum() > n // 4096
    _check_best_with_oracle(engine, lo.OracleTagger(dictionary, funcs), sents, whole, beam, _probes(n, 1, SUB, n))


KBEST_CASES = {'n4369_k15': (4369, 15),                # n * K + 1 = 65 536: scan_small at its limit
               'n1024_k64': (1024, 64),                # 65 537 entries: the first tiled k-best scan
               'n8200_k64': (8200, 64)}                # 524 801 entries: second scan_sums chunk


@pytest.mark.parametrize('name', list(KBEST_CASES))
def test_big_batch_all_survivors(big, name):
    n, beam = KBEST_CASES[name]
    assert (n * beam + 1 > SINGLE_LAUNCH_MAX) == (name != 'n4369_k15')
    dictionary, funcs, tagger, *_ = big
    engine = tagger._engine
    sents = _big_batch(big, n, stride=beam, seed=n)
    whole = engine.kbest_packed(sents, beam)
    bounds = _bounds(n, KBEST_SUB)
    parts = [engine.kbest_packed(sents[a:b], beam) for a, b in bounds]
    n_best, off, edges, scores, status = whole
    for (a, b), part in zip(bounds, parts):
        assert np.array_equal(off[a * beam:b * beam + 1] - off[a * beam], part[1]), (a, b)
    assert off[0] == 0 and off[-1] == len(edges)
    assert np.array_equal(n_best, np.concatenate([p[0] for p in parts]))
    assert _same_bits(edges, np.concatenate([p[2] for p in parts]))
    assert _same_bits(scores, np.concatenate([p[3] for p in parts]))
    assert np.array_equal(status, np.concatenate([p[4] for p in parts]))
    assert {0, 1, 3} <= set(status.tolist()) and (n_best == beam).any() and ((n_best > 0) & (n_best < beam)).any()
    _check_kbest_with_oracle(engine, lo.OracleTagger(dictionary, funcs), sents, whole, beam, _probes(n, beam, KBEST_SUB, n))


def _paths(engine, sents, packed):
    """Per sentence its path's `Word`s (no BOS / EOS; [] where the sentence failed)."""
    off = packed[0].tolist()
    records = packed[1].tolist()
    status = packed[3].tolist()
    return [engine.records_to_words(s.replace(' ', ''), records[off[i]:off[i + 1]]) if status[i] == 0 else []
            for i, s in enumerate(sents)]


def test_path_readers_on_the_largest_batch(big):
    """`lt_perceptron_delta` and `lt_evaluate` read path_off / path_out on the device: on the largest batch (tiled
    scan, second scan_sums chunk) they give what the sub-batches give.  The gold set mixes each sentence's own best
    path with its beam-1 path."""
    n = BEST_CASES['n528484']
    _, _, tagger, *_, func = big
    engine = tagger._engine
    sents = _big_batch(big, n, seed=n)
    beam = 5
    narrow = _paths(engine, sents, engine.tag_packed(sents, 1))
    own = _paths(engine, sents, engine.tag_packed(sents, beam))       # (the last search of the batch)
    gold = [own[i] if i % 2 == 0 else narrow[i] for i in range(n)]
    pathset = engine.upload_paths(gold)
    delta, differs, n_differ = engine.perceptron_delta(pathset, func)
    sent_class, counts, gold_scores, word_reason = engine.evaluate(pathset)
    pathset.close()
    assert 0 < n_differ == differs.sum() and delta.any()
    assert len(set(sent_class.tolist())) >= 3

    sub_delta = np.zeros_like(delta)
    sub_n_differ = 0
    sub = {'differs': [], 'class': [], 'counts': [], 'gold_scores': [], 'word_reason': []}
    for a, b in _bounds(n, SUB):
        engine.tag_packed(sents[a:b], beam)
        ps = engine.upload_paths(gold[a:b])
        d, df, nd = engine.perceptron_delta(ps, func)
        sub_delta += d
        sub_n_differ += nd
        sub['differs'].append(df)
        for key, value in zip(('class', 'counts', 'gold_scores', 'word_reason'), engine.evaluate(ps)):
            sub[key].append(value)
        ps.close()
    assert np.array_equal(delta, sub_delta) and n_differ == sub_n_differ
    assert np.array_equal(differs, np.concatenate(sub['differs']))
    assert np.array_equal(sent_class, np.concatenate(sub['class']))
    assert np.array_equal(counts, np.concatenate(sub['counts']))
    assert _same_bits(gold_scores, np.concatenate(sub['gold_scores']))
    assert np.array_equal(word_reason, np.concatenate(sub['word_reason']))


@pytest.mark.parametrize('knob,value', [('LT_SORT_BY_LENGTH', '0'), ('LT_PROLOGUE_CTAS', '1'), ('LT_PROLOGUE_CTAS', '32')])
def test_big_batch_work_order_knobs(big, monkeypatch, knob, value):
    """The 65 537-sentence batch (tiled scan, pack_paths) in input order and with other prologue shapes: the work
    order decides nothing but which warp takes which sentence.  (The knobs are read when the batch object is made.)"""
    dictionary, funcs, tagger, *_ = big
    sents = _big_batch(big, 65537, seed=65537)
    want = tagger._engine.tag_packed(sents, 5)
    monkeypatch.setenv(knob, value)
    other = pkg.Tagger(dictionary, score_funcs=funcs)
    got = other._engine.tag_packed(sents, 5)
    other.close()
    for a, b in zip(got, want):
        assert _same_bits(a, b)


# ---- B. every beam size ------------------------------------------------------------------------------------------

COARSE_GRID = {-1.0, -0.5, 0.0, 0.25, 0.5, 1.0}       # _cases.add_features' tie-making coefficient grid


# the score program each sweep case runs, as the LT_DEBUG trace names it
SWEEP_PROGRAMS = {'dense': 'other', 'reg_trigram': 'reg+trigram'}


def _sweep_case(name):
    if name == 'dense':
        # (SimpleTrigramFeatureScore, RegularizationScore) in that order: the generic-program instantiations
        case = _checks.dense_case(8)
        case['funcs'] = sorted(case['funcs'], key=lambda spec: spec['kind'] == 'reg')
        assert [spec['kind'] for spec in case['funcs']] == ['trigram', 'reg']
        _cases.add_features(case, _cases.observed_features(case, lo, seed=8), 8)
        assert set(case['coefficients']) <= COARSE_GRID
    else:
        # (RegularizationScore, SimpleTrigramFeatureScore) in that order: the instantiations specialised for it
        case = _cases.random_case(128, n_sent=10, features=True, prefs=False, max_sent_len=40)
        case['funcs'] = sorted(case['funcs'], key=lambda spec: spec['kind'] != 'reg')
        assert [spec['kind'] for spec in case['funcs']] == ['reg', 'trigram']
        _cases.add_features(case, _cases.observed_features(case, lo, seed=128), 128)
    dictionary, funcs = _cases.build_objects(case, pkg)
    with pytest.MonkeyPatch.context() as m:
        m.setenv('LT_DEBUG', '1')            # (read when the batch object is made: every new plan is traced)
        tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    return tagger, lo.OracleTagger(dictionary, funcs), case['sentences']


@pytest.fixture(scope='module')
def sweep():
    made = {}

    def get(name):
        if name not in made:
            made[name] = _sweep_case(name)
        return made[name]
    yield get
    for tagger, _, _ in made.values():
        tagger.close()


def _survivors(oracle, sent, beam):
    try:
        return oracle.survivors(sent, beam)
    except IndexError:
        return []


@pytest.mark.parametrize('name', ['dense', 'reg_trigram'])
@pytest.mark.parametrize('beam', range(1, 65))
def test_every_beam_size(sweep, capfd, name, beam):
    """Best path and all survivors at every K: rank counting (K <= 16), the 32-lane sorting network (17..32) and
    the two merged runs (33..64) change behaviour exactly at these boundaries.  The best-path search runs the
    generic-program instantiations on the dense case and the (reg, trigram) ones on the random case."""
    tagger, oracle, sents = sweep(name)
    capfd.readouterr()
    # the case does what it is built for: a full beam of K survivors, and at K = 16 / 32 / 64 (dense case) an
    # exact score tie between survivor K and survivor K + 1, decided by the generation order alone
    assert any(len(_survivors(oracle, s, beam)) == beam for s in sents)
    if name == 'dense' and beam in (16, 32, 64):
        wider = [_survivors(oracle, s, beam + 1) for s in sents]
        assert any(len(w) > beam and w[beam - 1].score == w[beam].score for w in wider)
    _checks.check_against_oracle(tagger, oracle, sents, (beam,))
    _checks.check_kbest(tagger, oracle, sents, (beam,))
    best_path_plans = {cell[3] for cell in _cells(capfd.readouterr().err) if cell[0] == 'beam' and not cell[5]}
    assert best_path_plans == {SWEEP_PROGRAMS[name]}


# ---- C. the planner's table ---------------------------------------------------------------------------------------

_BEAM_LINE = re.compile(r'\[lt\] beam kernel: beam (\d+) units (\d+)( \(sized instantiation\))?, .*, trail in (shared memory|HBM)'
                        r'(, reg\+trigram program)?(, k-best)?$')
_LATTICE_LINE = re.compile(r'\[lt\] lattice kernel( \(retry pass\))?: units (\d+)( \(sized instantiation\))? hcap (\d+)( any lookup)? ')


def _beam_kclass(beam, kbest):
    if not kbest and beam in (5, 10):
        return str(beam)
    if beam <= 16:
        return 'rank'
    if beam == 32 and not kbest:
        return '32'
    return 'sort' if beam <= 32 else 'merge'


def _cells(err):
    """The plans of an `LT_DEBUG=1` trace as table cells:
    ('beam', K class, units class, program, trail, k-best) / ('lattice', units class, hcap, lookup, pass)."""
    out = set()
    for line in err.splitlines():
        m = _BEAM_LINE.match(line)
        if m:
            beam, units, sized, trail, prog, kbest = m.groups()
            out.add(('beam', _beam_kclass(int(beam), bool(kbest)), int(units) if sized else 'generic',
                     'any' if kbest else ('reg+trigram' if prog else 'other'), 'smem' if trail == 'shared memory' else 'hbm',
                     bool(kbest)))
            continue
        m = _LATTICE_LINE.match(line)
        if m:
            retry, units, sized, hcap, any_lookup = m.groups()
            out.add(('lattice', int(units) if sized else 'generic', int(hcap) if sized else 'any',
                     'any' if any_lookup else 'morpheme', 'retry' if retry else 'main'))
            continue
        assert not line.startswith('[lt]'), line
    return out


HBM = {'LT_TRAIL_SMEM': '0'}
# beam_plan keeps the trail in shared memory only where that does not lower the beam kernel's residency, and
# LT_TRAIL_SMEM can only switch it off.  Worked out from beam_warp_smem and beam_plan's residency rule for every
# legal table (1..29 tags, 1..8 scorers, 0..8 of them trigram scorers) and array size:
_NEVER = 'unreachable for every table: the shared-memory trail always lowers residency here'
_FEW_SCORERS = ('unreachable with this case\'s two scorers: only some tables with 7 or 8 scorers, 5 or more of them '
                'trigram scorers, and 19 tags or more reach it')
_SMEM_TRAIL_UNREACHABLE = {
    # so beam_kernel<2, 5, 128, 1, 0, 1>, <2, 10, 64, 1, 0, 1> and <2, 10, 128, 1, 0, 1> are never launched
    ('5', 128, 'reg+trigram'): 'unreachable for every table with this program: the trail lowers residency here',
    ('10', 64, 'reg+trigram'): 'unreachable for every table with this program: the trail lowers residency here',
    ('10', 128, 'reg+trigram'): _NEVER,
    ('10', 128, 'other'): _NEVER,
    ('10', 'generic', 'reg+trigram'): _NEVER,
    ('10', 'generic', 'other'): _NEVER,
    ('5', 'generic', 'reg+trigram'): 'unreachable for every table with this program: it needs arrays of 3 768 units '
                                     'or more, and no table holds sentences beyond 3 016 units',
    # a program of two scorers behaves like (reg, trigram); more trigram scorers (more dense bytes) change that
    ('5', 128, 'other'): _FEW_SCORERS,
    ('10', 64, 'other'): _FEW_SCORERS,
    ('5', 'generic', 'other'): 'unreachable with this case\'s two scorers (as for (reg, trigram)); programs with more '
                               'trigram scorers reach it',
}


def _planner_table():
    """beam_plan / lattice_plan as explicit cells (lt_b200.cu), None where reachable, else why not.  Beams 5 and 10
    have instantiations for sentence arrays of 64 and 128 units (longest sentence <= 56 / <= 120 raw units); those
    for the (reg, trigram) program also fix at compile time where the back-pointers live.  The k-best search has
    one instantiation per selection mode, for any program.  The lattice kernel has sized instantiations for the
    default staging capacity (128) and twice that, a generic one per lookup family, and a retry pass for each."""
    table = {}
    for k in ('5', '10'):
        for units in (64, 128, 'generic'):
            for prog in ('reg+trigram', 'other'):
                table[('beam', k, units, prog, 'hbm', False)] = None
                table[('beam', k, units, prog, 'smem', False)] = _SMEM_TRAIL_UNREACHABLE.get((k, units, prog))
    for k in ('rank', 'sort', '32', 'merge'):
        for prog in ('reg+trigram', 'other'):
            for trail in ('smem', 'hbm'):
                table[('beam', k, 'generic', prog, trail, False)] = None
    for k in ('rank', 'sort', 'merge'):
        for trail in ('smem', 'hbm'):
            table[('beam', k, 'generic', 'any', trail, True)] = None
    for units in (64, 128):
        for hcap in (128, 256):
            table[('lattice', units, hcap, 'morpheme', 'main')] = None
    for lookup in ('morpheme', 'any'):
        for retry in ('main', 'retry'):
            table[('lattice', 'generic', 'any', lookup, retry)] = None
    return table


@pytest.fixture(scope='module')
def planner_case():
    case = _checks.make_case(4343, n_sent=24, prefs=False, max_sent_len=30)
    funcs = {'reg+trigram': sorted(case['funcs'], key=lambda spec: spec['kind'] != 'reg'),
             'other': sorted(case['funcs'], key=lambda spec: spec['kind'] == 'reg')}
    out = {}
    for prog, specs in funcs.items():
        dictionary, score_funcs = _cases.build_objects(dict(case, funcs=specs), pkg)
        out[prog] = (dictionary, score_funcs)
    pool = [s for s in case['sentences'] if s.strip()]
    return out, pool, case['sentences']


def _planner_inputs():
    """(program, lookup, knobs, longest sentence in raw units, beam, k-best): each reaches a cell no other one
    reaches.  Beams 5 and 10 at the class boundaries 56 / 57 and 120 / 121; the generic classes keep the trail in
    shared memory for the shortest arrays; LT_HIT_CAP = 256 selects the larger staging capacity, LT_HIT_CAP = 8
    sends eojeols to the retry pass."""
    inputs = []
    for prog in ('reg+trigram', 'other'):
        # (beam 5 at 56 and 57 units with the (reg, trigram) program: the LT_HIT_CAP = 256 inputs below)
        inputs += [(prog, 'morpheme', {}, 56, 5, False), (prog, 'morpheme', {}, 57, 5, False)] if prog == 'other' else []
        inputs += [(prog, 'morpheme', HBM, 56, 5, False), (prog, 'morpheme', {}, 121, 5, False),
                   (prog, 'morpheme', {}, 56, 10, False), (prog, 'morpheme', {}, 120, 10, False),
                   (prog, 'morpheme', {}, 121, 10, False)]
        for k_smem, k_hbm in ((3, 3), (24, 20), (32, 32), (33, 40)):
            # (beam 3 with the (reg, trigram) program and its trail in shared memory: the LT_HIT_CAP = 8 inputs)
            inputs += [(prog, 'morpheme', {}, 8, k_smem, False)] if (prog, k_smem) != ('reg+trigram', 3) else []
            inputs += [(prog, 'morpheme', HBM, 40, k_hbm, False)]
    for k_smem, smem_longest, k_hbm in ((3, 8, 12), (32, 8, 17), (64, 16, 64)):
        inputs += [('other', 'morpheme', {}, smem_longest, k_smem, True), ('other', 'morpheme', HBM, 40, k_hbm, True)]
    inputs += [('reg+trigram', 'morpheme', {'LT_HIT_CAP': '256'}, 56, 5, False),
               ('reg+trigram', 'morpheme', {'LT_HIT_CAP': '256'}, 57, 5, False),
               ('reg+trigram', 'morpheme', {'LT_HIT_CAP': '8'}, 40, 3, False),
               ('reg+trigram', 'lr', {'LT_HIT_CAP': '8'}, 40, 3, False)]
    return inputs


def test_planner_table(planner_case, monkeypatch, capfd):
    """Every reachable cell of the planner's table is reached by an input built for it and computes what the oracle
    does; the cells visited are exactly the reachable cells, and no input is redundant."""
    objects, pool, sents = planner_case
    dense = ''.join(pool).replace(' ', '')
    visited = []
    capfd.readouterr()
    for prog, lookup, knobs, longest, beam, kbest in _planner_inputs():
        dictionary, funcs = objects[prog]
        # the retry inputs need eojeols with more hits than the tiny staging area holds: no spaces
        batch = [dense[:longest] if 'LT_HIT_CAP' in knobs and knobs['LT_HIT_CAP'] == '8' else _exact(pool, longest)]
        batch += [s for s in sents if len(s) < longest][:8]
        assert max(len(s) for s in batch) == longest
        with monkeypatch.context() as m:
            m.setenv('LT_DEBUG', '1')
            for key, value in knobs.items():
                m.setenv(key, value)
            tagger = pkg.Tagger(dictionary, score_funcs=funcs,
                                **({'lookup': _checks.LOOKUPS[lookup](dictionary)} if lookup != 'morpheme' else {}))
            oracle = lo.OracleTagger(dictionary, funcs, lookup=lookup)
            if kbest:
                engine = tagger._engine
                _check_kbest_with_oracle(engine, oracle, batch, engine.kbest_packed(batch, beam), beam, range(len(batch)))
            else:
                _checks.check_against_oracle(tagger, oracle, batch, (beam,))
            tagger.close()
        visited.append(((prog, lookup, knobs, longest, beam, kbest), _cells(capfd.readouterr().err)))
    table = _planner_table()
    reached = set().union(*(cells for _, cells in visited))
    want = {cell for cell, why in table.items() if why is None}
    assert reached == want, ('not reached', sorted(map(str, want - reached)), 'outside the table', sorted(map(str, reached - want)))
    for i, (name, cells) in enumerate(visited):
        others = set().union(*(c for j, (_, c) in enumerate(visited) if j != i))
        assert cells - others, name          # removing this input would leave a cell unreached


def test_sentence_at_the_unit_limit(planner_case):
    """A sentence of exactly `unit_limit` raw units (the longest both kernels hold) is tagged at beams 1, 5 and 64;
    one unit more is LT_SENT_TOO_LONG."""
    objects, pool, sents = planner_case
    dictionary, funcs = objects['reg+trigram']
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    limit = tagger._engine.unit_limit
    at_limit = _exact(pool, limit)
    assert len(at_limit) == limit
    _checks.check_against_oracle(tagger, lo.OracleTagger(dictionary, funcs), [at_limit, sents[0]], (1, 5, 64))
    got = tagger.tag_batch([_exact(pool, limit + 1), sents[0]], beam_size=5, errors='none')
    assert list(got.status) == [_native.LT_SENT_TOO_LONG, _native.LT_SENT_OK] and got[0] is None
    tagger.close()
