"""Evaluation against gold paths on the C2 workload: `lt_evaluate` after a decode against the host loop that
computes the same numbers from `tag_batch`, `lattice_batch` and `score_paths`.

The gold corpus is built as in train_epoch.py: the best paths of a teacher tagger (same features, other seeded
weights), kept where every word stays inside one eojeol, with one word in twelve given a morpheme the dictionary
lacks (unreachable sentences).  The evaluated tagger has the features' own weights, so that most reachable
sentences are model errors.  Asserts that both ways give the same per-sentence classes,
counts, image scores and reason codes, and prints one JSON line: the decode, the evaluation step and the host
loop (host clock around calls that end in a stream synchronise), and the GPU name and power limit read in the
same run.

    python profiles/tools/evaluate_c2.py [--reps 20] [--out result.json]
"""

import argparse
import importlib.util
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import lattice_based_tagger_b200 as pkg  # noqa: E402
from lattice_based_tagger_b200 import _native, synth  # noqa: E402
from lattice_based_tagger_b200.dictionary import Word  # noqa: E402
from lattice_based_tagger_b200.tagset import BOS, EOS, Unk  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
WINDOW = _native.LT_WINDOW


def _train_epoch_tool():
    spec = importlib.util.spec_from_file_location('_train_epoch_tool', os.path.join(HERE, 'train_epoch.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _full(w):
    return (w.b, w.e, w.tag0, w.tag1, w.morph0, w.morph1)


def host_loop(tagger, sents, golds, beam):
    """What lt_evaluate returns, computed on the host: (classes, counts, image scores, reasons) per sentence."""
    predicted = tagger.tag_batch(sents, beam, errors='none').materialize()
    lattices = [words[1:-1] for words, _ in tagger.lattice_batch(sents)]
    rows, images = [], []
    for sent, gold, pred, lattice in zip(sents, golds, predicted, lattices):
        chars = sent.replace(' ', '')
        n = len(chars)
        P = pred.sequences[1:-1] if pred is not None else []
        by_b = {g.b: g for g in gold}
        seg = tag = full = unit = 0
        for p in P:
            g = by_b.get(p.b)
            if g is None or g.e != p.e:
                continue
            seg += 1
            same = (p.tag0, p.tag1) == (g.tag0, g.tag1)
            tag += same
            full += same and (p.morph0, p.morph1) == (g.morph0, g.morph1)
            unit += (p.morph0, p.tag0) == (g.morph0, g.tag0)
            unit += p.tag1 is not None and (p.morph1, p.tag1) == (g.morph1, g.tag1)
        units = [sum(1 + (w.tag1 is not None) for w in ws) for ws in (gold, P)]
        counts = [len(gold), len(P), seg, tag, full, units[0], units[1], unit]
        reasons, image = [], None
        if pred is not None:
            spans = {}
            for w in lattice:
                spans.setdefault((w.b, w.e), []).append(w)
            image = []
            for j, g in enumerate(gold):
                if g.b != (gold[j - 1].e if j else 0) or g.e > n or (j == len(gold) - 1 and g.e != n):
                    reasons.append(_native.LT_GOLD_BREAKS_TILING)
                    continue
                if g.e - g.b > WINDOW:
                    reasons.append(_native.LT_GOLD_BEYOND_WINDOW)
                    continue
                cands = spans.get((g.b, g.e), [])
                hit = next((w for w in cands if _full(w) == _full(g)), None)
                sub = chars[g.b:g.e]
                if hit is None and not cands and (g.tag0, g.tag1, g.morph0, g.morph1) == (Unk, None, sub, None):
                    hit = Word(sub, sub, None, Unk, None, g.e - g.b, g.b, g.e, False)
                r = _native.LT_GOLD_OK if hit is not None else _native.LT_GOLD_NOT_IN_LATTICE
                if hit is not None and g.tag0 == Unk and j and gold[j - 1].tag0 == Unk and g.b != max(0, g.e - WINDOW):
                    r = _native.LT_GOLD_UNK_AFTER_UNK
                reasons.append(r)
                image.append(hit)
            if any(r != _native.LT_GOLD_OK for r in reasons) or (not gold and n > 0):
                image = None
        else:
            reasons = [_native.LT_GOLD_UNCHECKED] * len(gold)
        exact = pred is not None and len(P) == len(gold) and full == len(gold)
        rows.append((pred, exact, counts, reasons, image, n))
        if image is not None:
            images.append([Word(BOS, BOS, None, BOS, None, 0, 0, 0, False)] + image + [Word(EOS, EOS, None, EOS, None, 0, n, n, False)])
    scored = iter(tagger.score_paths(images).tolist() if images else [])
    classes, counts, scores, reasons = [], [], [], []
    for pred, exact, c, r, image, n in rows:
        score = next(scored) if image is not None else math.nan
        if pred is None:
            cls = _native.LT_EVAL_FAILED
        elif exact:
            cls = _native.LT_EVAL_CORRECT
        elif image is None:
            cls = _native.LT_EVAL_UNREACHABLE
        else:
            cls = _native.LT_EVAL_SEARCH_ERROR if score > pred.score else _native.LT_EVAL_MODEL_ERROR
        classes.append(cls)
        counts.append(c)
        scores.append(score)
        reasons.append(r)
    return classes, counts, scores, reasons


def gpu_info():
    return _train_epoch_tool().gpu_info()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='c2')
    ap.add_argument('--n-sent', type=int, default=None)
    ap.add_argument('--reps', type=int, default=20, help='timed repetitions of the decode, the step and the host loop')
    ap.add_argument('--host-reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    tool = _train_epoch_tool()

    cfg, dictionary, sents = synth.build_workload(args.config, n_sent=args.n_sent)
    beam = cfg['beam']
    reg = pkg.beam.RegularizationScore()
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    sents = [s for s, st in zip(sents, probe.tag_batch_packed(sents, beam)[3]) if st == 0]
    feature_dic, coef = synth.make_features(
        sents[:1000], lambda s: probe.tag_batch(s, beam, errors='none'), probe.lattice_batch,
        cfg['n_feat'], list(dictionary.tag_to_morphs), seed=3)
    probe.close()
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
    other = np.random.default_rng(11).normal(0.0, 1.0, len(feature_dic))
    teacher = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(
        reg, pkg.beam.SimpleTrigramFeatureScore(encoder, other)))
    paths = [seq.sequences[1:-1] for seq in teacher.tag_batch(sents, beam)]
    teacher.close()
    # one gold word in twelve becomes a morpheme the dictionary does not have
    rng = np.random.default_rng(5)
    paths = [[w._replace(morph0=w.morph0 + '뷁') if rng.random() < 1 / 12 else w for w in p] for p in paths]
    pairs = [tool.annotation(s, p) for s, p in zip(sents, paths)]
    pairs = [p for p in pairs if p is not None]

    tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(
        reg, pkg.beam.SimpleTrigramFeatureScore(encoder, coef)))
    t0 = time.perf_counter()
    ev = pkg.trainer.evaluate(pairs, tagger, beam)
    ms_first_call = (time.perf_counter() - t0) * 1e3
    assert not ev.not_evaluated
    T = importlib.import_module('lattice_based_tagger_b200.trainer.train')
    gold = T._GoldCorpus(pairs, tagger)
    golds = [gold.golds[i][1:-1] for i in gold.device_idx]
    engine = tagger._engine

    host = host_loop(tagger, gold.device_sents, golds, beam)
    assert ev.sent_class.tolist() == host[0]
    assert ev.counts.tolist() == host[1]
    assert [None if math.isnan(x) else x for x in ev.gold_scores.tolist()] == [None if math.isnan(x) else x for x in host[2]]
    assert [r.tolist() for r in ev.word_reason] == host[3]

    # warm-up of every shape, then the timed calls
    engine.tag_packed(gold.device_sents, beam)
    engine.evaluate(gold.pathset)
    ms_decode, ms_step = [], []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        engine.tag_packed(gold.device_sents, beam)
        t1 = time.perf_counter()
        got = engine.evaluate(gold.pathset)
        t2 = time.perf_counter()
        ms_decode.append((t1 - t0) * 1e3)
        ms_step.append((t2 - t1) * 1e3)
    assert got[0].tolist() == host[0] and got[1].tolist() == host[1]
    counters = engine.counters()
    ms_host = []
    for _ in range(args.host_reps):
        t0 = time.perf_counter()
        again = host_loop(tagger, gold.device_sents, golds, beam)
        ms_host.append((time.perf_counter() - t0) * 1e3)
    assert again[0] == host[0] and again[1] == host[1] and again[3] == host[3]
    result = {
        'config': args.config, 'sentences': len(gold.device_idx), 'gold_words': gold.pathset.n_words,
        'features': len(feature_dic), 'beam': beam,
        'class_counts': ev.class_counts, 'f1': {lv: ev.f1(lv) for lv in ('seg', 'tag', 'full', 'morph')},
        'missing_word_types': len(ev.missing_words()),
        'same_results_as_host_loop': True,
        'ms_decode_median': float(np.median(ms_decode)), 'ms_evaluate_step_median': float(np.median(ms_step)),
        'ms_host_loop_median': float(np.median(ms_host)),
        'ms_decode_all': ms_decode, 'ms_evaluate_step_all': ms_step, 'ms_host_loop_all': ms_host,
        'ms_trainer_evaluate_first_call': ms_first_call,
        'decode_counters': {k: counters[k] for k in ('sentences', 'T', 'W')},
        'timing': 'host perf_counter around calls that end in a stream synchronise',
    }
    gold.close()
    result.update(gpu_info())
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
