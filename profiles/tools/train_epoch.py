"""Perceptron epoch on the C2 workload: the device step (`train_epoch`: weights in place, one decode, one
`lt_perceptron_delta`) against the host loop it replaced (kept below as the reference), epoch by epoch.

The gold paths are the best paths of a tagger with the same features and other seeded weights, so that most
sentences differ from the prediction.  Asserts that `coef` is identical after every epoch and prints one JSON
line: ms per epoch of each variant, the decode and delta-step times of the device step (host clock around
calls that end in a stream synchronise), and the GPU name and power limit read in the same run.

    python profiles/tools/train_epoch.py [--epochs 3] [--out result.json]
"""

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

import lattice_based_tagger_b200 as pkg  # noqa: E402
from lattice_based_tagger_b200 import synth  # noqa: E402
from lattice_based_tagger_b200.dictionary.text import text_to_words  # noqa: E402

T = importlib.import_module('lattice_based_tagger_b200.trainer.train')


def annotation(sent, words):
    """(word_text, morph_text) of a path over `sent`, or None when a word crosses an eojeol boundary."""
    eojeols, b = [], 0
    for piece in sent.split():
        eojeols.append((b, b + len(piece), [], []))
        b += len(piece)
    for w in words:
        box = next((e for e in eojeols if e[0] <= w.b < e[1]), None)
        if box is None or w.e > box[1]:
            return None
        box[2].append(w.word)
        box[3].append('%s/%s' % (w.morph0, w.tag0) + ('' if w.tag1 is None else '+%s/%s' % (w.morph1, w.tag1)))
    return '  '.join(' '.join(e[2]) for e in eojeols), '  '.join(' '.join(e[3]) for e in eojeols)


def reference_epoch(pairs, encoder, tagger, coef, beam_size):
    """The host loop: decode, re-parse every annotation, compare, count features one index at a time."""
    coef = np.asarray(coef, dtype=np.float64).copy()
    T._load_weights(tagger, encoder, coef)
    golds, sents = [], []
    for word_text, morph_text in pairs:
        golds.append(text_to_words(word_text, morph_text))
        sents.append(T._surface(word_text))
    update = np.zeros_like(coef)
    loss = 0
    for gold, seq in zip(golds, tagger.tag_batch(sents, beam_size=beam_size, errors='none')):
        if seq is not None and T._same_path(seq.sequences, gold):
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


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(',')]
        return {'gpu': name, 'power_limit': power}
    except Exception as exc:                          # reported, not guessed
        return {'gpu': None, 'power_limit': None, 'gpu_query_error': repr(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='c2')
    ap.add_argument('--epochs', type=int, default=3)
    ap.add_argument('--n-sent', type=int, default=None)
    ap.add_argument('--reps', type=int, default=10, help='timed repetitions of the decode and of the delta step')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()

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
    pairs = [annotation(s, seq.sequences[1:-1]) for s, seq in zip(sents, teacher.tag_batch(sents, beam))]
    teacher.close()
    pairs = [p for p in pairs if p is not None]

    def tagger():
        return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder)))

    dev, ref = tagger(), tagger()
    coef_dev = coef_ref = np.zeros(len(feature_dic))
    T._load_weights(dev, encoder, coef_dev)
    t0 = time.perf_counter()
    gold = T._GoldCorpus(pairs, dev)
    ms_upload = (time.perf_counter() - t0) * 1e3
    # warm-up of every shape the timed epochs use
    T.train_epoch(pairs, encoder, dev, coef_dev, 0, False, beam_size=beam, gold=gold)
    reference_epoch(pairs, encoder, ref, coef_ref, beam)
    ms_dev, ms_ref, losses = [], [], []
    for epoch in range(1, args.epochs + 1):
        t0 = time.perf_counter()
        coef_dev, loss_dev = T.train_epoch(pairs, encoder, dev, coef_dev, epoch, False, beam_size=beam, gold=gold)
        ms_dev.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        coef_ref, loss_ref = reference_epoch(pairs, encoder, ref, coef_ref, beam)
        ms_ref.append((time.perf_counter() - t0) * 1e3)
        assert loss_dev == loss_ref, (epoch, loss_dev, loss_ref)
        assert np.array_equal(coef_dev, coef_ref), epoch
        losses.append(loss_dev)

    # the two device calls of an epoch on their own, with the last epoch's weights
    engine = dev._engine
    func = dev.score_funcs.funcs.index(T._trigram_scorer(dev))
    ms_decode, ms_delta = [], []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        engine.tag_packed(gold.device_sents, beam)
        t1 = time.perf_counter()
        engine.perceptron_delta(gold.pathset, func)
        t2 = time.perf_counter()
        ms_decode.append((t1 - t0) * 1e3)
        ms_delta.append((t2 - t1) * 1e3)
    counters = engine.counters()
    gold_words = gold.pathset.n_words
    gold.close()
    result = {
        'config': args.config, 'sentences': len(pairs), 'device_sentences': len(gold.device_idx),
        'gold_words': gold_words,
        'features': len(feature_dic), 'beam': beam, 'epochs': args.epochs, 'loss_per_epoch': losses,
        'coef_identical_every_epoch': True,
        'ms_per_epoch_device_step': ms_dev, 'ms_per_epoch_host_loop': ms_ref,
        'ms_gold_upload_once': ms_upload,
        'ms_decode_median': float(np.median(ms_decode)), 'ms_delta_step_median': float(np.median(ms_delta)),
        'ms_decode_all': ms_decode, 'ms_delta_step_all': ms_delta,
        'decode_counters': {k: counters[k] for k in ('sentences', 'T', 'F', 'W')},
        'timing': 'host perf_counter around calls that end in a stream synchronise',
    }
    result.update(gpu_info())
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
