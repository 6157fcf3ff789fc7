"""Mini-batch perceptron on the C2 workload (`lt_trainer_step`, `fit_parameter(batch_size=...)`).

Three phases, each its own process (the profiler phase must not slow the timed ones):

  epoch    ms per epoch at B = 256 and B = 1024: the device trainer (weights and their average stay in HBM) against
           the same online loop composed from the per-step API (`_load_weights` -> `lt_tables_update_weights`,
           `tag_packed`, `lt_perceptron_delta` on the mini-batch's own path set, `np.add.at`).  Asserts identical
           `coef` and averaged weights after every epoch.  Host clock around work that ends in a synchronise.
  kernels  the step's update kernels (count buffer clear, gather_coef_counts, apply_coef_delta, scatter_coef) under
           torch.profiler, at the C2 feature count (100 k) and the C5 one (10 M; the C2 dictionary with features
           padded by synth.make_features' word n-grams, as bench.py builds C5's table).
  f1       a teacher-student split of C2 (gold = a teacher's best paths; 80 % train, 20 % held out): held-out
           `trainer.evaluate` after the same number of epochs for batch_size=None, mini-batches and averaged
           mini-batches.

Every phase prints one JSON line with the GPU name and power limit read in the same run.

    python profiles/tools/train_minibatch.py --phase epoch|kernels|f1 [--out result.json]
"""

import argparse
import importlib
import importlib.util
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import lattice_based_tagger_b200 as pkg  # noqa: E402
from lattice_based_tagger_b200 import synth  # noqa: E402

T = importlib.import_module('lattice_based_tagger_b200.trainer.train')
_spec = importlib.util.spec_from_file_location('_train_epoch_tool', os.path.join(ROOT, 'profiles', 'tools', 'train_epoch.py'))
tool = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(tool)


def c2_pairs(n_sent=None):
    """C2 sentences annotated with a teacher's best paths (profiles/tools/train_epoch.py)."""
    cfg, dictionary, sents = synth.build_workload('c2', n_sent=n_sent)
    beam = cfg['beam']
    reg = pkg.beam.RegularizationScore()
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    sents = [s for s, st in zip(sents, probe.tag_batch_packed(sents, beam)[3]) if st == 0]
    feature_dic, _ = synth.make_features(sents[:1000], lambda s: probe.tag_batch(s, beam, errors='none'), probe.lattice_batch,
                                         cfg['n_feat'], list(dictionary.tag_to_morphs), seed=3)
    probe.close()
    encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
    other = np.random.default_rng(11).normal(0.0, 1.0, len(feature_dic))
    teacher = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder, other)))
    pairs = [tool.annotation(s, seq.sequences[1:-1]) for s, seq in zip(sents, teacher.tag_batch(sents, beam))]
    teacher.close()
    return beam, dictionary, reg, encoder, [p for p in pairs if p is not None]


def student(dictionary, reg, encoder):
    return pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder)))


class ComposedLoop:
    """The online perceptron from the per-step API: weights to the tables, decode, delta to the host, update."""

    def __init__(self, tagger, encoder, sents, golds, batch):
        self.tagger, self.encoder, self.sents = tagger, encoder, sents
        self.coef = np.zeros(len(encoder.feature_dic))
        self.u = np.zeros_like(self.coef)
        self.t = 0
        T._load_weights(tagger, encoder, self.coef)
        engine = tagger._engine
        self.func = tagger.score_funcs.funcs.index(T._trigram_scorer(tagger))
        self.desc_func, self.desc_fdic = engine.tables.desc_sources()
        self.ranges = [(f, min(batch, len(sents) - f)) for f in range(0, len(sents), batch)]
        self.pathsets = [engine.upload_paths([g[1:-1] for g in golds[f:f + c]]) for f, c in self.ranges]

    def epoch(self, beam):
        engine = self.tagger._engine
        for (first, count), pathset in zip(self.ranges, self.pathsets):
            self.t += 1
            T._load_weights(self.tagger, self.encoder, self.coef)
            engine.tag_packed(self.sents[first:first + count], beam)
            delta, _, _ = engine.perceptron_delta(pathset, self.func)
            hit = np.flatnonzero((self.desc_func == self.func) & (delta != 0))
            update = np.zeros_like(self.coef)
            np.add.at(update, self.desc_fdic[hit], delta[hit].astype(np.float64))
            self.coef = self.coef + update
            self.u = self.u + (self.t - 1) * update

    def close(self):
        for p in self.pathsets:
            p.close()


def phase_epoch(args):
    beam, dictionary, reg, encoder, pairs = c2_pairs(args.n_sent)
    out = {'sentences': len(pairs), 'features': len(encoder.feature_dic), 'beam': beam, 'epochs': args.epochs, 'batch': {}}
    for batch in (256, 1024):
        dev, ref = student(dictionary, reg, encoder), student(dictionary, reg, encoder)
        coef = np.zeros(len(encoder.feature_dic))
        scorer = T._load_weights(dev, encoder, coef)
        gold = T._GoldCorpus(pairs, dev)
        engine = dev._engine
        func = dev.score_funcs.funcs.index(scorer)
        desc_func, desc_fdic = engine.tables.desc_sources()
        trainer = engine.trainer(gold.device_sents, gold.pathset, func, len(coef), np.where(desc_func == func, desc_fdic, -1), coef)
        golds = [gold.golds[i] for i in gold.device_idx]
        composed = ComposedLoop(ref, encoder, gold.device_sents, golds, batch)
        n = len(gold.device_sents)
        ms_dev, ms_ref, mistakes = [], [], []
        for epoch in range(args.epochs + 1):              # epoch 0 warms up every shape
            t0 = time.perf_counter()
            for first in range(0, n, batch):
                trainer.step(first, min(batch, n - first), beam)
            w, mean, steps, m, _ = trainer.fetch()
            t1 = time.perf_counter()
            composed.epoch(beam)
            t2 = time.perf_counter()
            assert np.array_equal(w, composed.coef), (batch, epoch)
            assert np.array_equal(mean, composed.coef - composed.u / composed.t), (batch, epoch)
            if epoch:
                ms_dev.append((t1 - t0) * 1e3)
                ms_ref.append((t2 - t1) * 1e3)
            mistakes.append(m - sum(mistakes))
        trainer.close()
        composed.close()
        gold.close()
        dev.close()
        ref.close()
        out['batch'][str(batch)] = {
            'steps_per_epoch': -(-n // batch), 'mistakes_per_epoch': mistakes[1:],
            'ms_per_epoch_device_trainer': ms_dev, 'ms_per_epoch_composed_api': ms_ref,
            'ms_per_epoch_device_trainer_median': float(np.median(ms_dev)),
            'ms_per_epoch_composed_api_median': float(np.median(ms_ref)),
            'coef_and_averaged_identical_every_epoch': True}
    out['timing'] = 'host perf_counter around an epoch that ends in a synchronise (lt_trainer_fetch / the last delta copy)'
    return out


def phase_kernels(args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    cfg, dictionary, sents = synth.build_workload('c2', n_sent=args.kernel_sents)
    beam = cfg['beam']
    reg = pkg.beam.RegularizationScore()
    probe = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg))
    sents = [s for s, st in zip(sents, probe.tag_batch_packed(sents, beam)[3]) if st == 0]
    golds = [list(seq.sequences) for seq in probe.tag_batch(sents, beam)]
    vocab = [(m, t) for t, ms in dictionary.tag_to_morphs.items() for m in sorted(ms)]
    out = {'sentences_per_step': len(sents), 'steps': args.kernel_steps, 'sizes': {}}
    for name, n_feat in (('c2', 100_000), ('c5', 10_000_000)):
        feature_dic, _ = synth.make_features(sents, lambda s: probe.tag_batch(s, beam, errors='none'), probe.lattice_batch,
                                             n_feat, list(dictionary.tag_to_morphs), seed=3, vocab=vocab)
        encoder = pkg.features.SimpleTrigramEncoder(feature_dic)
        coef = np.random.default_rng(3).normal(0.0, 1.0, len(feature_dic))
        tagger = pkg.Tagger(dictionary, score_funcs=pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(encoder, coef)))
        engine = tagger._engine
        pathset = engine.upload_paths([g[1:-1] for g in golds])
        desc_func, desc_fdic = engine.tables.desc_sources()
        trainer = engine.trainer(sents, pathset, 1, len(coef), np.where(desc_func == 1, desc_fdic, -1), coef)
        for _ in range(3):
            trainer.step(0, len(sents), beam)
        trainer.fetch()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.kernel_steps):
                trainer.step(0, len(sents), beam)
            trainer.fetch()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            key = ev.name
            if any(k in key for k in ('gather_coef_counts', 'apply_coef_delta', 'scatter_coef', 'perceptron_kernel', 'Memset')):
                short = ('memset' if 'Memset' in key else key.split('(')[0].split('::')[-1].split('<')[0])
                per.setdefault(short, []).append(ev.device_time if hasattr(ev, 'device_time') else ev.cuda_time)
        steps = args.kernel_steps
        us = {k: float(np.sum(v)) / steps for k, v in per.items()}
        update = sum(us.get(k, 0.0) for k in ('gather_coef_counts', 'apply_coef_delta', 'scatter_coef', 'memset'))
        out['sizes'][name] = {'n_feat_desc': int(engine.tables.n_desc), 'n_coef': len(coef),
                              'us_per_step': us, 'us_update_kernels_per_step': update,
                              'launches_seen': {k: len(v) for k, v in per.items()}}
        trainer.close()
        pathset.close()
        tagger.close()
    probe.close()
    out['timing'] = 'torch.profiler CUDA activity, kernel device time summed over the profiled steps / steps (memset: the count buffer clear)'
    return out


def phase_f1(args):
    beam, dictionary, reg, encoder, pairs = c2_pairs(args.n_sent)
    rng = np.random.default_rng(7)
    order = rng.permutation(len(pairs))
    cut = int(0.8 * len(pairs))
    train_pairs = [pairs[i] for i in order[:cut]]
    held = [pairs[i] for i in order[cut:]]
    out = {'train_pairs': len(train_pairs), 'held_out_pairs': len(held), 'epochs': args.f1_epochs, 'runs': {}}
    for label, batch, averaged in (('batch_size=None', None, False), ('batch_size=256', 256, False),
                                   ('batch_size=256,averaged', 256, True), ('batch_size=1024', 1024, False),
                                   ('batch_size=1024,averaged', 1024, True)):
        tagger = student(dictionary, reg, encoder)
        t0 = time.perf_counter()
        coef = T.fit_parameter(train_pairs, encoder, tagger, max_epochs=args.f1_epochs, beam_size=beam,
                               patience=args.f1_epochs + 1, batch_size=batch, averaged=averaged)
        ms = (time.perf_counter() - t0) * 1e3
        T._load_weights(tagger, encoder, coef)
        ev = T.evaluate(held, tagger, beam_size=beam)
        tr = T.evaluate(train_pairs, tagger, beam_size=beam)
        out['runs'][label] = {'held_out_f1': {lv: ev.f1(lv) for lv in ('seg', 'tag', 'full')},
                              'held_out_exact_sentences': float(np.mean(ev.exact)) if len(ev) else 0.0, 'train_f1_full': tr.f1('full'), 'ms_fit': ms}
        tagger.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--phase', choices=['epoch', 'kernels', 'f1'], required=True)
    ap.add_argument('--epochs', type=int, default=3)
    ap.add_argument('--n-sent', type=int, default=None, help='C2 sentences (default: all of C2)')
    ap.add_argument('--kernel-sents', type=int, default=256)
    ap.add_argument('--kernel-steps', type=int, default=20)
    ap.add_argument('--f1-epochs', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    result = {'phase': args.phase}
    result.update({'epoch': phase_epoch, 'kernels': phase_kernels, 'f1': phase_f1}[args.phase](args))
    result.update(tool.gpu_info())
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
