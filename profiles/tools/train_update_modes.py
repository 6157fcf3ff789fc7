"""The perceptron's update modes on the C2 workload (`lt_trainer_set_update`, `fit_parameter(update=...)`), on the
corpus and split of profiles/tools/train_minibatch.py (C2 sentences, gold = a teacher's best paths, 80 % train).

  epoch    ms per epoch for 'full', 'early' and 'max_violation' at B = 256 and 1024: a host clock around an epoch
           that ends in a synchronise (`lt_trainer_fetch`), after one warm-up epoch.
  kernels  device time per step under torch.profiler (a run of its own): the beam kernel in each mode (FULL keeps
           the back-pointers in shared memory, the others in HBM), violation_kernel against perceptron_kernel, and
           the 0xFF memset of the trail.
  f1       held-out `trainer.evaluate` F1 ('full' level) and exact sentences after 10 epochs, for every mode x
           {plain, averaged} x B in {256, 1024}.

Every phase prints one JSON line with the GPU name and power limit read in the same run.

    python profiles/tools/train_update_modes.py --phase epoch|kernels|f1 [--out result.json]
"""

import argparse
import importlib.util
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
_spec = importlib.util.spec_from_file_location('_train_minibatch_tool', os.path.join(ROOT, 'profiles', 'tools', 'train_minibatch.py'))
mb = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mb)
T = mb.T

MODES = ('full', 'early', 'max_violation')


def _split(args):
    beam, dictionary, reg, encoder, pairs = mb.c2_pairs(args.n_sent)
    order = np.random.default_rng(7).permutation(len(pairs))
    cut = int(0.8 * len(pairs))
    return beam, dictionary, reg, encoder, [pairs[i] for i in order[:cut]], [pairs[i] for i in order[cut:]]


def _trainer(dictionary, reg, encoder, pairs, mode):
    tagger = mb.student(dictionary, reg, encoder)
    coef = np.zeros(len(encoder.feature_dic))
    scorer = T._load_weights(tagger, encoder, coef)
    gold = T._GoldCorpus(pairs, tagger)
    engine = tagger._engine
    func = tagger.score_funcs.funcs.index(scorer)
    desc_func, desc_fdic = engine.tables.desc_sources()
    trainer = engine.trainer(gold.device_sents, gold.pathset, func, len(coef), np.where(desc_func == func, desc_fdic, -1), coef,
                             update=mode)
    return tagger, gold, trainer, len(gold.device_sents)


def phase_epoch(args):
    beam, dictionary, reg, encoder, train_pairs, _ = _split(args)
    out = {'train_sentences': len(train_pairs), 'beam': beam, 'epochs': args.epochs, 'runs': {}}
    for batch in (256, 1024):
        for mode in MODES:
            tagger, gold, trainer, n = _trainer(dictionary, reg, encoder, train_pairs, mode)
            ms = []
            for epoch in range(args.epochs + 1):          # epoch 0 warms up every shape
                t0 = time.perf_counter()
                for first in range(0, n, batch):
                    trainer.step(first, min(batch, n - first), beam)
                trainer.fetch()
                if epoch:
                    ms.append((time.perf_counter() - t0) * 1e3)
            trainer.close()
            gold.close()
            tagger.close()
            out['runs']['%s,B=%d' % (mode, batch)] = {'ms_per_epoch': ms, 'ms_per_epoch_median': float(np.median(ms))}
    out['timing'] = 'host perf_counter around an epoch that ends in a synchronise (lt_trainer_fetch)'
    return out


def phase_kernels(args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    beam, dictionary, reg, encoder, train_pairs, _ = _split(args)
    out = {'train_sentences': len(train_pairs), 'beam': beam, 'batch': args.batch, 'runs': {}}
    for mode in MODES:
        tagger, gold, trainer, n = _trainer(dictionary, reg, encoder, train_pairs, mode)
        ranges = [(f, min(args.batch, n - f)) for f in range(0, n, args.batch)]
        for first, count in ranges:
            trainer.step(first, count, beam)
        trainer.fetch()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for first, count in ranges:
                trainer.step(first, count, beam)
            trainer.fetch()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            key = ev.name
            for name in ('beam_kernel', 'violation_kernel', 'perceptron_kernel', 'Memset'):
                if name in key:
                    per.setdefault(name, []).append(ev.device_time if hasattr(ev, 'device_time') else ev.cuda_time)
        steps = len(ranges)
        out['runs'][mode] = {'steps': steps, 'us_per_step': {k: float(np.sum(v)) / steps for k, v in per.items()},
                             'launches_seen': {k: len(v) for k, v in per.items()}}
        trainer.close()
        gold.close()
        tagger.close()
    out['timing'] = ('torch.profiler CUDA activity, device time summed over one profiled epoch / steps; Memset: every memset '
                     'of the step (the count buffer clear in all modes, the 0xFF trail fill in early / max_violation)')
    return out


def phase_f1(args):
    beam, dictionary, reg, encoder, train_pairs, held = _split(args)
    out = {'train_pairs': len(train_pairs), 'held_out_pairs': len(held), 'epochs': args.f1_epochs, 'runs': {}}
    for batch in (256, 1024):
        for mode in MODES:
            for averaged in (False, True):
                tagger = mb.student(dictionary, reg, encoder)
                coef = T.fit_parameter(train_pairs, encoder, tagger, max_epochs=args.f1_epochs, beam_size=beam,
                                       patience=args.f1_epochs + 1, batch_size=batch, averaged=averaged, update=mode)
                T._load_weights(tagger, encoder, coef)
                ev = T.evaluate(held, tagger, beam_size=beam)
                out['runs']['%s,B=%d%s' % (mode, batch, ',averaged' if averaged else '')] = {
                    'held_out_f1_full': ev.f1('full'), 'held_out_exact_sentences': float(np.mean(ev.exact)) if len(ev) else 0.0}
                tagger.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--phase', choices=['epoch', 'kernels', 'f1'], required=True)
    ap.add_argument('--epochs', type=int, default=3)
    ap.add_argument('--batch', type=int, default=256, help='kernels phase: sentences per step')
    ap.add_argument('--n-sent', type=int, default=None, help='C2 sentences (default: all of C2)')
    ap.add_argument('--f1-epochs', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    result = {'phase': args.phase}
    result.update({'epoch': phase_epoch, 'kernels': phase_kernels, 'f1': phase_f1}[args.phase](args))
    result.update(mb.tool.gpu_info())
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
