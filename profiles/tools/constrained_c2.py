"""The constrained search on the C2 workload (10 000 sentences, beam 5, reg + trigram scorers) in three settings:
no constraints, two constraints per sentence taken from its best path, and every word of its best path constrained
(with its tag; words of the Unknown tag as any-word spans).

Per setting: the device time of constraint_prep_kernel and beam_kernel per step (torch.profiler with CUDA
activities, in a phase of its own), `Engine.tag_packed` end to end with the constraint set bound once (the text
packed on the host, then `lt_tag_batch_host`; host clock around calls that end in a stream synchronise; reported as
`ms_lt_tag_batch_host_*`), the same through `Tagger.tag_batch_packed(constraints=...)`
(which also validates, uploads and binds the set), and an oracle parity sample (tests/_constrained_oracle.py).
Prints one JSON line with the GPU name and power limit read in the same run.

    python profiles/tools/constrained_c2.py [--reps 50] [--out profiles/constrained_c2.json]
"""

import argparse
import ctypes
import importlib.util
import json
import os
import random
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import lattice_based_tagger_b200 as pkg  # noqa: E402
from lattice_based_tagger_b200 import _native, synth  # noqa: E402
from lattice_based_tagger_b200.tagset import Unk  # noqa: E402
from tests import _constrained_oracle as co  # noqa: E402
from oracle import lattice_oracle as lo  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def gpu_info():
    spec = importlib.util.spec_from_file_location('_train_epoch_tool', os.path.join(HERE, 'train_epoch.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.gpu_info()


def settings(best):
    """{name: per-sentence constraint lists} from each sentence's best path."""
    rng = random.Random(7)
    out = {'none': None, 'two_per_sentence': [], 'every_word': []}
    for words in best:
        items = [(w.b, w.e) if w.tag0 == Unk else (w.b, w.e, w.tag0) for w in words if w.e - w.b <= _native.LT_WINDOW]
        out['every_word'].append(items)
        out['two_per_sentence'].append(sorted(rng.sample(items, min(2, len(items)))))
    return out


def kernel_times(engine, sents, beam, reps):
    """Median device time per step of the constraint preparation and the beam kernel (torch.profiler)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    engine.tag_packed(sents, beam)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            engine.tag_packed(sents, beam)
        torch.cuda.synchronize()
    times = {'constraint_prep_kernel': [], 'beam_kernel': []}
    for ev in prof.events():
        if ev.device_type.name != 'CUDA':
            continue
        for name in times:
            if name in ev.name:
                times[name].append(ev.time_range.elapsed_us() / 1e3)
    return {('ms_' + k + '_median'): (float(np.median(v)) if v else 0.0) for k, v in times.items()} | \
           {('launches_' + k): len(v) for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='c2')
    ap.add_argument('--n-sent', type=int, default=None)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--oracle-sample', type=int, default=60)
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
    funcs = pkg.beam.BeamScoreFunctions(reg, pkg.beam.SimpleTrigramFeatureScore(pkg.features.SimpleTrigramEncoder(feature_dic), coef))
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    engine = tagger._engine
    best = [seq.sequences[1:-1] for seq in tagger.tag_batch(sents, beam)]
    oracle = lo.OracleTagger(dictionary, funcs)
    sample = random.Random(1).sample(range(len(sents)), min(args.oracle_sample, len(sents)))

    result = {'config': args.config, 'sentences': len(sents), 'beam': beam, 'features': len(feature_dic), 'settings': {}}
    for name, cons in settings(best).items():
        row = {'constraints': 0 if cons is None else sum(len(c) for c in cons)}
        handle = None
        if cons is not None:
            arr, off = engine.pack_constraints(sents, cons)
            handle = ctypes.c_void_p()
            _native.check(engine._lib.lt_constraints_create(engine.tables.handle, len(sents), _native.ptr(arr), _native.ptr(off),
                                                            ctypes.byref(handle)))
            _native.check(engine._lib.lt_batch_set_constraints(engine.batch, handle))
        try:
            packed = engine.tag_packed(sents, beam)
            assert (packed[3] == 0).all()
            ms = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                engine.tag_packed(sents, beam)
                ms.append((time.perf_counter() - t0) * 1e3)
            row['ms_lt_tag_batch_host_median'] = float(np.median(ms))
            row['ms_lt_tag_batch_host_all'] = ms
            row.update(kernel_times(engine, sents, beam, args.reps))
        finally:
            if handle is not None:
                engine._lib.lt_batch_set_constraints(engine.batch, None)
                engine._lib.lt_constraints_destroy(handle)
        ms = []
        for _ in range(max(3, args.reps // 10)):
            t0 = time.perf_counter()
            again = tagger.tag_batch_packed(sents, beam, constraints=cons)
            ms.append((time.perf_counter() - t0) * 1e3)
        row['ms_tag_batch_packed_python_median'] = float(np.median(ms))
        assert all(a.tobytes() == b.tobytes() for a, b in zip(packed, again))
        # parity sample against the oracle
        seqs = engine.unpack(sents, packed, 'raise')
        for i in sample:
            want = co.survivors(oracle, sents[i], beam, [] if cons is None else [tuple(c) + (None,) * (3 - len(c)) for c in cons[i]])[0]
            assert [tuple(w) for w in seqs[i].sequences] == want.words and seqs[i].score == want.score, i
        row['oracle_sample_identical'] = len(sample)
        if name == 'every_word':
            row['best_path_unchanged'] = all(s.sequences[1:-1] == b for s, b in zip(seqs, best))
        result['settings'][name] = row
    result['timing'] = ('end to end: host perf_counter around lt_tag_batch_host (ends in a stream synchronise); kernels: '
                        'torch.profiler CUDA activity, median per launch')
    result.update(gpu_info())
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
