"""The C ABI's host layer: malformed imported lattices are rejected before anything reads past the caller's arrays,
and every entry point gives back all the device memory it took (through the SIMT emulator's buffer registry)."""

import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from lattice_based_tagger_b200 import _native
from lattice_based_tagger_b200.dictionary.text import text_to_words
from lattice_based_tagger_b200.engine import pack_sentences
from lattice_based_tagger_b200.trainer.train import _surface
from tests.test_gpu_paths import PAIRS, _toy_tagger

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BMP_PAIRS = [p for p in PAIRS if all(ord(c) < 0x10000 for c in p[0])]      # (the device text is UTF-16 code units)
SENTS = [_surface(w) for w, _ in BMP_PAIRS]
INVALID = 1                                                                   # LT_ERR_INVALID


def _import_arrays(engine, sents):
    """The arguments of lt_lattice_import for the device's own lattices of `sents`, as numpy arrays."""
    text, offsets = pack_sentences(sents)
    flat, counts = [], np.zeros(int(offsets[-1]), dtype=np.int64)
    for i, words in enumerate(engine.lattice_words(sents)):
        for w in sorted(words, key=lambda w: (w.e, w.b)):
            flat.append(w)
            counts[int(offsets[i]) + w.e - 1] += 1
    end_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    edges, units, str_off, n_strings = engine.pack_words(flat)
    return dict(text=text, offsets=offsets, edges=edges, end_off=end_off, units=units, str_off=str_off, n_strings=n_strings)


@pytest.mark.gpu
def test_c_abi_rejects_malformed_imports():
    tagger = _toy_tagger()[0]
    lib, batch = tagger._lib, tagger._batch
    good = _import_arrays(tagger._engine, SENTS)

    def run(**change):
        a = dict(good, **change)
        return lib.lt_lattice_import(batch, _native.ptr(a['text']), _native.ptr(a['offsets']), len(SENTS), _native.ptr(a['edges']),
                                     _native.ptr(a['end_off']), _native.ptr(a['units']), _native.ptr(a['str_off']), a['n_strings'])

    def edited(name, index, field=None, value=None):
        arr = good[name].copy()
        if field is None:
            arr[index] = value
        else:
            arr[index][field] = value
        return arr

    edges, end_off, str_off = good['edges'], good['end_off'], good['str_off']
    # two edges of one end position with different begins, in order
    k = next(k for k in range(len(edges) - 1) if edges[k]['e'] == edges[k + 1]['e'] and edges[k]['b'] < edges[k + 1]['b']
             and int(np.searchsorted(end_off, k, 'right')) == int(np.searchsorted(end_off, k + 1, 'right')))
    swapped = edges.copy()
    swapped[[k, k + 1]] = swapped[[k + 1, k]]
    lemma = edited('edges', 0, 'flags', _native.LT_EDGE_LEMMA)
    assert lemma[0]['rule'] != _native.LT_NO_RULE
    invalid = {
        'end_off not monotone': run(end_off=edited('end_off', 1, value=end_off[2] + 1)),
        'edge not ending at its position': run(edges=edited('edges', 0, 'e', edges[0]['e'] + 1)),
        'b >= e': run(edges=edited('edges', 0, 'b', edges[0]['e'])),
        'begins not sorted': run(edges=swapped),
        'tag out of range': run(edges=edited('edges', 0, 'tag0', 40)),
        'string index out of range': run(edges=edited('edges', 0, 'rule', good['n_strings'] // 3)),
        'n_strings % 3': run(n_strings=good['n_strings'] - 1),
        'str_off not monotone': run(str_off=edited('str_off', 1, value=str_off[2] + 1)),
        'lemma edge with a rule, not explicit': run(edges=lemma),
    }
    assert invalid == {what: INVALID for what in invalid}
    # (rejected before the first edge or string is read)
    assert run(end_off=edited('end_off', 0, value=-1)) == INVALID and b'end_off[0]' in lib.lt_last_error()
    assert run(str_off=edited('str_off', 0, value=-1)) == INVALID and b'str_off[0]' in lib.lt_last_error()
    assert run() == _native.LT_OK
    assert lib.lt_beam_kbest(batch, 5, None) == _native.LT_OK
    tagger.close()


def _leak_check():
    """Every entry point once (in a process with LT_SIMT_MEMCHECK=1 and tiny staging / edge buffers, so that the
    first batch grows them and runs again); prints the live device buffers before and after."""
    from tests import _emu
    lib = _emu.emu_lib()
    lib.simt_live_buffers.restype = ctypes.c_size_t
    before = lib.simt_live_buffers()
    with _emu.emulated():
        tagger = _toy_tagger(extra_tags=['Suffix'])[0]
        engine = tagger._engine
        tagger.timings()                                         # stage events from now on
        tagger.tag_batch(SENTS, errors='none')                   # lt_tag_batch_host, grown and rerun
        assert tagger.info()['reruns'] > 0
        tagger.tag_batch_kbest(SENTS, beam_size=5, errors='none')
        engine.kbest_packed(SENTS, 5, imported=engine.lattice_words(SENTS))   # lt_lattice_host, lt_lattice_import
        gold = engine.upload_paths([text_to_words(w, m)[1:-1] for w, m in BMP_PAIRS])
        engine.eval_paths(gold, func=1)
        engine.tag_packed(SENTS, 5)
        engine.perceptron_delta(gold, 1)
        engine.evaluate(gold)
        tagger.update_weights()
        gold.close()
        tagger.close()
    print('live device buffers: %d %d' % (before, lib.simt_live_buffers()))


def test_no_device_buffer_outlives_its_owner():
    env = dict(os.environ, LT_SIMT_MEMCHECK='1', LT_HIT_CAP='8', LT_EDGE_CAP='16')
    out = subprocess.run([sys.executable, '-c', 'from tests import test_host_layer; test_host_layer._leak_check()'],
                         cwd=ROOT, env=env, capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    before, after = out.stdout.split('live device buffers:')[1].split()
    assert int(before) == 0 and int(after) == 0, out.stdout
