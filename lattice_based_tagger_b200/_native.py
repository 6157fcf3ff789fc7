"""ctypes binding of the C-ABI library `liblt_b200.so` (include/lt_b200.h).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no
alternative implementation behind this module: if the library is missing, or no CUDA device is
usable, the calls raise.
"""

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'liblt_b200.so')

LT_ABI_VERSION = 8
LT_OK = 0
LT_SENT_OK, LT_SENT_NO_EDGES, LT_SENT_BAD_SPACE, LT_SENT_TOO_LONG, LT_SENT_UNSUPPORTED_CHAR, LT_SENT_BAD_CONSTRAINT = 0, 1, 2, 3, 4, 5
LT_NO_TAG = 0xFF
LT_NO_RULE = 0xFFFFFFFF
LT_EDGE_IS_L, LT_EDGE_UNK, LT_EDGE_LEMMA, LT_EDGE_SKIP2, LT_EDGE_EXPLICIT, LT_EDGE_FORCED = 1, 2, 4, 8, 16, 32
(LT_LOOKUP_MORPHEME, LT_LOOKUP_LR, LT_LOOKUP_LR_ALL, LT_LOOKUP_WORD, LT_LOOKUP_WORD_ALL,
 LT_LOOKUP_EXACT) = range(6)
LT_FUNC_REG, LT_FUNC_MPREF, LT_FUNC_WPREF, LT_FUNC_TRIGRAM = 1, 2, 3, 4
LT_MAX_BEAM = 64
LT_WINDOW = 8
LT_EVAL_CORRECT, LT_EVAL_FAILED, LT_EVAL_UNREACHABLE, LT_EVAL_SEARCH_ERROR, LT_EVAL_MODEL_ERROR = range(5)
LT_GOLD_OK, LT_GOLD_BREAKS_TILING, LT_GOLD_BEYOND_WINDOW, LT_GOLD_NOT_IN_LATTICE, LT_GOLD_UNK_AFTER_UNK = range(5)
LT_GOLD_UNCHECKED = 0xFF
(LT_EVAL_GOLD_WORDS, LT_EVAL_PRED_WORDS, LT_EVAL_SEG, LT_EVAL_TAG, LT_EVAL_FULL, LT_EVAL_GOLD_UNITS, LT_EVAL_PRED_UNITS,
 LT_EVAL_UNIT_MATCH) = range(8)
LT_EVAL_N_COUNTS = 8
LT_UPDATE_FULL, LT_UPDATE_EARLY, LT_UPDATE_MAX_VIOLATION = range(3)
LT_MAX_FUNCS = 8

#: numpy view of `lt_edge` (16 bytes)
EDGE_DTYPE = np.dtype([('b', '<u2'), ('e', '<u2'), ('len', '<u2'), ('tag0', 'u1'), ('tag1', 'u1'),
                       ('rule', '<u4'), ('split', '<u2'), ('flags', 'u1'), ('reserved', 'u1')])
assert EDGE_DTYPE.itemsize == 16

#: numpy view of `lt_constraint` (8 bytes)
CONSTRAINT_DTYPE = np.dtype([('b', '<u2'), ('e', '<u2'), ('tag', 'u1'), ('reserved', 'u1', (3,))])
assert CONSTRAINT_DTYPE.itemsize == 8

_p = ctypes.c_void_p


class lt_func(ctypes.Structure):
    _fields_ = [('kind', ctypes.c_int32), ('reserved', ctypes.c_int32), ('p', ctypes.c_double * 3)]


class lt_tables_desc(ctypes.Structure):
    _fields_ = [
        ('abi_version', ctypes.c_int32), ('n_tags', ctypes.c_int32),
        ('n_dict', ctypes.c_int64), ('dict_chars', _p), ('dict_off', _p), ('dict_tagmask', _p),
        ('dict_lemma', _p), ('n_tag_order', ctypes.c_int32), ('tag_order', _p),
        ('max_len', ctypes.c_int32), ('reserved0', ctypes.c_int32),
        ('n_rule_keys', ctypes.c_int64), ('rule_key_chars', _p), ('rule_key_len', _p),
        ('rule_k3_first', _p), ('rule_first', _p), ('n_rules', ctypes.c_int64), ('rule_chars', _p),
        ('rule_stem_off', _p), ('rule_eomi_off', _p),
        ('n_funcs', ctypes.c_int32), ('reserved1', ctypes.c_int32), ('funcs', _p),
        ('n_fstr', ctypes.c_int64), ('fstr_chars', _p), ('fstr_off', _p),
        ('n_feat', ctypes.c_int64), ('feat_func', _p), ('feat_template', _p), ('feat_s', _p),
        ('feat_a', _p), ('feat_weight', _p),
        ('n_pref', ctypes.c_int64), ('pref_func', _p), ('pref_tag', _p), ('pref_s', _p),
        ('pref_value', _p),
    ]


class lt_counters(ctypes.Structure):
    _fields_ = [(name, ctypes.c_uint64) for name in ('sentences', 'L', 'P', 'E', 'T', 'F', 'Bk', 'W')]

    def as_dict(self):
        return {name: int(getattr(self, name)) for name, _ in self._fields_}


class lt_timings(ctypes.Structure):
    _fields_ = [(name, ctypes.c_float) for name in ('ms_h2d', 'ms_lattice', 'ms_reserved0', 'ms_reserved1',
                                                    'ms_beam', 'ms_pack', 'ms_d2h', 'ms_total')]

    def as_dict(self):
        return {name: float(getattr(self, name)) for name, _ in self._fields_}


class lt_info(ctypes.Structure):
    _fields_ = ([('launches', ctypes.c_int64), ('edge_cap', ctypes.c_int64), ('n_edges', ctypes.c_int64)] +
                [(name, ctypes.c_int32) for name in (
                    'reruns', 'hcap', 'retry_hcap', 'retried', 'unit_limit', 'lattice_warps', 'lattice_ctas_per_sm',
                    'lattice_smem', 'beam_warps', 'beam_ctas_per_sm', 'beam_smem', 'beam_trail_smem', 'sm_count')] +
                [('reserved', ctypes.c_int32 * 3)])

    def as_dict(self):
        return {name: int(getattr(self, name)) for name, _ in self._fields_ if name != 'reserved'}


#: every symbol include/lt_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    'lt_last_error': (ctypes.c_char_p, []),
    'lt_abi_version': (ctypes.c_int, []),
    'lt_tables_create': (ctypes.c_int, [ctypes.POINTER(lt_tables_desc), ctypes.c_int, ctypes.POINTER(_p)]),
    'lt_tables_destroy': (None, [_p]),
    'lt_tables_device_bytes': (ctypes.c_int64, [_p]),
    'lt_tables_max_sentence_units': (ctypes.c_int32, [_p]),
    'lt_tables_update_weights': (ctypes.c_int, [_p, _p, ctypes.c_int64]),
    'lt_batch_create': (ctypes.c_int, [_p, ctypes.POINTER(_p)]),
    'lt_batch_destroy': (None, [_p]),
    'lt_batch_set_lookup': (ctypes.c_int, [_p, ctypes.c_int32]),
    'lt_lattice_import': (ctypes.c_int, [_p, _p, _p, ctypes.c_int32, _p, _p, _p, _p, ctypes.c_int64]),
    'lt_beam_kbest': (ctypes.c_int, [_p, ctypes.c_int32, _p]),
    'lt_tag_batch_host_kbest': (ctypes.c_int, [_p, _p, _p, ctypes.c_int32, ctypes.c_int32]),
    'lt_kbest_size': (ctypes.c_int, [_p, ctypes.POINTER(ctypes.c_int64)]),
    'lt_kbest_fetch': (ctypes.c_int, [_p, _p, _p, _p, ctypes.c_int64, _p, _p]),
    'lt_lattice_status': (ctypes.c_int, [_p, _p, _p]),
    'lt_batch_info': (ctypes.c_int, [_p, ctypes.POINTER(lt_info)]),
    'lt_tag_batch_host': (ctypes.c_int, [_p, _p, _p, ctypes.c_int32, ctypes.c_int32, _p, _p, ctypes.c_int64, _p, _p]),
    'lt_lattice': (ctypes.c_int, [_p, _p, _p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, _p]),
    'lt_lattice_host': (ctypes.c_int, [_p, _p, _p, ctypes.c_int32]),
    'lt_beam': (ctypes.c_int, [_p, ctypes.c_int32, _p]),
    'lt_tag_batch_device': (ctypes.c_int, [_p, _p, _p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, _p]),
    'lt_lattice_size': (ctypes.c_int, [_p, ctypes.POINTER(ctypes.c_int64)]),
    'lt_lattice_fetch': (ctypes.c_int, [_p, _p, ctypes.c_int64, _p]),
    'lt_paths_size': (ctypes.c_int, [_p, ctypes.POINTER(ctypes.c_int64)]),
    'lt_paths_fetch': (ctypes.c_int, [_p, _p, _p, ctypes.c_int64, _p, _p]),
    'lt_batch_counters': (ctypes.c_int, [_p, ctypes.POINTER(lt_counters)]),
    'lt_batch_timings': (ctypes.c_int, [_p, ctypes.POINTER(lt_timings)]),
    'lt_batch_set_stage_timing': (ctypes.c_int, [_p, ctypes.c_int32]),
    'lt_pathset_create': (ctypes.c_int, [_p, ctypes.c_int32, _p, _p, _p, _p, ctypes.c_int64, ctypes.POINTER(_p)]),
    'lt_pathset_destroy': (None, [_p]),
    'lt_pathset_eval': (ctypes.c_int, [_p, _p, ctypes.c_int32, _p, _p, _p, ctypes.c_int64]),
    'lt_perceptron_delta': (ctypes.c_int, [_p, _p, ctypes.c_int32, _p, ctypes.c_int64, _p, ctypes.POINTER(ctypes.c_int64)]),
    'lt_evaluate': (ctypes.c_int, [_p, _p, _p, _p, _p, _p]),
    'lt_trainer_create': (ctypes.c_int, [_p, ctypes.c_int32, _p, _p, ctypes.c_int32, _p, ctypes.c_int64, _p, _p, ctypes.POINTER(_p)]),
    'lt_trainer_step': (ctypes.c_int, [_p, _p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]),
    'lt_trainer_fetch': (ctypes.c_int, [_p, _p, _p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64), _p]),
    'lt_trainer_destroy': (None, [_p]),
    'lt_trainer_set_update': (ctypes.c_int, [_p, ctypes.c_int32]),
    'lt_trainer_fetch_update': (ctypes.c_int, [_p, _p, _p]),
    'lt_constraints_create': (ctypes.c_int, [_p, ctypes.c_int32, _p, _p, ctypes.POINTER(_p)]),
    'lt_constraints_destroy': (None, [_p]),
    'lt_batch_set_constraints': (ctypes.c_int, [_p, _p]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load():
    """Load liblt_b200.so (once).  Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            '%s is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc, sm_100a). The tagger has no CPU fallback.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.lt_abi_version() != LT_ABI_VERSION:
        raise NativeLibraryError('liblt_b200.so has ABI version %d, expected %d; rebuild it'
                                 % (lib.lt_abi_version(), LT_ABI_VERSION))
    _lib = lib
    return lib


def check(rc):
    if rc != LT_OK:
        message = load().lt_last_error().decode('utf-8', 'replace')
        raise NativeLibraryError('liblt_b200: error %d: %s' % (rc, message))


def ptr(array):
    """Raw pointer of a C-contiguous numpy array (the caller keeps the array alive)."""
    if array is None:
        return None
    assert array.flags['C_CONTIGUOUS']
    return array.ctypes.data_as(_p)
