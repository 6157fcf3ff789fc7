"""Differential fuzzing of the kernel SOURCES against the oracle on the CPU (test infrastructure; not
collected by pytest): random dictionaries / rules / features / sentences per seed, every sentence's
lattice, best path, fp64 score and work counters compared bit for bit through the SIMT emulator, with
the beam sizes, sentence lengths, k-best survivors and lookup modes rotating over the seeds.  Every seed
also scores and featurizes random tilings of its sentences and runs the perceptron step against gold
paths that include near misses (tests/test_gpu_path_edges.py, `check_path_stage`); the 110- and
200-syllable sentences give paths of more than one 32-word chunk.  Every odd seed also runs the constrained
search (tests/test_gpu_constraint_edges.py, `pattern_constraints`) with its beam sizes against the constrained
oracle, survivor for survivor.

    python tests/fuzz_emulated.py FIRST_SEED LAST_SEED        # prints `ok SEED` / `FAIL SEED` + traceback
    python tests/fuzz_emulated.py FIRST_SEED LAST_SEED knobs  # + the library's debugging knobs rotating over the seeds

With `knobs` every seed also picks one of KNOBS (tiny staging / edge buffers: retry pass and grow-and-rerun;
every eojeol ranked by the sort; back-pointers in HBM; unsorted work order; a wide "device" with the CTAs run
last to first).  LT_SIMT_MEMCHECK=1 in the environment adds the emulator's guard pages (tests/simt/simt.h).
"""

import os
import random
import sys
import traceback

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import lattice_based_tagger_b200 as pkg                      # noqa: E402
from oracle import lattice_oracle as lo                      # noqa: E402
from tests import _cases, _checks, _emu                      # noqa: E402
from tests import _constrained_oracle as co                  # noqa: E402
from tests import test_gpu_constraint_edges as constraint_edges  # noqa: E402
from tests import test_gpu_constraints as constraints        # noqa: E402
from tests import test_gpu_path_edges as path_edges          # noqa: E402

BEAMS = [(1, 5), (2, 10), (3, 33), (7, 64), (16, 40)]
LENGTHS = (8, 25, 60, 110, 200)
KNOBS = [
    {},
    {'LT_HIT_CAP': '8', 'LT_EDGE_CAP': '16'},
    {'LT_SORT_MIN': '1', 'LT_HIT_CAP': '32'},
    {'LT_TRAIL_SMEM': '0'},
    {'LT_SORT_BY_LENGTH': '0', 'LT_HIT_CAP': '64', 'LT_EDGE_CAP': '64'},
    {'LT_SIMT_SMS': '16', 'LT_SIMT_BLOCK_ORDER': 'reverse', 'LT_PROLOGUE_CTAS': '3'},
    {'LT_HIT_CAP': '16', 'LT_ADAPT_DIV': '1', 'LT_SORT_MIN': '4'},
]
KNOB_NAMES = sorted({name for knobs in KNOBS for name in knobs})


def run_seed(seed, knobs=False):
    if knobs:
        for name in KNOB_NAMES:
            os.environ.pop(name, None)
        os.environ.update(KNOBS[(seed // 3) % len(KNOBS)])           # read when the Tagger creates its batch object
    case = _checks.make_case(seed, n_sent=6 + seed % 13, max_sent_len=LENGTHS[seed % 5])
    dictionary, funcs = _cases.build_objects(case, pkg)
    tagger = pkg.Tagger(dictionary, score_funcs=funcs)
    oracle = lo.OracleTagger(dictionary, funcs)
    beams = BEAMS[(seed // 5) % 5]
    _checks.check_against_oracle(tagger, oracle, case['sentences'], beams, counters=True)
    if seed % 3 == 0:
        _checks.check_kbest(tagger, oracle, case['sentences'], (beams[0], 5))
    path_edges.check_path_stage(case, funcs, tagger, seed, beams[0])
    if seed % 2:
        check_constrained(case, tagger, oracle, seed, beams)
    if seed % 7 == 0:
        _checks.check_lookup_modes(case)


def check_constrained(case, tagger, oracle, seed, beams):
    """The constrained search against the constrained oracle: random constraints, every span constrained back to
    back, and 8-syllable constraints end to end, rotating over the sentences."""
    rng = random.Random(seed ^ 0xC0)
    cons = []
    for i, sent in enumerate(case['sentences']):
        try:
            survivor = rng.choice(co.survivors(oracle, sent, 5, [])).words[1:-1]
        except IndexError:
            survivor = None
        kind = ('random', 'back_to_back', 'eight')[i % 3]
        cons.append(constraint_edges.pattern_constraints(kind, rng, sent, oracle.lattice(sent), case['tags'], survivor))
    constraints.check_parity(tagger, oracle, case['sentences'], cons, beams)


def main(first, last, knobs=False):
    fails = 0
    with _emu.emulated():
        for seed in range(first, last):
            try:
                run_seed(seed, knobs)
                print('ok', seed, flush=True)
            except Exception:
                fails += 1
                print('FAIL', seed, flush=True)
                traceback.print_exc()
    print('done: %d seeds, %d failures' % (last - first, fails))
    return 1 if fails else 0


if __name__ == '__main__':
    sys.exit(main(int(sys.argv[1]), int(sys.argv[2]), knobs=len(sys.argv) > 3 and sys.argv[3] == 'knobs'))
