"""`Evaluation` — a tagger's output compared with gold analyses (`Tagger.evaluate`, `trainer.evaluate`).

Everything per sentence comes from one `lt_evaluate` call (include/lt_b200.h): the sentence's class, the
word-level counts, the score of the gold path's image and a reason code per gold word.  This class only
sums and presents them.

Classes, one per sentence:
    correct        the best path is the gold path (b, e, tags and morphemes of every word)
    failed         the search did not tag the sentence (no dictionary edge, too long, bad whitespace)
    unreachable    the gold path is outside the search space: fix the dictionary (`missing_words()`)
    search_error   the gold path scores higher than the path found, which the beam pruned: a larger beam
    model_error    the model prefers the wrong path: more training, or more features

Levels of word matching: `seg` (b, e), `tag` (b, e, tag0, tag1), `full` (b, e, tags, morphemes) count words;
`morph` counts units, (morph0, tag0) of every word and (morph1, tag1) of two-morpheme words, matched within
words of equal span.
"""

from collections import Counter

import numpy as np

from .. import _native

CLASSES = ('correct', 'failed', 'unreachable', 'search_error', 'model_error')
LEVELS = ('seg', 'tag', 'full', 'morph')
REASONS = {_native.LT_GOLD_OK: 'ok', _native.LT_GOLD_BREAKS_TILING: 'breaks_tiling',
           _native.LT_GOLD_BEYOND_WINDOW: 'beyond_window', _native.LT_GOLD_NOT_IN_LATTICE: 'not_in_lattice',
           _native.LT_GOLD_UNK_AFTER_UNK: 'unk_after_unk', _native.LT_GOLD_UNCHECKED: 'unchecked'}
# (gold, predicted, matched) columns of the counts per level
_COLUMNS = {
    'seg': (_native.LT_EVAL_GOLD_WORDS, _native.LT_EVAL_PRED_WORDS, _native.LT_EVAL_SEG),
    'tag': (_native.LT_EVAL_GOLD_WORDS, _native.LT_EVAL_PRED_WORDS, _native.LT_EVAL_TAG),
    'full': (_native.LT_EVAL_GOLD_WORDS, _native.LT_EVAL_PRED_WORDS, _native.LT_EVAL_FULL),
    'morph': (_native.LT_EVAL_GOLD_UNITS, _native.LT_EVAL_PRED_UNITS, _native.LT_EVAL_UNIT_MATCH),
}


class Evaluation:
    """Per-sentence results (numpy arrays, in the order of the evaluated sentences) and their totals.

    sent_class        uint8, index into `CLASSES` (= the LT_EVAL_* codes)
    counts            int32 [n, 8]: gold words, predicted words, seg / tag / full matches, gold units,
                      predicted units, unit matches (LT_EVAL_GOLD_WORDS ...)
    gold_scores       float64, the model's score of the gold path's image; NaN unless it is reachable
    predicted_scores  float64, the score of the path found; NaN where the search did not tag the sentence
    status            int32 LT_SENT_* of the search
    word_reason       list of uint8 arrays, one code per gold word (LT_GOLD_*, names in `REASONS`)
    golds             list of the gold words of each sentence (BOS / EOS left out)
    indices           position of each evaluated sentence in the caller's input
    not_evaluated     positions in the caller's input that were left out of every count
    """

    def __init__(self, sent_class, counts, gold_scores, predicted_scores, status, word_reason, golds, indices=None,
                 not_evaluated=()):
        self.sent_class = sent_class
        self.counts = counts
        self.gold_scores = gold_scores
        self.predicted_scores = predicted_scores
        self.status = status
        self.word_reason = word_reason
        self.golds = golds
        self.indices = list(range(len(sent_class))) if indices is None else list(indices)
        self.not_evaluated = list(not_evaluated)

    def __len__(self):
        return len(self.sent_class)

    @property
    def exact(self):
        """Per sentence: the best path is the gold path."""
        return self.sent_class == _native.LT_EVAL_CORRECT

    @property
    def class_counts(self):
        """{class name: number of sentences}, every class present."""
        got = np.bincount(self.sent_class, minlength=len(CLASSES))
        return {name: int(got[i]) for i, name in enumerate(CLASSES)}

    def totals(self, level='full'):
        """(gold, predicted, matched) summed over the sentences at `level` ('seg', 'tag', 'full', 'morph')."""
        if level not in _COLUMNS:
            raise ValueError('level must be one of %s' % (LEVELS,))
        return tuple(int(self.counts[:, c].sum()) for c in _COLUMNS[level])

    def precision(self, level='full'):
        _, predicted, matched = self.totals(level)
        return matched / predicted if predicted else 0.0

    def recall(self, level='full'):
        gold, _, matched = self.totals(level)
        return matched / gold if gold else 0.0

    def f1(self, level='full'):
        gold, predicted, matched = self.totals(level)
        return 2.0 * matched / (gold + predicted) if gold + predicted else 0.0

    def missing_words(self):
        """Counter of (morph0, tag0, morph1, tag1) over the gold words the lattice does not contain
        (LT_GOLD_NOT_IN_LATTICE): the entries a dictionary lacks for these gold paths."""
        out = Counter()
        for words, reasons in zip(self.golds, self.word_reason):
            for w, r in zip(words, reasons.tolist()):
                if r == _native.LT_GOLD_NOT_IN_LATTICE:
                    out[w.morph0, w.tag0, w.morph1, w.tag1] += 1
        return out

    def __repr__(self):
        return 'Evaluation(%d sentences, %s, full F1 %.4f)' % (len(self), self.class_counts, self.f1('full'))


def ordered(paths):
    """Every word with b < e and b strictly increasing along its path (what lt_evaluate requires)."""
    for words in paths:
        prev = -1
        for w in words:
            if not (w.b < w.e and w.b > prev):
                return False
            prev = w.b
    return True


def evaluate_pathset(engine, sents, golds, pathset, beam_size, indices=None, not_evaluated=()):
    """One decode of `sents` and one lt_evaluate against `pathset` (the uploaded `golds`) -> `Evaluation`."""
    _, _, scores, status = engine.tag_packed(sents, beam_size)
    sent_class, counts, gold_scores, word_reason = engine.evaluate(pathset)
    predicted = np.where(status == _native.LT_SENT_OK, scores, np.nan)
    off = pathset.path_off.tolist()
    reasons = [word_reason[off[i]:off[i + 1]] for i in range(len(sents))]
    return Evaluation(sent_class, counts, gold_scores, predicted, status, reasons, golds, indices, not_evaluated)
