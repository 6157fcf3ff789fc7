"""Trainer around the batched GPU decoder (SURVEY §8f, row f2).

The reference's `train()` (`trainer/train.py:1-42`) scans the features of a tagged corpus, builds
`BeamScoreFunctions(regularity_func, score_func.set_encoder(encoder))`, creates a `Tagger` and
calls `fit_parameter` -> `train_epoch` — which is a stub there (`train.py:61-65` returns `coef`
unchanged, and `train()` itself stops on undefined names before it gets that far).  This module
keeps the reference's functions, arguments and result format (`{'idx_to_feature',
'coefficient'}`, `train.py:34-37`) and supplies the missing epoch: a structured perceptron whose
decoding step is `Tagger.tag_batch` — the whole corpus in one device pass per epoch.

    w <- w + phi(gold) - phi(predicted)          for every sentence whose prediction is not the gold path

with phi = counts of the trigram features of a path (`SimpleTrigramEncoder.encode_sequence`,
`features/feature.py:62-68`).  All sentences of an epoch are decoded with the same weights (the
updates of one epoch are summed).  The gold paths go to the device once per `fit_parameter` call; an
epoch is then a weight update, one decode of the corpus and one `lt_perceptron_delta` call, which
compares every prediction with its gold path and counts the features of both on the device.

With `batch_size` the perceptron is online instead: the corpus is cut into consecutive mini-batches, and
each one is decoded with the weights the previous ones left (`lt_trainer_step`), optionally averaged over
all steps.  The weights and their running average then stay on the device for the whole run.  `update` picks
the prefix a mini-batch step updates on: 'full' (the whole path), 'early' (up to the first gold word that fell out
of the beam) or 'max_violation' (where the best hypothesis beats the gold prefix by the most); see
`lt_trainer_set_update`.
There is no CPU decoder: without the CUDA library `Tagger` raises.
"""

import numpy as np

from ..beam import BeamScoreFunctions
from ..dictionary.text import text_to_words
from ..features.utils import scan_features
from ..compile import _is_bmp
from ..tagger import Tagger
from ..tagset import BUILTIN_TAGS, MAX_TAGS


def _surface(word_text):
    """'너무너무너무 는  아이오아이 의' -> '너무너무너무는 아이오아이의' (the string `Tagger.tag` receives)."""
    return ' '.join(eojeol.replace(' ', '') for eojeol in word_text.split('  '))


def _same_path(predicted, gold):
    """Word-by-word identity of two [BOS .. EOS] lists on what the annotation defines:
    span, morphemes and tags (`Word.len` and `Word.is_l` follow from those)."""
    if len(predicted) != len(gold):
        return False
    for p, g in zip(predicted, gold):
        if (p.b, p.e, p.morph0, p.morph1, p.tag0, p.tag1) != (g.b, g.e, g.morph0, g.morph1, g.tag0, g.tag1):
            return False
    return True


def train(word_morph_pairs, dictionary, encoder, score_func, regularity_func,
          max_epochs=100, min_feature_count=1, predefined_features=None,
          verbose=False, debug=False, beam_size=5, device=0, batch_size=None, averaged=False, update='full'):
    """Reference `train()` (`trainer/train.py:1-42`): -> {'idx_to_feature': [...], 'coefficient': [...]}
    `batch_size`, `averaged` and `update` are passed to `fit_parameter`."""
    _check_update(update, batch_size)
    word_morph_pairs = list(word_morph_pairs)
    if verbose:
        print('Scanning features ...')
    if predefined_features is None:
        # length-of-unknown-word features (template 6), lengths 1..8 (`train.py:9-12`)
        predefined_features = {(6, length): min_feature_count for length in range(1, 9)}

    idx_to_feature, feature_to_idx, idx_to_feature_count = scan_features(
        word_morph_pairs, encoder, min_count=min_feature_count, verbose=verbose, debug=debug,
        predefined_features=predefined_features)

    encoder.feature_dic = feature_to_idx
    funcs = BeamScoreFunctions(regularity_func, score_func.set_encoder(encoder))
    tagger = Tagger(dictionary, encoder=encoder, score_funcs=funcs, device=device,
                    extra_tags=_gold_tags(word_morph_pairs, dictionary))

    if verbose:
        print('Estimating parameter ...')
    try:
        coef = fit_parameter(word_morph_pairs, encoder, tagger, max_epochs, verbose=verbose, beam_size=beam_size,
                             averaged=averaged, batch_size=batch_size, update=update)
    finally:
        tagger.close()

    params = {'idx_to_feature': idx_to_feature, 'coefficient': [float(c) for c in coef]}
    if debug:
        params['idx_to_feature_count'] = idx_to_feature_count
    return params


def _gold_tags(word_morph_pairs, dictionary):
    """Tags of the annotation that the dictionary lacks, as long as the device tables can hold them all: gold
    paths that name them are then evaluated on the device, and the features that name them are kept in the
    tables (no dictionary word carries such a tag, so decoding is unchanged)."""
    known = set(BUILTIN_TAGS) | set(dictionary.tag_to_morphs)
    extra = {}
    for word_text, morph_text in word_morph_pairs:
        try:
            words = text_to_words(word_text, morph_text)
        except Exception:
            continue
        for w in words:
            for tag in (w.tag0, w.tag1):
                if tag is not None and tag not in known:
                    extra[tag] = None
    return list(extra) if len(known) + len(extra) <= MAX_TAGS else []


class _GoldCorpus:
    """The annotation of a corpus, parsed and packed once: the surfaces the tagger receives, the gold
    paths of the sentences the device can compare (uploaded as a path set on the tagger's tables), and
    the rest — text outside the BMP, a tag the tables do not know — for the host loop."""

    def __init__(self, word_morph_pairs, tagger):
        self.golds, self.sents, self.pair_idx = [], [], []
        for p, (word_text, morph_text) in enumerate(word_morph_pairs):
            try:
                gold = text_to_words(word_text, morph_text)
            except Exception:                          # malformed pairs are skipped, as scan_features does
                continue
            self.golds.append(gold)
            self.sents.append(_surface(word_text))
            self.pair_idx.append(p)
        self.pathset = self.tables = None
        self.device_idx, self.host_idx = list(range(len(self.golds))), []
        engine = tagger._engine
        if tagger.eojeol_lookup.flatten:                # no lt_tag_batch_host paths: everything on the host
            self.device_idx, self.host_idx = [], self.device_idx
            return
        tag_ids = engine.tables.tag_ids
        usable, rest = [], []
        for i, (gold, sent) in enumerate(zip(self.golds, self.sents)):
            ok = _is_bmp(sent) and all(_is_bmp(w.word) and _is_bmp(w.morph0) and (w.morph1 is None or _is_bmp(w.morph1)) and
                                       w.tag0 in tag_ids and (w.tag1 is None or w.tag1 in tag_ids) for w in gold[1:-1])
            (usable if ok else rest).append(i)
        self.device_idx, self.host_idx = usable, rest
        self.device_sents = [self.sents[i] for i in usable]
        self.pathset = engine.upload_paths([self.golds[i][1:-1] for i in usable])
        self.tables = engine.tables

    def close(self):
        if self.pathset is not None:
            self.pathset.close()
            self.pathset = None


def evaluate(word_morph_pairs, tagger, beam_size=5):
    """The tagger's output on an annotated corpus (`word_morph_pairs` as for `train`) against the annotation,
    on the device: one decode, one `lt_evaluate` -> `Evaluation` (classes, precision / recall / F1 per level,
    gold-path scores, `missing_words()`).  Pairs the device cannot compare are listed by position in
    `Evaluation.not_evaluated` and left out of every count: a malformed annotation, text outside the BMP, a
    tag the tagger's tables do not know.  `Evaluation.indices` gives the position of each evaluated pair.
    A `flatten=True` tagger raises `ValueError` (see `Tagger.evaluate`)."""
    from ..tagger.evaluation import evaluate_pathset, ordered
    if tagger.eojeol_lookup.flatten:
        raise ValueError('evaluate() does not support a flatten=True lookup: its lattices hold single-morpheme words')
    word_morph_pairs = list(word_morph_pairs)
    gold = _GoldCorpus(word_morph_pairs, tagger)
    try:
        golds = [gold.golds[i][1:-1] for i in gold.device_idx]
        if not ordered(golds):
            raise ValueError('an annotation yields a word with b >= e or out of order')
        indices = [gold.pair_idx[i] for i in gold.device_idx]
        parsed = set(gold.pair_idx)
        left_out = sorted([p for p in range(len(word_morph_pairs)) if p not in parsed] + [gold.pair_idx[i] for i in gold.host_idx])
        return evaluate_pathset(tagger._engine, gold.device_sents, golds, gold.pathset, beam_size, indices, left_out)
    finally:
        gold.close()


UPDATE_MODES = ('full', 'early', 'max_violation')


def _check_update(update, batch_size):
    if update not in UPDATE_MODES:
        raise ValueError('update must be one of %s, got %r' % (', '.join(UPDATE_MODES), update))
    if update != 'full' and batch_size is None:
        raise ValueError("update=%r needs batch_size: it reads the back-pointers of each mini-batch's search on the device "
                         "(one decode of the whole corpus is batch_size=len(corpus))" % (update,))


def fit_parameter(word_morph_pairs, encoder, tagger, max_epochs=100, verbose=False, beam_size=5, patience=5,
                  averaged=False, batch_size=None, update='full'):
    """Reference `fit_parameter()` (`train.py:44-59`).  Stops once an epoch makes no mistake, or when the
    number of mistakes has not improved for `patience` epochs (a corpus with an unreachable gold path — a word the
    dictionary cannot produce — never reaches zero); returns the best weights seen (`averaged=True`: the mean of
    the weights of all epochs, the averaged perceptron).

    With an integer `batch_size`: mini-batch perceptron steps on the device, see `_fit_minibatch`; `update` ('full',
    'early' or 'max_violation') is their update, and anything but 'full' needs `batch_size`."""
    _check_update(update, batch_size)
    if batch_size is not None:
        return _fit_minibatch(word_morph_pairs, encoder, tagger, max_epochs, verbose, beam_size, patience, averaged, batch_size,
                              update)
    coef = np.zeros(len(encoder.feature_dic), dtype=np.float64)
    best_loss, best_coef, stale = None, coef, 0
    total = np.zeros_like(coef)
    epochs = 0
    _load_weights(tagger, encoder, coef)               # the tables the gold paths are uploaded to
    gold = _GoldCorpus(word_morph_pairs, tagger)
    try:
        for epoch in range(1, max_epochs + 1):
            decoded_with = coef
            coef, loss = train_epoch(word_morph_pairs, encoder, tagger, coef, epoch, verbose, beam_size=beam_size, gold=gold)
            total += coef
            epochs += 1
            if best_loss is None or loss < best_loss:
                best_loss, best_coef, stale = loss, decoded_with, 0       # `loss` was measured with the weights the epoch started from
            else:
                stale += 1
            if loss == 0 or stale >= patience:
                break
    finally:
        gold.close()
    if averaged:
        return total / max(1, epochs)
    return best_coef


def _fit_minibatch(word_morph_pairs, encoder, tagger, max_epochs, verbose, beam_size, patience, averaged, batch_size, update):
    """The online perceptron: the sentences the device can compare, in corpus order, cut into consecutive mini-batches
    of `batch_size` (the last one may be shorter); every epoch walks them in that order, one `lt_trainer_step` each.
    An epoch's loss is its number of mistakes; it stops on loss 0 or after `patience` epochs without a new minimum.
    Returns the weights after the last step (`averaged=True`: their mean over all steps) — not the "best" ones, since an
    online epoch's mistakes measure no single weight vector — and leaves them in the scorer and the tables.  Pairs the
    device cannot compare are left out."""
    if tagger.eojeol_lookup.flatten:
        raise ValueError('mini-batch training does not support a flatten=True lookup: its lattices hold single-morpheme words')
    if int(batch_size) != batch_size or batch_size < 1:
        raise ValueError('batch_size must be a positive integer, got %r' % (batch_size,))
    batch_size = int(batch_size)
    coef = np.zeros(len(encoder.feature_dic), dtype=np.float64)
    scorer = _load_weights(tagger, encoder, coef)
    word_morph_pairs = list(word_morph_pairs)
    gold = _GoldCorpus(word_morph_pairs, tagger)
    try:
        n = len(gold.device_idx)
        if verbose:
            print('mini-batch training on %d of %d pairs (%d left out: malformed, outside the BMP or an unknown tag)'
                  % (n, len(word_morph_pairs), len(word_morph_pairs) - n))
        if n:
            engine = tagger._engine
            func = tagger.score_funcs.funcs.index(scorer)
            desc_func, desc_fdic = engine.tables.desc_sources()
            feat_coef = np.where(desc_func == func, desc_fdic, -1)
            trainer = engine.trainer(gold.device_sents, gold.pathset, func, len(coef), feat_coef, coef, update=update)
            try:
                best_loss, stale, seen = None, 0, 0
                for epoch in range(1, max_epochs + 1):
                    for first in range(0, n, batch_size):
                        trainer.step(first, min(batch_size, n - first), beam_size)
                    w, mean, steps, mistakes, _ = trainer.fetch()
                    loss, seen = mistakes - seen, mistakes
                    if verbose:
                        print('epoch %d: %d of %d sentences differ from the annotation (%d steps)' % (epoch, loss, n, steps))
                    if best_loss is None or loss < best_loss:
                        best_loss, stale = loss, 0
                    else:
                        stale += 1
                    if loss == 0 or stale >= patience:
                        break
                coef = mean if averaged else w
            finally:
                trainer.close()
    finally:
        gold.close()
    _load_weights(tagger, encoder, coef)
    return coef


def _trigram_scorer(tagger):
    from ..beam import SimpleTrigramFeatureScore
    for func in tagger.score_funcs.funcs:
        if isinstance(func, SimpleTrigramFeatureScore):
            return func
    raise ValueError('the tagger has no SimpleTrigramFeatureScore to train')


def _load_weights(tagger, encoder, coef):
    """Put `coef` into the tagger's trigram scorer and the device tables; -> the scorer."""
    scorer = _trigram_scorer(tagger)
    if scorer.encoder is encoder and scorer.coefficients is not None and len(scorer.coefficients) == len(coef) \
            and getattr(tagger, '_trained_features', None) is encoder.feature_dic:
        scorer.coefficients = coef
        tagger.update_weights()                        # same features as the device tables hold: weights in place
    else:
        scorer.set_encoder(encoder, coef)
        tagger.refresh()                               # first epoch: feature table compiled once
        tagger._trained_features = encoder.feature_dic
    return scorer


def train_epoch(word_morph_pairs, encoder, tagger, coef, epoch, verbose, beam_size=5, gold=None):
    """One perceptron pass (the reference's TODO, `train.py:61-65`): -> (coef, loss).

    loss = number of sentences whose best path under `coef` differs from the annotation.  `gold`: the
    corpus as `fit_parameter` prepared it (parsed and uploaded once for all epochs).  The sentences on the
    device are decoded, compared and counted there (`lt_perceptron_delta`); the update of an epoch is a sum
    of +-1 counts, so it is exact in any order.
    """
    coef = np.asarray(coef, dtype=np.float64).copy()
    scorer = _load_weights(tagger, encoder, coef)
    own = gold is None or gold.pathset is not None and gold.tables is not tagger._engine.tables
    if own:
        gold = _GoldCorpus(word_morph_pairs, tagger)
    try:
        update = np.zeros_like(coef)
        loss = 0
        if gold.device_idx:
            engine = tagger._engine
            func = tagger.score_funcs.funcs.index(scorer)
            engine.tag_packed(gold.device_sents, beam_size)
            delta, _, n_differ = engine.perceptron_delta(gold.pathset, func)
            desc_func, desc_fdic = engine.tables.desc_sources()
            hit = np.flatnonzero((desc_func == func) & (delta != 0))
            np.add.at(update, desc_fdic[hit], delta[hit].astype(np.float64))     # a feature_dic need not be one-to-one
            loss += n_differ
        if gold.host_idx:
            loss += _host_update(encoder, tagger, [gold.golds[i] for i in gold.host_idx],
                                 [gold.sents[i] for i in gold.host_idx], beam_size, update)
    finally:
        if own:
            gold.close()
    coef += update
    if verbose:
        print('epoch %d: %d of %d sentences differ from the annotation' % (epoch, loss, len(gold.golds)))
    return coef, loss


def _host_update(encoder, tagger, golds, sents, beam_size, update):
    """The epoch's counting on the host for sentences the device cannot compare: update += phi(gold) -
    phi(predicted) per mistaken sentence; -> the number of mistakes."""
    predicted = tagger.tag_batch(sents, beam_size=beam_size, errors='none')
    loss = 0
    for gold, seq in zip(golds, predicted):
        if seq is not None and _same_path(seq.sequences, gold):
            continue
        loss += 1
        for idxs in encoder.encode_sequence(gold):
            for idx in idxs:
                update[idx] += 1.0
        if seq is not None:
            for idxs in encoder.encode_sequence(seq.sequences):
                for idx in idxs:
                    update[idx] -= 1.0
    return loss
