"""The constrained beam search, spelled out on the host: the specification `lt_batch_set_constraints` and the
`constraints=` keyword of `Tagger.tag_batch` are tested against (include/lt_b200.h, DESIGN.md "Constrained search").

`beam_search(..., constraints=None)` is `oracle.lattice_oracle.beam_search` itself.  With a list of `(b, e, tag)`
constraints (tag a tag name, or None for any word) it is that search with three changes to the candidates of end e
and begin b:
  1. (b, e) is blocked when a constraint overlaps it without being equal to it: no candidate at all;
  2. (b, e) equal to a constraint: its lattice edges of the constraint's tag (all for None); if there is none, the
     unknown word for None, else the forced word (chars[b:e], chars[b:e], None, tag, None, e - b, b, e, is_l);
  3. an unknown word may follow an unknown word only from the first begin the constraints leave open.
"""

from oracle import lattice_oracle as lo

B, E, TAG0 = 6, 7, 3


class BadConstraint(Exception):
    """A constraint ends beyond the sentence: LT_SENT_BAD_CONSTRAINT."""


def is_l_of(sent):
    """Per syllable of the space-stripped sentence: is it the first syllable of an eojeol."""
    out = []
    for i, ch in enumerate(sent):
        if ch != ' ':
            out.append(i == 0 or sent[i - 1] == ' ')
    return out


def blocked(b, e, constraints):
    return any(b < ce and cb < e and (b, e) != (cb, ce) for cb, ce, _ in constraints)


def exact(b, e, constraints):
    for c in constraints:
        if (c[0], c[1]) == (b, e):
            return c
    return None


def open_begins(e, constraints):
    return [b for b in range(max(0, e - lo.WINDOW), e) if not blocked(b, e, constraints)]


def candidates(bindex, chars, is_l, b, e, constraints):
    """The words of span (b, e) by rules 1 and 2 (the span must not be blocked)."""
    expansions = [edge for edge in bindex[b] if edge[E] == e]
    c = exact(b, e, constraints)
    sub = chars[b:e]
    if c is not None and c[2] is not None:
        expansions = [edge for edge in expansions if edge[TAG0] == c[2]]
        if not expansions:
            return [(sub, sub, None, c[2], None, e - b, b, e, is_l[b])]
    if not expansions:
        expansions = [(sub, sub, None, lo.UNK, None, e - b, b, e, False)]
    return expansions


def beam_search(bindex, chars, program, beam_size=5, counters=None, constraints=None, is_l=None):
    if constraints is None:
        return lo.beam_search(bindex, chars, program, beam_size, counters)
    constraints = [tuple(c) + (None,) * (3 - len(c)) for c in constraints]
    length = len(chars)
    if length and not bindex:
        raise IndexError('list index out of range')          # as the unconstrained search: no dictionary edge
    if any(ce > length for _, ce, _ in constraints):
        raise BadConstraint()
    bos = (lo.BOS, lo.BOS, None, lo.BOS, None, 0, 0, 0, False)
    eos = (lo.EOS, lo.EOS, None, lo.EOS, None, 0, length, length, False)
    beams = [[lo.Hypothesis([bos], 0)]]
    for e in range(1, length + 1):
        grown = []
        opens = open_begins(e, constraints)
        for b in opens:
            for hyp in beams[b]:
                for edge in candidates(bindex, chars, is_l, b, e, constraints):
                    if hyp.num_unk > 0 and edge[TAG0] == lo.UNK and b != opens[0]:
                        continue
                    word_i = None if len(hyp.words) == 1 else hyp.words[-2]
                    grown.append(hyp.extended(edge, program.increment(word_i, hyp.words[-1], edge, counters)))
        beams.append(sorted(grown, key=lambda h: -h.score)[:beam_size])
    return [h.extended(eos, 0) for h in beams[-1]]


def survivors(oracle, sent, beam_size, constraints=None):
    """`OracleTagger.survivors` with constraints: every survivor, best first."""
    chars = sent.replace(' ', '')
    edges = oracle.lattice(sent)
    return beam_search(lo.begin_index(sent, edges), chars, oracle.program, beam_size, constraints=constraints,
                       is_l=is_l_of(sent))


def brute_force(bindex, chars, program, constraints, is_l):
    """Every complete path of the constrained search space, enumerated from rules 1-3 directly: list of
    (words without BOS / EOS, score)."""
    constraints = [tuple(c) + (None,) * (3 - len(c)) for c in constraints]
    length = len(chars)
    bos = (lo.BOS, lo.BOS, None, lo.BOS, None, 0, 0, 0, False)
    out = []

    def walk(b, words, score):
        if b == length:
            out.append((words[1:], score))
            return
        for e in range(b + 1, min(length, b + lo.WINDOW) + 1):
            if blocked(b, e, constraints):
                continue
            for edge in candidates(bindex, chars, is_l, b, e, constraints):
                if words[-1][TAG0] == lo.UNK and edge[TAG0] == lo.UNK and b != open_begins(e, constraints)[0]:
                    continue
                word_i = None if len(words) == 1 else words[-2]
                walk(e, words + [edge], score + program.increment(word_i, words[-1], edge))

    walk(0, [bos], 0)
    return out
