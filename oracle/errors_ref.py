"""Plain-Python restatement of the recognition-error output W2S_OUT_ERRORS (include/w2s.h): greedy decode, word split
and Levenshtein distance on lists of label ids."""
from __future__ import annotations

import numpy as np

LABELS, WORDS = "labels", "words"


def greedy_ids(frame_logits, blank: int = 0) -> list:
    """Per-frame argmax (the lowest id among equal maxima, as numpy.argmax), repeats collapsed, then blanks dropped."""
    out, prev = [], None
    for row in np.asarray(frame_logits):
        a = int(np.argmax(row))
        if a != prev and a != blank:
            out.append(a)
        prev = a
    return out


def split_words(ids, delimiter: int = 4) -> list:
    """Runs of labels between delimiters, as tuples; empty runs (leading, trailing, repeated delimiters) dropped."""
    words, cur = [], []
    for v in ids:
        if v == delimiter:
            if cur:
                words.append(tuple(cur))
            cur = []
        else:
            cur.append(v)
    if cur:
        words.append(tuple(cur))
    return words


def levenshtein(a, b) -> int:
    """Unit-cost edit distance (substitution, insertion, deletion) between two sequences, compared element by element."""
    prev = list(range(len(b) + 1))
    for i, x in enumerate(a, 1):
        cur = [i] + [0] * len(b)
        for j, y in enumerate(b, 1):
            cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (x != y))
        prev = cur
    return prev[len(b)]


def errors(hyp_ids, ref_ids, unit: str = WORDS, delimiter: int = 4) -> int:
    if unit == LABELS:
        return levenshtein(list(hyp_ids), list(ref_ids))
    return levenshtein(split_words(hyp_ids, delimiter), split_words(ref_ids, delimiter))


def evaluate(logits, refs, unit: str = WORDS, blank: int = 0, delimiter: int = 4) -> np.ndarray:
    """logits [n, T, V] -> [n, D] float64: the edit distance of every row's greedy transcript to every reference."""
    logits = np.asarray(logits)
    out = np.zeros((logits.shape[0], len(refs)))
    for r in range(logits.shape[0]):
        hyp = greedy_ids(logits[r], blank)
        for d, y in enumerate(refs):
            out[r, d] = errors(hyp, [int(v) for v in y], unit, delimiter)
    return out
