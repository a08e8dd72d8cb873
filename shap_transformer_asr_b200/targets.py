"""Target selection: which (frame, token) outputs a clip is explained for (host side, once per clip)."""
from __future__ import annotations

import numpy as np

PAD_ID = 0     # CTC blank (<pad>), shap_calculation.py:221-254 / visualization.py:320-321
SPACE_ID = 4   # "|"
MAX_TRANSCRIPT = 512   # W2S_MAX_TRANSCRIPT (include/w2s.h)


def greedy_transcript(logits, blank: int = PAD_ID) -> np.ndarray:
    """The model's own greedy transcription of a clip as CTC label ids: the per-frame argmax with repeats collapsed and
    blanks dropped (int32 [U]; empty when every frame's argmax is the blank).  ``metrics.greedy_ctc_decode`` maps the
    same argmax sequence to its string."""
    ids = np.asarray(logits).argmax(-1).reshape(-1)
    keep = ids != blank
    keep[1:] &= ids[1:] != ids[:-1]
    return ids[keep].astype(np.int32)


def reference_length(ref, unit: str = "words", delimiter: int = SPACE_ID) -> int:
    """Units N of a reference of the recognition-error output: its labels, or its words -- the runs between
    ``delimiter`` labels, empty ones dropped.  Error counts divided by N are the label or word error rates."""
    y = np.asarray(ref).reshape(-1)
    if unit == "labels":
        return int(y.size)
    word = y != delimiter
    return int(np.count_nonzero(word[1:] & ~word[:-1]) + (word.size > 0 and word[0]))


def frames_needed(transcript) -> int:
    """Frames a CTC alignment of ``transcript`` needs: one per label plus one blank between equal adjacent labels."""
    y = np.asarray(transcript).reshape(-1)
    return int(y.size + np.count_nonzero(y[1:] == y[:-1]))


def transcript_arrays(transcripts, blank: int = PAD_ID, vocab_size: int = None):
    """Validated packed form of ``transcripts`` (a list of label-id sequences, or one sequence of ints) for
    ``w2s_set_transcripts``: (labels int32 [sum U], offsets int32 [D + 1]).  Raises ValueError, before any library call,
    for no transcripts, a transcript longer than MAX_TRANSCRIPT, a label outside [0, vocab_size) or equal to ``blank``,
    and ``blank`` outside [0, vocab_size)."""
    if isinstance(transcripts, np.ndarray) and transcripts.ndim == 1 or \
            (isinstance(transcripts, (list, tuple)) and transcripts and np.isscalar(transcripts[0])):
        transcripts = [transcripts]
    seqs = [np.asarray(t, dtype=np.int64).reshape(-1) for t in transcripts]
    if not seqs:
        raise ValueError("need at least one transcript (D >= 1)")
    if vocab_size is not None and not 0 <= blank < vocab_size:
        raise ValueError(f"blank {blank} outside the vocabulary [0, {vocab_size})")
    for d, y in enumerate(seqs):
        if y.size > MAX_TRANSCRIPT:
            raise ValueError(f"transcript {d} has {y.size} labels, at most {MAX_TRANSCRIPT} are supported")
        if y.size and (y.min() < 0 or (vocab_size is not None and y.max() >= vocab_size)):
            raise ValueError(f"transcript {d}: label outside the vocabulary [0, {vocab_size})")
        if np.any(y == blank):
            raise ValueError(f"transcript {d}: label equal to the blank {blank}")
    offsets = np.zeros(len(seqs) + 1, dtype=np.int32)
    offsets[1:] = np.cumsum([y.size for y in seqs])
    labels = np.ascontiguousarray(np.concatenate(seqs) if offsets[-1] else np.zeros(0), dtype=np.int32)
    return labels, offsets


def check_offsets(offsets, num_labels: int) -> np.ndarray:
    """Explicit offsets [D + 1] into a flat label array: D >= 1, offsets[0] == 0, non-decreasing, offsets[-1] ==
    num_labels.  Raises ValueError otherwise."""
    o = np.asarray(offsets, dtype=np.int64).reshape(-1)
    if o.size < 2:
        raise ValueError("need at least one transcript (D >= 1)")
    if o[0] != 0 or o[-1] != num_labels:
        raise ValueError(f"offsets must start at 0 and end at the label count {num_labels}")
    if np.any(np.diff(o) < 0):
        raise ValueError("offsets must be non-decreasing")
    return np.ascontiguousarray(o, dtype=np.int32)


def char_targets(logits, pad_id: int = PAD_ID, space_id: int = SPACE_ID, all_frames_if_empty: bool = True):
    """Per-character frames (visualization.py:319-327): greedy argmax, keep the frames where a new
    non-blank, non-'|' token starts; the explained token is that frame's unmasked argmax
    (feasability_tests/w2v2conformer.py:97-108).  With random-init weights the set can be empty; then
    every frame with its argmax token is used."""
    ids = np.asarray(logits).argmax(-1)
    keep = (ids != pad_id) & (ids != space_id)
    keep[1:] &= ids[1:] != ids[:-1]
    frames = np.nonzero(keep)[0].astype(np.int32)
    if frames.size == 0 and all_frames_if_empty:
        frames = np.arange(len(ids), dtype=np.int32)
    return frames, ids[frames].astype(np.int32)


def first_char_target(logits, special_ids=(0, 1, 2, 3), space_id: int = SPACE_ID):
    """feasability_tests/w2v2conformer.py:93-110: the first non-special, non-'|' frame, else the middle."""
    ids = np.asarray(logits).argmax(-1)
    for i, t in enumerate(ids):
        if int(t) not in special_ids and int(t) != space_id:
            return int(i), int(t)
    mid = len(ids) // 2
    return int(mid), int(ids[mid])
