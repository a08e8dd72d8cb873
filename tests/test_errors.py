"""CPU: the recognition-error output W2S_OUT_ERRORS -- the oracle against a brute-force DP and against metrics.wer, the
host tables of w2s_set_references (decoded, and driven through a lane-by-lane restatement of the device's bit-parallel
step), and the argument checks, which raise before the library is called."""
import dataclasses

import numpy as np
import pytest

from helpers import VARIANTS
from oracle import errors_ref as ER
from shap_transformer_asr_b200 import metrics, targets
from shap_transformer_asr_b200.engine import Engine, error_tables

DELIM = targets.SPACE_ID


def brute_force_distance(a, b):
    """The edit distance as the shortest path through the full (|a| + 1) x (|b| + 1) grid, by relaxation to a fixpoint."""
    INF = 1 << 30
    D = np.full((len(a) + 1, len(b) + 1), INF, dtype=np.int64)
    D[0, 0] = 0
    changed = True
    while changed:
        changed = False
        for i in range(len(a) + 1):
            for j in range(len(b) + 1):
                best = D[i, j]
                if i:
                    best = min(best, D[i - 1, j] + 1)
                if j:
                    best = min(best, D[i, j - 1] + 1)
                if i and j:
                    best = min(best, D[i - 1, j - 1] + (a[i - 1] != b[j - 1]))
                if best < D[i, j]:
                    D[i, j] = best
                    changed = True
    return int(D[len(a), len(b)])


def test_levenshtein_matches_a_brute_force_grid():
    rng = np.random.default_rng(0)
    for _ in range(150):
        a = list(rng.integers(0, 4, rng.integers(0, 9)))
        b = list(rng.integers(0, 4, rng.integers(0, 9)))
        assert ER.levenshtein(a, b) == brute_force_distance(a, b), (a, b)
    assert ER.levenshtein([], [1, 2, 3]) == 3 and ER.levenshtein([1, 2], []) == 2
    assert ER.levenshtein([(1, 2), (3,)], [(3,), (1, 2)]) == 2


def test_greedy_ids_ties_collapse_and_blanks():
    V = 40
    z = np.zeros((6, V))
    z[0, [7, 39]] = 1.0            # tie across lanes of one id block: 7 wins
    z[1, [3, 35]] = 1.0            # tie inside a lane (3 and 3 + 32): 3 wins
    z[2, 0] = 1.0                  # blank
    z[3, 3] = 1.0                  # 3 again after a blank: a new label
    z[4, [3, 2]] = 1.0             # tie 2 / 3: 2
    z[5, 2] = 1.0                  # repeat of 2: collapsed
    assert ER.greedy_ids(z, blank=0) == [7, 3, 3, 2]
    assert ER.greedy_ids(z, blank=3) == [7, 0, 2]
    rng = np.random.default_rng(1)
    for _ in range(20):
        lg = np.round(rng.standard_normal((40, 33)), 1)      # rounded: many exact ties
        assert ER.greedy_ids(lg, 5) == targets.greedy_transcript(lg, 5).tolist()


def test_split_words_drops_empty_words():
    assert ER.split_words([4, 4, 5, 6, 4, 4, 7, 4], 4) == [(5, 6), (7,)]
    assert ER.split_words([4, 4], 4) == [] and ER.split_words([], 4) == []


def _text(ids):
    """labels -> the string metrics.greedy_ctc_decode would print for them (the label sequence is not collapsed)"""
    return " ".join("".join(" " if t == DELIM else metrics.VOCAB[t] for t in ids).split())


def test_word_errors_equal_wer_times_words_on_vocab_strings():
    rng = np.random.default_rng(2)
    alphabet = [4, 4, 4, 5, 6, 7, 1, 2, 3, 27]         # delimiters, letters and the multi-character special tokens
    for _ in range(300):
        ref = [int(v) for v in rng.choice(alphabet, rng.integers(0, 25))]
        if rng.random() < 0.3:                         # repeated labels in the reference stay as they are
            ref = [v for v in ref for _ in (0, 1)]
        hyp = [int(v) for v in rng.choice(alphabet, rng.integers(0, 25))]
        if rng.random() < 0.5 and ref:                 # a few edits of the reference: many equal words
            hyp = list(ref)
            for _ in range(rng.integers(0, 4)):
                hyp[rng.integers(0, len(hyp))] = int(rng.choice(alphabet))
        n_words = targets.reference_length(ref, "words", DELIM)
        got = ER.errors(hyp, ref, "words", DELIM)
        want = metrics.wer(_text(ref), _text(hyp)) * n_words if n_words else len(_text(hyp).split())
        assert got == round(want), (ref, hyp, got, want)
        assert n_words == len(_text(ref).split())


def test_reference_length():
    assert targets.reference_length([4, 5, 5, 4, 4, 6, 4], "words", 4) == 2
    assert targets.reference_length([4, 5, 5, 4, 4, 6, 4], "labels", 4) == 7
    assert targets.reference_length([], "words", 4) == 0 and targets.reference_length([5], "words", 4) == 1


# ---------------------------------------------------------------------------------------------------------------------
# host tables
# ---------------------------------------------------------------------------------------------------------------------
LANES = 16


def decode_tables(tab, D, V, unit):
    """per reference: (units as symbols, distinct words, longest word) read back from the tables"""
    out = []
    for d in range(D):
        m, peq, dw, nd, maxw = (int(v) for v in tab[8 * d:8 * d + 5])
        assert not np.any(tab[8 * d + 5:8 * d + 8])
        rows = V if unit == "labels" else nd
        masks = tab[peq:peq + rows * LANES].view(np.uint32).reshape(rows, LANES)
        sym = []
        for i in range(m):
            hits = [s for s in range(rows) if masks[s, i // 32] >> (i % 32) & 1]
            assert len(hits) == 1, (d, i, hits)
            sym.append(hits[0])
        assert int(np.unpackbits(masks.view(np.uint8)).sum()) == m          # no bit past the units
        words = [tuple(int(v) for v in tab[tab[dw + 2 * j]:tab[dw + 2 * j] + tab[dw + 2 * j + 1]]) for j in range(nd)]
        out.append((sym, words, maxw, masks))
    return out


def myers_lanes(masks, m, hyp_syms):
    """The device's err_step restated on 32 lanes of uint32 (lanes 16 .. 31 start as the device's do): the carry lookahead
    over ballots, the shift of the horizontal deltas between lanes, and the final popcount."""
    M32 = 0xFFFFFFFF
    vp, vn = [M32] * 32, [0] * 32
    lanes = range(32)
    for s in hyp_syms:
        eq = [int(masks[s, k]) if s >= 0 and k < LANES else 0 for k in lanes]
        x = [eq[k] | vn[k] for k in lanes]
        sm = [((x[k] & vp[k]) + vp[k]) & M32 for k in lanes]
        g = sum(1 << k for k in lanes if sm[k] < vp[k])
        p = sum(1 << k for k in lanes if sm[k] == M32)
        cin = ((g + (g | p)) ^ p) & M32
        d0 = [((((sm[k] + (cin >> k & 1)) & M32) ^ vp[k]) | x[k]) for k in lanes]
        hn = [vp[k] & d0[k] for k in lanes]
        hp = [(vn[k] | ~(vp[k] | d0[k])) & M32 for k in lanes]
        tp = sum(1 << k for k in lanes if hp[k] >> 31)
        tn = sum(1 << k for k in lanes if hn[k] >> 31)
        hps = [((hp[k] << 1) & M32) | ((((tp << 1) | 1) >> k) & 1) for k in lanes]
        hns = [((hn[k] << 1) & M32) | (((tn << 1) >> k) & 1) for k in lanes]
        vn = [hps[k] & d0[k] for k in lanes]
        vp = [(hns[k] | ~(hps[k] | d0[k])) & M32 for k in lanes]
    total = len(hyp_syms)
    for k in lanes:
        lo = 32 * k
        keep = M32 if m >= lo + 32 else ((1 << (m - lo)) - 1 if m > lo else 0)
        total += bin(vp[k] & keep).count("1") - bin(vn[k] & keep).count("1")
    return total


def _hyp_symbols(hyp, unit, words):
    if unit == "labels":
        return list(hyp)
    return [words.index(w) if w in words else -1 for w in ER.split_words(hyp, DELIM)]


@pytest.mark.parametrize("unit", ["labels", "words"])
def test_host_tables_decode_and_drive_the_lane_recurrence_to_the_oracle(unit):
    rng = np.random.default_rng(3 + (unit == "words"))
    V = 33
    for U in (0, 1, 31, 32, 33, 63, 64, 65, 511, 512):
        pool = [4, 5, 6, 7, 8] if unit == "words" else list(range(1, V))
        refs = [[int(v) for v in rng.choice(pool, U)], [5, 4, 5, 6, 4, 4, 6, 5, 4][:min(U, 9)], []]
        tab = error_tables(refs, V, unit)
        for y, (sym, words, maxw, masks) in zip(refs, decode_tables(tab, len(refs), V, unit)):
            if unit == "labels":
                assert sym == y and words == [] and maxw == 0
            else:
                ws = ER.split_words(y, DELIM)
                assert [words[s] for s in sym] == ws and len(set(words)) == len(words)
                assert maxw == max((len(w) for w in ws), default=0)
            for _ in range(3):
                hyp = list(y)
                for _ in range(int(rng.integers(0, 12))):
                    op, i = rng.integers(0, 3), int(rng.integers(0, len(hyp) + 1))
                    if op == 0 and i < len(hyp):
                        del hyp[i]
                    else:
                        hyp.insert(i, int(rng.choice(pool)))
                got = myers_lanes(masks, len(sym), _hyp_symbols(hyp, unit, words))
                assert got == ER.errors(hyp, y, unit, DELIM), (U, len(hyp))


def test_host_tables_refuse_bad_arguments():
    with pytest.raises(ValueError, match="delimiter"):
        error_tables([[5]], 32, "words", blank=0, delimiter=0)


# ---------------------------------------------------------------------------------------------------------------------
# argument checks before any library call
# ---------------------------------------------------------------------------------------------------------------------
class _NoLib:
    def __getattr__(self, name):
        raise AssertionError(f"library called: {name}")


def _engine_without_device():
    eng = Engine.__new__(Engine)
    eng.lib = _NoLib()
    eng._h = None
    eng.config = dataclasses.replace(VARIANTS["tiny_group"])
    return eng


@pytest.mark.parametrize("refs,kw,match", [
    ([[5, 32]], {}, "vocabulary"),                               # label >= V
    ([[5, -1]], {}, "vocabulary"),
    ([[5, 0, 6]], {}, "blank"),                                  # label == blank
    ([[5, 6]], dict(blank=32), "blank 32"),                      # blank out of range
    ([[5, 6]], dict(blank=-1), "blank -1"),
    ([list(range(1, 31)) * 18], {}, "at most 512"),              # U > cap
    ([], {}, "D >= 1"),                                          # D = 0
    ([[5]], dict(unit="chars"), "unit"),
    ([[5]], dict(delimiter=32), "delimiter 32"),                 # delimiter out of range (words)
    ([[5]], dict(delimiter=-2), "delimiter -2"),
    ([[5]], dict(delimiter=0), "equal to the blank"),            # delimiter == blank
    ([[5]], dict(delimiter=7, blank=7), "equal to the blank 7"),
])
def test_set_references_validation_raises_before_any_library_call(refs, kw, match):
    eng = _engine_without_device()
    with pytest.raises(ValueError, match=match):
        eng.set_references(refs, **kw)


def test_labels_unit_ignores_the_delimiter():
    from shap_transformer_asr_b200.engine import reference_arrays
    labels, offsets = reference_arrays([[5, 4]], "labels", delimiter=0, vocab_size=32)
    assert labels.tolist() == [5, 4] and offsets.tolist() == [0, 2]


def test_explain_errors_mode_on_a_mock_engine():
    """explain(mode="errors"): the default reference is the greedy transcription of the one-row logits pass, the result
    carries it with its word count, and explicit targets are used as given."""
    from test_kernelshap import _MockEngine
    from shap_transformer_asr_b200.kernelshap import KernelShapExplainer

    class Eng(_MockEngine):
        def set_references(self, refs, unit="words", blank=0, delimiter=4):
            self.references = [np.asarray(t, dtype=np.int32) for t in refs]
            self.mode = "errors"
            self.calls.append(f"set_references:{len(refs)}:{unit}:{delimiter}")

    M = 8
    eng = Eng(M, 1)
    eng.logit_table[:] = 0.0
    eng.logit_table[np.arange(6), [5, 4, 6, 6, 0, 7]] = 1.0
    res = KernelShapExplainer(eng, nsamples=100, seed=0).explain(np.zeros(1000, np.float32), num_segments=M, mode="errors")
    assert [r.tolist() for r in res["references"]] == [[5, 4, 6, 7]] and res["reference_lengths"] == [2]
    assert "eval:logits:1" in eng.calls and "set_references:1:words:4" in eng.calls
    eng = Eng(M, 2)
    res = KernelShapExplainer(eng, nsamples=100, seed=0).explain(np.zeros(1000, np.float32), num_segments=M, mode="errors",
                                                               targets=[[5, 6], [7, 4, 7]], unit="labels")
    assert res["reference_lengths"] == [2, 3] and "eval:logits:1" not in eng.calls
