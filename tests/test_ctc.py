"""CPU: the transcript-level output (log p_CTC of a label sequence) -- the oracle against the HF loss, the greedy
transcript and the host-side argument checks, which raise before the library is called."""
import dataclasses

import numpy as np
import pytest
import torch

from helpers import VARIANTS, build_model
from oracle import ctc_ref
from oracle import w2v2_forward as W
from shap_transformer_asr_b200 import metrics, targets
from shap_transformer_asr_b200.engine import Engine


def _hf_loss(model, x, y):
    model.config.ctc_loss_reduction = "sum"
    model.config.ctc_zero_infinity = False
    with torch.no_grad():
        return float(model(torch.from_numpy(x)[None], labels=torch.as_tensor(y, dtype=torch.long)[None]).loss)


@pytest.mark.parametrize("variant", ["tiny_group", "tiny_layer_stable", "tiny_conformer_rel", "tiny_conformer_rotary"])
def test_oracle_transcript_mode_equals_the_hf_ctc_loss(variant):
    cfg = VARIANTS[variant]
    model = build_model(cfg)
    sd, d = W.state_dict_of(model), cfg.to_dict()
    x = np.random.default_rng(1).standard_normal(8000).astype(np.float32)
    T = cfg.num_frames(8000)
    ys = [[5, 6, 6, 7], [9], list(np.random.default_rng(2).integers(1, cfg.vocab_size, T // 2))]
    got = ctc_ref.evaluate(sd, d, x[None], transcripts=ys, blank=0)[0]
    for j, y in enumerate(ys):
        ref = -_hf_loss(model, x, y)
        assert abs(got[j] - ref) <= 2e-6 * max(1.0, abs(ref)), (j, got[j], ref)


def test_oracle_transcript_mode_equals_the_hf_ctc_loss_wavlm():
    from oracle.make_golden_wavlm import VARIANTS as WV, build as build_wavlm
    cfg = WV["tiny_wavlm"]
    model = build_wavlm(cfg)
    x = np.random.default_rng(3).standard_normal(6000).astype(np.float32)
    y = [5, 8, 8, 2]
    with torch.no_grad():
        logits = model(torch.from_numpy(x)[None]).logits
    got = ctc_ref.reduce_logits(logits, "transcript", transcripts=[y], blank=0)[0, 0].item()
    ref = -_hf_loss(model, x, y)
    assert abs(got - ref) <= 2e-6 * max(1.0, abs(ref))


def test_empty_transcript_is_the_all_blank_path():
    z = torch.randn(2, 17, 32, dtype=torch.float64)
    got = ctc_ref.ctc_logp(z, [[]], blank=3)[:, 0]
    want = torch.log_softmax(z, -1)[:, :, 3].sum(1)
    assert torch.allclose(got, want, rtol=0, atol=1e-12)


def test_greedy_transcript_collapse_and_blank_rules():
    V = 32
    ids = [0, 5, 5, 0, 5, 6, 6, 6, 0, 0, 4, 7, 0]
    logits = np.full((len(ids), V), -1.0)
    logits[np.arange(len(ids)), ids] = 1.0
    assert targets.greedy_transcript(logits).tolist() == [5, 5, 6, 4, 7]
    # another blank id: 0 is then a label
    assert targets.greedy_transcript(logits, blank=6).tolist() == [0, 5, 0, 5, 0, 4, 7, 0]
    # all blank: the empty transcript
    assert targets.greedy_transcript(np.eye(V)[[0, 0, 0]]).size == 0
    # the string form agrees with greedy_ctc_decode on the same argmax sequence
    rng = np.random.default_rng(0)
    for _ in range(20):
        lg = rng.standard_normal((50, V)) + 3.0 * (rng.random((50, 1)) < 0.5) * np.eye(V)[np.zeros(50, int)]
        y = targets.greedy_transcript(lg)
        s = " ".join("".join(" " if t == 4 else metrics.VOCAB[t] for t in y).split())
        assert s == metrics.greedy_ctc_decode(lg.argmax(-1))


def test_frames_needed_counts_repeats():
    assert targets.frames_needed([]) == 0
    assert targets.frames_needed([3, 3, 3]) == 5
    assert targets.frames_needed([3, 4, 3]) == 3


class _NoLib:
    """Stands in for the ctypes library: any call means the host checks let a bad argument through."""

    def __getattr__(self, name):
        raise AssertionError(f"library called: {name}")


def _engine_without_device():
    eng = Engine.__new__(Engine)
    eng.lib = _NoLib()
    eng._h = None
    eng.config = dataclasses.replace(VARIANTS["tiny_group"])
    return eng


@pytest.mark.parametrize("transcripts,blank,offsets,match", [
    ([[5, 32]], 0, None, "vocabulary"),                        # label >= V
    ([[5, 0, 6]], 0, None, "blank"),                           # label == blank
    ([[5, 6]], 32, None, "blank 32"),                          # blank out of range
    ([[5, 6]], -1, None, "blank -1"),
    ([list(range(1, 31)) * 18], 0, None, "at most 512"),       # U > cap
    ([], 0, None, "D >= 1"),                                   # D = 0
    ([5, 6, 7], 0, [0, 2], "label count"),                     # offsets that do not cover the labels
    ([5, 6, 7], 0, [0, 2, 1, 3], "non-decreasing"),               # non-ascending offsets
    ([5, 6, 7], 0, [1, 3], "start at 0"),
    ([5, 6, 7], 0, [0], "D >= 1"),
])
def test_host_validation_raises_before_any_library_call(transcripts, blank, offsets, match):
    eng = _engine_without_device()
    with pytest.raises(ValueError, match=match):
        eng.set_transcripts(transcripts, blank=blank, offsets=offsets)


def test_transcript_arrays_pack_in_order():
    labels, offsets = targets.transcript_arrays([[1, 2], [], [3]], vocab_size=32)
    assert labels.tolist() == [1, 2, 3] and offsets.tolist() == [0, 2, 2, 3]
    labels, offsets = targets.transcript_arrays([7, 7], vocab_size=32)    # one sequence of ints is one transcript
    assert labels.tolist() == [7, 7] and offsets.tolist() == [0, 2]


def test_explain_transcript_mode_on_a_mock_engine():
    """explain(mode="transcript"): the default transcript is the greedy transcription of the one-row logits pass, the
    result carries it, and a greedy transcript longer than the cap is refused with a ValueError naming it."""
    from test_kernelshap import _MockEngine
    from shap_transformer_asr_b200.kernelshap import KernelShapExplainer

    class Eng(_MockEngine):
        def set_transcripts(self, transcripts, blank=0):
            self.transcripts = [np.asarray(t, dtype=np.int32) for t in transcripts]
            self.mode = "transcript"
            self.calls.append(f"set_transcripts:{len(transcripts)}")

    M = 8
    eng = Eng(M, 1)
    res = KernelShapExplainer(eng, nsamples=100, seed=0).explain(np.zeros(1000, np.float32), num_segments=M,
                                                               mode="transcript")
    want = targets.greedy_transcript(eng.logit_table)
    assert len(res["transcripts"]) == 1 and np.array_equal(res["transcripts"][0], want)
    assert "eval:logits:1" in eng.calls and "set_transcripts:1" in eng.calls
    assert np.abs(res["phi"].numpy() - eng.W).max() < 1e-5
    eng = Eng(M, 1, frames=2 * targets.MAX_TRANSCRIPT + 2)
    eng.logit_table[:] = -1.0
    eng.logit_table[np.arange(eng.logit_table.shape[0]), 1 + np.arange(eng.logit_table.shape[0]) % 2] = 1.0
    with pytest.raises(ValueError, match="1026 labels"):
        KernelShapExplainer(eng, nsamples=100, seed=0).explain(np.zeros(1000, np.float32), num_segments=M,
                                                               mode="transcript")
