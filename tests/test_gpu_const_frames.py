"""The feature encoder's constant-frame skip against the dense front end (W2S_FLAG_DENSE_FRONTEND): raw logits of every
frame and vocabulary entry must be bit-identical, whichever blocks the skip leaves out."""
import numpy as np
import pytest
import torch

from shap_transformer_asr_b200 import MODELS, Engine, KernelShapExplainer, synthetic_clip
from shap_transformer_asr_b200 import preprocess as P
from shap_transformer_asr_b200.modelzoo import build_random_init_model

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engines():
    cfg = MODELS["wav2vec2-base"]
    model = build_random_init_model(cfg, seed=0)
    # max_batch 40: on a 5 s clip every conv layer of a full tile runs the list contraction (conv6: 2 x 2 x 40 = 160 tiles
    # >= 148 SMs); the ragged last tile of 13 coalitions runs conv6 on the single-CTA kernel, dense
    pair = {d: Engine(model, cfg, max_batch=40, dense_frontend=d) for d in (False, True)}
    yield cfg, model, pair
    for e in pair.values():
        e.close()


def both(pair, clip, Z, bounds=None, num_segments=None, baseline=0.0, mode="logits"):
    outs = []
    for d in (False, True):
        e = pair[d]
        e.set_clip(clip, num_segments=num_segments or (len(bounds) - 1), bounds=bounds, baseline=baseline)
        e.set_targets(mode)
        outs.append(e.eval_bits(e.bits_to_device(np.asarray(Z, np.uint8))).cpu().numpy())
    return outs


def coalitions(M):
    Z = [np.zeros(M), np.ones(M)]
    for at in (0, M // 2, M - 1):
        z = np.zeros(M)
        z[at] = 1
        Z.append(z)
    Z.append(np.arange(M) % 2)
    Z.append(1 - np.arange(M) % 2)
    rng = np.random.default_rng(0)
    Z += list(rng.integers(0, 2, (45, M)))
    return np.asarray(Z, np.uint8)


@pytest.mark.parametrize("L,M", [(80000, 100), (16000, 20)])
def test_skip_matches_dense(engines, L, M):
    _, _, pair = engines
    clip = synthetic_clip(L)
    a, b = both(pair, clip, coalitions(M), num_segments=M)
    assert np.isfinite(a).all()
    assert np.array_equal(a, b)


def test_short_segments_and_baseline(engines):
    _, _, pair = engines
    L = 48000
    rng = np.random.default_rng(5)
    cuts = np.sort(rng.integers(0, L, 63))   # many segments shorter than the 400-sample receptive field
    bounds = np.concatenate([[0], cuts, [L]]).astype(np.int32)
    clip = synthetic_clip(L)
    for base in (0.0, 0.37):
        a, b = both(pair, clip, coalitions(64), bounds=bounds, baseline=base)
        assert np.array_equal(a, b)


def test_explain_matches_dense(engines):
    _, _, pair = engines
    clip = synthetic_clip(32000)
    res = [KernelShapExplainer(pair[d], nsamples=256, seed=0).explain(clip, num_segments=40) for d in (False, True)]
    assert torch.equal(res[0]["y"], res[1]["y"])
    assert torch.equal(res[0]["phi"], res[1]["phi"])


def test_background_unchanged(engines):
    _, _, pair = engines
    L, M = 32000, 16
    clip = synthetic_clip(L)
    bg = np.stack([synthetic_clip(L, seed=s) for s in (3, 4)])
    Z = coalitions(M)
    outs = []
    for d in (False, True):
        e = pair[d]
        e.set_clip(clip, num_segments=M)
        e.set_targets("logits")
        e.set_background(bg)
        outs.append(e.eval_bits(e.bits_to_device(Z)).cpu().numpy())
        e.clear_background()
    assert np.array_equal(outs[0], outs[1])


def test_skip_is_engaged(engines):
    """The skip arm contracts fewer conv1 blocks than the dense arm, and fills blocks up to conv6."""
    _, _, pair = engines
    clip = synthetic_clip(80000)
    Z = coalitions(100)[:40]          # one full tile, the all-dropped coalition included
    prof = {}
    for d in (False, True):
        e = pair[d]
        e.set_clip(clip, num_segments=100)
        e.set_targets("logits")
        bits = e.bits_to_device(Z)
        e.eval_bits(bits)
        torch.cuda.synchronize()
        e.profile(True)
        e.eval_bits(bits)
        torch.cuda.synchronize()
        prof[d] = e.profile_read()
        e.profile(False)
    skip, dense = prof[False], prof[True]
    assert "frontend_lists" in skip and "frontend_lists" not in dense
    assert 0 < skip["conv1"]["flops"] < 0.9 * dense["conv1"]["flops"]
    for l in range(1, 7):
        assert f"conv{l}_fill" in skip
    assert skip["conv6_fill"]["bytes"] > 0     # the all-dropped coalition: one conv6 block contracted, one filled


def test_table_survives_a_workspace_rebuild(engines):
    """eval_waveforms at another length rebuilds the workspace; the next coalition evaluation rebuilds it for the clip
    and must find the clip's block table again."""
    _, _, pair = engines
    L, M = 48000, 30
    clip = synthetic_clip(L)
    Z = coalitions(M)
    outs = []
    for d in (False, True):
        e = pair[d]
        e.set_clip(clip, num_segments=M)
        e.set_targets("logits")
        e.eval_waveforms(torch.as_tensor(synthetic_clip(9000), device="cuda")[None].contiguous())
        e.set_targets("logits")
        outs.append(e.eval_bits(e.bits_to_device(Z)).cpu().numpy())
    assert np.array_equal(outs[0], outs[1])


def test_band_cells_unchanged(engines):
    _, _, pair = engines
    L, M, F = 32000, 16, 4
    clip = synthetic_clip(L)
    comp = P.band_components(clip, P.mel_band_edges(F))
    rng = np.random.default_rng(7)
    Z = np.concatenate([np.zeros((1, M * F)), np.ones((1, M * F)), rng.integers(0, 2, (30, M * F))]).astype(np.uint8)
    outs = []
    for d in (False, True):
        e = pair[d]
        e.set_clip(clip, num_segments=M)
        e.set_targets("logits")
        e.set_bands(comp)
        outs.append(e.eval_bits(e.bits_to_device(Z)).cpu().numpy())
        e.clear_bands()
    assert np.array_equal(outs[0], outs[1])
