"""CPU: WavLMForCTC support without a GPU -- the library's relative-position buckets against transformers, the WavLM
oracle against the live transformers model and the committed golden vectors, and the oracle's sensitivity to the bias
(a test that cannot fail pins nothing)."""
import os

import numpy as np
import pytest
import torch

import __graft_entry__ as entry
from oracle import wavlm_forward as WL
from oracle.make_golden_wavlm import VARIANTS as WAVLM_VARIANTS, build
from shap_transformer_asr_b200 import _lib, relative_buckets
from shap_transformer_asr_b200.config import MODELS, WORKLOADS, ModelConfig
from helpers import weight_checksum

LOGIT_TOL = 0.025   # the GPU parity tolerance (max |gpu - ref| / max |ref|)


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        entry.build()
    return _lib.load()


def hf_buckets(d_max, num_buckets=320, max_distance=800):
    from transformers.models.wavlm.modeling_wavlm import WavLMAttention
    att = WavLMAttention(128, 2, num_buckets=num_buckets, max_distance=max_distance)
    return att._relative_positions_bucket(torch.arange(-d_max, d_max + 1)).numpy()


def test_relative_buckets_match_transformers_for_every_clip_length(lib):
    """T' = 1 .. 2048: |d| up to 2047 covers d = +-713 (where the log lands at 75.99996) and the clamp from |d| = 778."""
    ref = hf_buckets(2047)
    for T in range(1, 2049):
        got = relative_buckets(T)
        assert np.array_equal(got, ref[2047 - (T - 1):2047 + T]), T
    # d = 713: 80 + 80 log(713 / 80) / log(10) = 155.99996, truncated to 155 -- a float32 rounding up would give 156
    assert ref[2047 + 713] == 160 + 155 and ref[2047 - 713] == 155
    assert ref[2047 + 778] == ref[2047 + 2047] == 319 and ref[2047 - 778] == ref[0] == 159
    # the oracle's restatement of the bucket function, too
    assert np.array_equal(WL.relative_positions_bucket(torch.arange(-2047, 2048), 320, 800).numpy(), ref)


def test_relative_buckets_other_parameters_and_bad_arguments(lib):
    ref = hf_buckets(300, num_buckets=64, max_distance=128)
    assert np.array_equal(relative_buckets(301, 64, 128), ref)
    for bad in [(0, 320, 800), (5, 2, 800), (5, 320, 80)]:
        with pytest.raises(ValueError):
            relative_buckets(*bad)


def test_config_knows_wavlm():
    import transformers
    c = ModelConfig.from_hf(transformers.WavLMConfig())
    assert c == MODELS["wavlm-base-plus"] and c.kind == "wavlm"
    large = MODELS["wavlm-large"]
    assert (large.hidden_size, large.num_hidden_layers, large.num_attention_heads, large.intermediate_size) == (1024, 24, 16, 4096)
    assert large.feat_extract_norm == "layer" and large.conv_bias and large.do_stable_layer_norm
    c6, c2 = WORKLOADS["C6"], WORKLOADS["C2"]
    assert c6.model == "wavlm-base-plus"
    assert (c6.num_samples, c6.num_segments, c6.num_coalitions) == (c2.num_samples, c2.num_segments, c2.num_coalitions)
    assert _lib.W2SConfig._fields_[-2:] == [("num_buckets", _lib.C.c_int32), ("max_bucket_distance", _lib.C.c_int32)]


@pytest.mark.parametrize("name", list(WAVLM_VARIANTS))
@pytest.mark.parametrize("L", [4000, 288080])   # the golden length (T' = 12) and T' = 900, past the bucket clamp
def test_wavlm_oracle_matches_transformers_live(name, L):
    cfg = WAVLM_VARIANTS[name]
    model = build(cfg)
    x = torch.randn(2, L, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        ref = model(x).logits
        out = WL.ctc_logits(WL.state_dict_of(model), cfg.to_dict(), x)
    assert ref.shape == out.shape and (L < 10000 or ref.shape[1] == 900)
    assert (ref - out).abs().max().item() <= 2e-4


def golden_case(name, golden_dir):
    g = np.load(os.path.join(golden_dir, f"{name}.npz"))
    cfg = WAVLM_VARIANTS[name]
    model = build(cfg)
    assert abs(weight_checksum(model) - float(g["checksum"])) <= 1e-6 * float(g["checksum"]), "weight RNG drift"
    return g, cfg, WL.state_dict_of(model)


@pytest.mark.parametrize("name", list(WAVLM_VARIANTS))
def test_wavlm_oracle_matches_golden(name, golden_dir):
    g, cfg, sd = golden_case(name, golden_dir)
    with torch.no_grad():
        out = WL.ctc_logits(sd, cfg.to_dict(), torch.from_numpy(g["x"])).numpy()
    assert np.abs(out - g["logits"]).max() <= 2e-4


@pytest.mark.parametrize("name", list(WAVLM_VARIANTS))
@pytest.mark.parametrize("mutation", ["no_bias", "shift_by_one"])
def test_wrong_bias_misses_the_golden_by_far(name, mutation, golden_dir, monkeypatch):
    """Dropping the bias or shifting the relative position by one moves the logits by more than 10x the GPU tolerance,
    so a model-level test catches either mistake in the CUDA path."""
    g, cfg, sd = golden_case(name, golden_dir)
    right = WL.position_bias

    def wrong(sd_, cfg_, T, dtype):
        if mutation == "no_bias":
            return torch.zeros_like(right(sd_, cfg_, T, dtype))
        pos = torch.arange(T)
        b = WL.relative_positions_bucket(pos[None, :] - pos[:, None] + 1, cfg_["num_buckets"], cfg_["max_bucket_distance"])
        return sd_[WL.PREFIX + "encoder.layers.0.attention.rel_attn_embed.weight"].to(dtype)[b].permute(2, 0, 1)

    monkeypatch.setattr(WL, "position_bias", wrong)
    with torch.no_grad():
        out = WL.ctc_logits(sd, cfg.to_dict(), torch.from_numpy(g["x"])).numpy()
    assert np.abs(out - g["logits"]).max() > 10 * LOGIT_TOL * np.abs(g["logits"]).max()
