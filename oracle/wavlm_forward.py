"""ORACLE (test infrastructure, never shipped or measured as the product).

CPU restatement of the WavLMForCTC eval-mode forward (HF = site-packages/transformers/models/,
wavlm/modeling_wavlm.py of the installed 5.5.0), in fp32 (or fp64 with ``dtype=torch.float64``).  Everything but
the attention is wav2vec2's (feature encoder, feature projection, positional conv, post-LN / stable-LN layers, FFN,
head), so those pieces are taken from ``w2v2_forward``; the new operation is the gated relative-position bias of
every attention layer.

Pinning: tests/test_wavlm_oracle.py checks this file against the installed ``transformers`` WavLMForCTC with
shared random-init weights and against tests/golden/tiny_wavlm*.npz, which ``oracle/make_golden_wavlm.py``
generated from ``transformers`` itself.
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F

from . import w2v2_forward as W

PREFIX = "wavlm."


def relative_positions_bucket(rel: torch.Tensor, num_buckets: int, max_distance: int) -> torch.Tensor:
    """HF modeling_wavlm.py:253-271 (_relative_positions_bucket), restated on an int64 tensor of j - i."""
    nb = num_buckets // 2                                                            # :254
    buckets = (rel > 0).to(torch.long) * nb                                         # :256
    a = rel.abs()                                                                   # :257
    max_exact = nb // 2                                                             # :259
    is_small = a < max_exact                                                        # :260
    large = torch.log(a.float() / max_exact) / math.log(max_distance / max_exact) * (nb - max_exact)  # :262-264
    large = (max_exact + large).to(torch.long)                                      # :265
    large = torch.clamp(large, max=nb - 1)                                          # :266-268
    return buckets + torch.where(is_small, a, large)                                # :270


def position_bias(sd, cfg, T: int, dtype) -> torch.Tensor:
    """HF :243-251 (compute_bias) of layer 0, the only layer with rel_attn_embed: [heads, T, T], E[bucket(j - i), h].
    HF passes this ungated bias from layer 0 down the whole stack (:410-430)."""
    pos = torch.arange(T)
    bucket = relative_positions_bucket(pos[None, :] - pos[:, None], cfg["num_buckets"], cfg["max_bucket_distance"])
    E = sd[PREFIX + "encoder.layers.0.attention.rel_attn_embed.weight"].to(dtype)   # [num_buckets, heads]
    return E[bucket].permute(2, 0, 1)


def _wavlm_attention(sd, p, h, n_heads, bias):
    """HF :147-186 + torch_multi_head_self_attention :188-241 (no mask, eval mode): scores scaled by d^-0.5, then the
    gated bias added (F.multi_head_attention_forward adds attn_mask after scaling)."""
    B, T, H = h.shape
    d = H // n_heads
    q = F.linear(h, sd[p + "q_proj.weight"], sd[p + "q_proj.bias"]).view(B, T, n_heads, d).transpose(1, 2)
    k = F.linear(h, sd[p + "k_proj.weight"], sd[p + "k_proj.bias"]).view(B, T, n_heads, d).transpose(1, 2)
    v = F.linear(h, sd[p + "v_proj.weight"], sd[p + "v_proj.bias"]).view(B, T, n_heads, d).transpose(1, 2)
    # gate (:166-176): the attention input per head through gru_rel_pos_linear [8, d], 8 outputs summed in two groups of 4
    x = h.view(B, T, n_heads, d).permute(0, 2, 1, 3)
    proj = F.linear(x, sd[p + "gru_rel_pos_linear.weight"], sd[p + "gru_rel_pos_linear.bias"]).view(B, n_heads, T, 2, 4).sum(-1)
    ga, gb = torch.sigmoid(proj).chunk(2, dim=-1)
    gate = ga * (gb * sd[p + "gru_rel_pos_const"].view(1, n_heads, 1, 1) - 1.0) + 2.0          # [B, heads, T, 1]
    s = torch.matmul(q, k.transpose(2, 3)) * (d ** -0.5) + gate * bias[None]                    # :179
    a = torch.softmax(s, dim=-1)
    o = torch.matmul(a, v).transpose(1, 2).reshape(B, T, H)
    return F.linear(o, sd[p + "out_proj.weight"], sd[p + "out_proj.bias"])


def encoder_wavlm(sd, cfg, h, prefix=PREFIX):
    """HF :376-447 (post-LN, layer :298-336) / :450-522 (stable-LN, layer :339-373)."""
    eps = cfg["layer_norm_eps"]
    act = W._act(cfg["hidden_act"])
    e = prefix + "encoder."
    bias = position_bias(sd, cfg, h.shape[1], h.dtype)
    h = h + W.pos_conv_embed(sd, cfg, h, prefix)
    if not cfg["do_stable_layer_norm"]:
        h = W._ln(sd, e + "layer_norm.", h, eps)
    nh = cfg["num_attention_heads"]
    for i in range(cfg["num_hidden_layers"]):
        p = f"{e}layers.{i}."
        if cfg["do_stable_layer_norm"]:
            h = h + _wavlm_attention(sd, p + "attention.", W._ln(sd, p + "layer_norm.", h, eps), nh, bias)
            h = h + W._ffn(sd, p + "feed_forward.", W._ln(sd, p + "final_layer_norm.", h, eps), act)
        else:
            h = W._ln(sd, p + "layer_norm.", h + _wavlm_attention(sd, p + "attention.", h, nh, bias), eps)
            h = W._ln(sd, p + "final_layer_norm.", h + W._ffn(sd, p + "feed_forward.", h, act), eps)
    if cfg["do_stable_layer_norm"]:
        h = W._ln(sd, e + "layer_norm.", h, eps)
    return h


def ctc_logits(sd: Dict[str, torch.Tensor], cfg: dict, x: torch.Tensor) -> torch.Tensor:
    """waveform [B, L] -> logits [B, T', vocab] (HF :1176-1215 ForCTC -> :1039-1103 Model -> lm_head :1209); other model
    kinds go to w2v2_forward.ctc_logits."""
    if cfg.get("kind") != "wavlm":
        return W.ctc_logits(sd, cfg, x)
    dtype = x.dtype
    sd = {k: v.to(dtype) if v.is_floating_point() else v for k, v in sd.items()}
    feats = W.feature_encoder(sd, cfg, x, PREFIX).transpose(1, 2)
    h = W.feature_projection(sd, cfg, feats, PREFIX)
    h = encoder_wavlm(sd, cfg, h)
    return F.linear(h, sd["lm_head.weight"], sd["lm_head.bias"])


def build_hf_model(cfg: dict, seed: int = 0):
    """Random-init transformers WavLMForCTC of the given architecture, eval mode."""
    import transformers

    torch.manual_seed(seed)
    hf_cfg = transformers.WavLMConfig(
        conv_dim=list(cfg["conv_dim"]), conv_kernel=list(cfg["conv_kernel"]), conv_stride=list(cfg["conv_stride"]),
        conv_bias=cfg["conv_bias"], feat_extract_norm=cfg["feat_extract_norm"], hidden_size=cfg["hidden_size"],
        num_hidden_layers=cfg["num_hidden_layers"], num_attention_heads=cfg["num_attention_heads"],
        intermediate_size=cfg["intermediate_size"], num_conv_pos_embeddings=cfg["num_conv_pos_embeddings"],
        num_conv_pos_embedding_groups=cfg["num_conv_pos_embedding_groups"], vocab_size=cfg["vocab_size"],
        layer_norm_eps=cfg["layer_norm_eps"], hidden_act=cfg["hidden_act"], num_feat_extract_layers=len(cfg["conv_dim"]),
        do_stable_layer_norm=cfg["do_stable_layer_norm"], num_buckets=cfg["num_buckets"],
        max_bucket_distance=cfg["max_bucket_distance"])
    return transformers.WavLMForCTC(hf_cfg).eval()


def randomize_affine(model, seed: int = 1):
    """w2v2_forward.randomize_affine (LayerNorm / GroupNorm affine terms), then gru_rel_pos_const, which random init
    leaves at 1, from a generator of its own (rel_attn_embed is already N(0, 1), so the bias is not negligible).
    v_proj and out_proj are scaled by 4: with the 0.02-std init the attention branch adds a few percent to the residual
    stream and a wrong bias would move the logits by little more than the GPU tolerance; scaled, dropping the bias or
    shifting it by one position moves them by 25-55 % of their maximum."""
    W.randomize_affine(model, seed)
    g = torch.Generator().manual_seed(seed + 1000)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith("gru_rel_pos_const"):
                p.add_(0.25 * torch.randn(p.shape, generator=g))
            elif name.endswith("attention.v_proj.weight") or name.endswith("attention.out_proj.weight"):
                p.mul_(4.0)
    return model


def state_dict_of(model) -> Dict[str, torch.Tensor]:
    """Detached fp32 state dict with the pos-conv weight_norm folded into a plain ``weight``."""
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    if PREFIX + "encoder.pos_conv_embed.conv.parametrizations.weight.original0" in sd:
        sd[PREFIX + "encoder.pos_conv_embed.conv.weight"] = W.pos_conv_weight(sd, PREFIX)
    return sd
