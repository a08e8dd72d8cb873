"""Random-init models of the named architectures (synthetic weights for benchmarks and sweeps).

The reference loads hub checkpoints (shap_calculation.py:218-219); the hub is unreachable here, so benchmarks
use config-constructed `transformers` models with a fixed seed, put in eval mode (a config-constructed model
starts in train mode: dropout / LayerDrop / SpecAugment would fire otherwise, SURVEY.md 3.2), with the affine
terms that random init leaves at (1, 0) perturbed so that every term of the forward is exercised.
"""
from __future__ import annotations

import torch

from .config import ModelConfig


def build_random_init_model(cfg: ModelConfig, seed: int = 0, perturb_affine: bool = True):
    import transformers

    torch.manual_seed(seed)
    common = dict(
        conv_dim=list(cfg.conv_dim), conv_kernel=list(cfg.conv_kernel), conv_stride=list(cfg.conv_stride),
        conv_bias=cfg.conv_bias, feat_extract_norm=cfg.feat_extract_norm, hidden_size=cfg.hidden_size,
        num_hidden_layers=cfg.num_hidden_layers, num_attention_heads=cfg.num_attention_heads,
        intermediate_size=cfg.intermediate_size, num_conv_pos_embeddings=cfg.num_conv_pos_embeddings,
        num_conv_pos_embedding_groups=cfg.num_conv_pos_embedding_groups, vocab_size=cfg.vocab_size,
        layer_norm_eps=cfg.layer_norm_eps, hidden_act=cfg.hidden_act, num_feat_extract_layers=len(cfg.conv_dim))
    if cfg.kind == "conformer":
        hf_cfg = transformers.Wav2Vec2ConformerConfig(
            position_embeddings_type=cfg.position_embeddings_type,
            conv_depthwise_kernel_size=cfg.conv_depthwise_kernel_size, rotary_embedding_base=cfg.rotary_embedding_base,
            max_source_positions=cfg.max_source_positions, **common)
        model = transformers.Wav2Vec2ConformerForCTC(hf_cfg)
    elif cfg.kind == "wavlm":
        hf_cfg = transformers.WavLMConfig(do_stable_layer_norm=cfg.do_stable_layer_norm, num_buckets=cfg.num_buckets,
                                          max_bucket_distance=cfg.max_bucket_distance, **common)
        model = transformers.WavLMForCTC(hf_cfg)
    else:
        hf_cfg = transformers.Wav2Vec2Config(do_stable_layer_norm=cfg.do_stable_layer_norm, **common)
        model = transformers.Wav2Vec2ForCTC(hf_cfg)
    model = model.eval()
    if perturb_affine:
        g = torch.Generator().manual_seed(seed + 1)
        with torch.no_grad():
            for name, p in model.named_parameters():
                if name.endswith("layer_norm.weight") or name.endswith("batch_norm.weight"):
                    p.add_(0.1 * torch.randn(p.shape, generator=g))
                elif name.endswith("layer_norm.bias") or name.endswith("batch_norm.bias"):
                    p.add_(0.05 * torch.randn(p.shape, generator=g))
                elif name.endswith("pos_bias_u") or name.endswith("pos_bias_v"):
                    p.add_(0.05 * torch.randn(p.shape, generator=g))
                elif name.endswith("gru_rel_pos_const"):   # WavLM: random init leaves it at 1
                    p.add_(0.25 * torch.randn(p.shape, generator=g))
            for name, b in model.named_buffers():
                if name.endswith("running_mean"):
                    b.add_(0.05 * torch.randn(b.shape, generator=g))
                elif name.endswith("running_var"):
                    b.mul_(1.0 + 0.2 * torch.rand(b.shape, generator=g))
    return model
