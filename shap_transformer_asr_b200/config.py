"""Architecture and workload definitions for the masked-coalition evaluation path.

The reference never stores an architecture itself: it pulls
``facebook/wav2vec2-base-960h`` (shap_calculation.py:20) and
``facebook/wav2vec2-conformer-rel-pos-large-960h-ft``
(feasability_tests/w2v2conformer.py:57) from the hub.  The hub is unreachable
here, so the hyper-parameters below ARE the definition of the named
architectures for this repo (SURVEY.md section 8c).  Field names follow
``transformers.Wav2Vec2Config`` / ``Wav2Vec2ConformerConfig`` / ``WavLMConfig`` so a
config object of any of them can be converted with :func:`ModelConfig.from_hf`.
"""
from __future__ import annotations

from dataclasses import dataclass, field, asdict
from typing import Tuple


@dataclass(frozen=True)
class ModelConfig:
    kind: str = "wav2vec2"                      # "wav2vec2" | "conformer" | "wavlm"
    conv_dim: Tuple[int, ...] = (512,) * 7
    conv_kernel: Tuple[int, ...] = (10, 3, 3, 3, 3, 2, 2)
    conv_stride: Tuple[int, ...] = (5, 2, 2, 2, 2, 2, 2)
    conv_bias: bool = False
    feat_extract_norm: str = "group"            # "group" | "layer"
    hidden_size: int = 768
    num_hidden_layers: int = 12
    num_attention_heads: int = 12
    intermediate_size: int = 3072
    num_conv_pos_embeddings: int = 128
    num_conv_pos_embedding_groups: int = 16
    vocab_size: int = 32
    layer_norm_eps: float = 1e-5
    do_stable_layer_norm: bool = False
    # conformer only
    position_embeddings_type: str = "relative"  # "relative" | "rotary"
    conv_depthwise_kernel_size: int = 31
    hidden_act: str = "gelu"                    # conformer hub checkpoints use "swish"
    rotary_embedding_base: int = 10000
    max_source_positions: int = 5000
    # WavLM only: gated relative-position bias buckets
    num_buckets: int = 320
    max_bucket_distance: int = 800

    @property
    def head_dim(self) -> int:
        return self.hidden_size // self.num_attention_heads

    def num_frames(self, num_samples: int) -> int:
        """L -> T' (HF modeling_wav2vec2.py:1005-1024: floor((n-k)/s)+1 per layer)."""
        n = int(num_samples)
        for k, s in zip(self.conv_kernel, self.conv_stride):
            n = (n - k) // s + 1
        return n

    def conv_lengths(self, num_samples: int):
        n = int(num_samples)
        out = []
        for k, s in zip(self.conv_kernel, self.conv_stride):
            n = (n - k) // s + 1
            out.append(n)
        return out

    def to_dict(self):
        return asdict(self)

    @staticmethod
    def from_hf(cfg) -> "ModelConfig":
        """Build from a transformers Wav2Vec2Config / Wav2Vec2ConformerConfig / WavLMConfig (duck-typed)."""
        name = type(cfg).__name__
        kind = "conformer" if "Conformer" in name else "wavlm" if "WavLM" in name else "wav2vec2"
        kw = dict(
            kind=kind,
            conv_dim=tuple(cfg.conv_dim), conv_kernel=tuple(cfg.conv_kernel),
            conv_stride=tuple(cfg.conv_stride), conv_bias=bool(cfg.conv_bias),
            feat_extract_norm=cfg.feat_extract_norm, hidden_size=cfg.hidden_size,
            num_hidden_layers=cfg.num_hidden_layers,
            num_attention_heads=cfg.num_attention_heads,
            intermediate_size=cfg.intermediate_size,
            num_conv_pos_embeddings=cfg.num_conv_pos_embeddings,
            num_conv_pos_embedding_groups=cfg.num_conv_pos_embedding_groups,
            vocab_size=cfg.vocab_size, layer_norm_eps=cfg.layer_norm_eps,
            do_stable_layer_norm=bool(getattr(cfg, "do_stable_layer_norm", False)),
            hidden_act=cfg.hidden_act,
        )
        if kind == "conformer":
            kw.update(position_embeddings_type=cfg.position_embeddings_type,
                      conv_depthwise_kernel_size=cfg.conv_depthwise_kernel_size,
                      rotary_embedding_base=cfg.rotary_embedding_base,
                      max_source_positions=cfg.max_source_positions)
        if kind == "wavlm":
            kw.update(num_buckets=cfg.num_buckets, max_bucket_distance=cfg.max_bucket_distance)
        return ModelConfig(**kw)


MODELS = {
    # transformers.Wav2Vec2Config() defaults == facebook/wav2vec2-base-960h
    "wav2vec2-base": ModelConfig(),
    # facebook/wav2vec2-large-960h (group-norm front end, post-LN encoder)
    "wav2vec2-large": ModelConfig(hidden_size=1024, num_hidden_layers=24,
                                  num_attention_heads=16, intermediate_size=4096),
    # facebook/wav2vec2-conformer-rel-pos-large-960h-ft (w2v2conformer.py:57)
    "wav2vec2-conformer-large": ModelConfig(
        kind="conformer", hidden_size=1024, num_hidden_layers=24, num_attention_heads=16,
        intermediate_size=4096, conv_bias=True, feat_extract_norm="layer",
        position_embeddings_type="relative", hidden_act="swish"),
    # transformers.WavLMConfig() defaults == microsoft/wavlm-base-plus (group-norm front end, post-LN encoder)
    "wavlm-base-plus": ModelConfig(kind="wavlm"),
    # microsoft/wavlm-large (layer-norm front end with conv bias, stable-LN encoder)
    "wavlm-large": ModelConfig(kind="wavlm", hidden_size=1024, num_hidden_layers=24, num_attention_heads=16,
                               intermediate_size=4096, feat_extract_norm="layer", conv_bias=True,
                               do_stable_layer_norm=True),
    # tiny variants used by the CPU/GPU parity tests (same code paths, seconds on CPU)
    "wav2vec2-tiny": ModelConfig(hidden_size=128, num_hidden_layers=2, num_attention_heads=2,
                                 intermediate_size=256, conv_dim=(64,) * 7,
                                 num_conv_pos_embeddings=16, num_conv_pos_embedding_groups=4),
}


@dataclass(frozen=True)
class Workload:
    """One BASELINE.json config: clip length, segment count, coalition count."""
    name: str
    model: str
    num_samples: int
    num_segments: int
    num_coalitions: int
    description: str = ""


WORKLOADS = {
    "C1": Workload("C1", "wav2vec2-base", 16000, 32, 256,
                   "wav2vec2-base 1 s clip, 32 segments, 256 coalitions (CPU-runnable)"),
    "C2": Workload("C2", "wav2vec2-base", 80000, 100, 2048,
                   "wav2vec2-base 5 s clip, 100 segments, 2048 coalitions"),
    "C3": Workload("C3", "wav2vec2-large", 160000, 200, 8192,
                   "wav2vec2-large 10 s clip, 200 segments, 8192 coalitions"),
    "C4": Workload("C4", "wav2vec2-conformer-large", 80000, 100, 4096,
                   "wav2vec2-conformer-large 5 s clip, 100 segments, 4096 coalitions"),
    # C2's shape on WavLM: the attention cost of the gated relative-position bias compares directly with C2
    "C6": Workload("C6", "wavlm-base-plus", 80000, 100, 2048,
                   "wavlm-base-plus 5 s clip, 100 segments, 2048 coalitions"),
}
