"""B200-native masked-coalition evaluation path of SHAP-Transformer-ASR (see DESIGN.md).

Host side in Python/PyTorch (plumbing only); all compute in ``libw2s.so`` (hand-written CUDA for
sm_100a behind the C ABI of ``include/w2s.h``).  There is no CPU fallback.
"""
from .config import MODELS, WORKLOADS, ModelConfig, Workload  # noqa: F401
from .preprocess import band_components, band_filters, mel_band_edges, normalize_clip, pack_coalitions, segment_bounds, synthetic_clip  # noqa: F401
from .targets import char_targets, first_char_target, greedy_transcript  # noqa: F401
from .kernelshap import KernelShapExplainer, expand_to_samples, kmeans_background, sample_coalitions  # noqa: F401
from .callbacks import CoalitionCallback, ModelWrapper, make_lime_predict_fn, make_predict_function, masker  # noqa: F401
from .engine import Engine, background_arrays, band_arrays, debug_attention, debug_attention_bias, debug_attention_bwd, debug_ctc, debug_errors, debug_gemm, error_tables, reference_arrays, relative_buckets  # noqa: F401
from .metrics import eta_raw, eta_raw_segments, greedy_ctc_decode, wer  # noqa: F401
from .sweep import add_noise, explain_test_set, make_test_set  # noqa: F401
from .modelzoo import build_random_init_model  # noqa: F401
from .expected_gradients import ExpectedGradientsExplainer, make_background  # noqa: F401
from .deeplift import DeepLiftExplainer  # noqa: F401
