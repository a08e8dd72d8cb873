"""The reference's model-evaluation callbacks, re-hosted on the B200 engine (same names, argument
meaning and return shapes), plus the fused coalition form.

==============================  =====================================================================
reference interface             replacement here
==============================  =====================================================================
``ModelWrapper`` (torch module) shap_calculation.py:23-52          -> :class:`ModelWrapper`
``predict_function`` (numpy)    feasability_tests/w2v2conformer.py:116-131 -> :func:`make_predict_function`
``lime_predict_fn`` (numpy)     feasability_tests/lime_shap_wav2vec2_comparison.py:60-71 -> :func:`make_lime_predict_fn`
``masker(x, mask)``             feasability_tests/conformer_test.ipynb:138-141 -> :func:`masker`
masker + model pair             (what an explainer calls per coalition batch) -> :class:`CoalitionCallback`
==============================  =====================================================================
"""
from __future__ import annotations

import numpy as np
import torch

from .preprocess import pack_coalitions


class _MaxLogitFunction(torch.autograd.Function):
    """ModelWrapper's output as an autograd node: forward = the evaluation path, backward = the device
    vector-Jacobian product (w2s_vjp_waveforms), so `outputs[:, idx]` can be differentiated w.r.t. the waveform exactly
    as shap.GradientExplainer does (traceback in conformer_test.ipynb:95: `autograd.grad(selected, x)`)."""

    @staticmethod
    def forward(ctx, x, engine):
        ctx.engine = engine
        ctx.save_for_backward(x)
        engine.set_targets("max")
        return engine.eval_waveforms(x)

    @staticmethod
    def backward(ctx, gout):
        (x,) = ctx.saved_tensors
        return ctx.engine.vjp_waveforms(x, gout), None


class ModelWrapper(torch.nn.Module):
    """forward(x[B, L] | [B, 1, L] | [B, 1, 1, L]) -> max logit per frame [B, T'] (shap_calculation.py:31-50).

    The all-ones attention mask of the reference (:39) is a no-op in HF and is not modelled; the
    DEBUG statistics of :45-47 (three device syncs per call) are deliberately not reproduced.  When the input
    requires grad the output carries an autograd node whose backward is the device input-gradient path (configurations
    it does not cover yet raise at backward time)."""

    def __init__(self, engine):
        super().__init__()
        self.engine = engine

    def forward(self, x):
        if x.dim() == 4:
            x = x.squeeze(1).squeeze(1)
        elif x.dim() == 3:
            x = x.squeeze(1)
        x = x.to(device=self.engine.device, dtype=torch.float32)
        if x.stride(-1) != 1:
            x = x.contiguous()
        if torch.is_grad_enabled() and x.requires_grad:
            return _MaxLogitFunction.apply(x, self.engine)
        self.engine.set_targets("max")
        return self.engine.eval_waveforms(x)


def make_predict_function(engine, timestep_to_explain: int, token_id_to_explain: int, mode: str = "logit"):
    """numpy [n, L] or [L] (any float dtype) -> numpy float32 [n]: logits[:, t*, tok*]
    (feasability_tests/w2v2conformer.py:116-131; 1-D input is promoted as at :124-125)."""

    def predict_function(x):
        xt = torch.from_numpy(np.ascontiguousarray(x)).float()
        if xt.ndim == 1:
            xt = xt.unsqueeze(0)
        xt = xt.to(engine.device)
        engine.set_targets(mode, [timestep_to_explain], [token_id_to_explain])
        return engine.eval_waveforms(xt)[:, 0].cpu().numpy()

    return predict_function


def make_lime_predict_fn(engine):
    """numpy [n_samples, n_features] -> numpy [n_samples, 1]: mean logit over vocab and time
    (feasability_tests/lime_shap_wav2vec2_comparison.py:60-71)."""

    def lime_predict_fn(inputs):
        xt = torch.from_numpy(np.ascontiguousarray(inputs)).float().to(engine.device)
        engine.set_targets("mean")
        return engine.eval_waveforms(xt).cpu().numpy()

    return lime_predict_fn


def masker(x, mask, baseline: float = 0.0):
    """Host restatement of the notebook masker's fill rule (conformer_test.ipynb:138-141) in shap's
    keep-convention: samples where ``mask`` is true are kept, the rest become ``baseline`` (0.0)."""
    return np.where(np.asarray(mask, dtype=bool), np.asarray(x, dtype=np.float32), np.float32(baseline))


class CoalitionCallback:
    """The fused masker + model callable handed to an explainer: f(Z[n, M]) -> [n, D].

    ``Z`` is a host numpy {0,1} matrix [n, engine.num_features] (1 = segment, or with bands time-frequency cell, kept).
    Each call bit-packs it, copies it to the
    device through pinned memory, runs mask -> Wav2Vec2 -> per-character reduction on the B200 and
    copies the [n, D] result back -- the end-to-end path timed as ``e2e`` by bench.py."""

    def __init__(self, engine):
        self.engine = engine
        self._pin_in = None
        self._pin_out = None
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def __call__(self, Z):
        eng = self.engine
        Z = np.atleast_2d(np.asarray(Z))
        eng.check_coalition_width(Z.shape[1], packed=False)
        words = pack_coalitions(Z).view(np.int32)
        if self._pin_in is None or self._pin_in.shape != words.shape:
            self._pin_in = torch.empty(words.shape, dtype=torch.int32).pin_memory()
        self._pin_in.numpy()[...] = words
        bits = self._pin_in.to(eng.device, non_blocking=True)
        out = eng.eval_bits(bits)
        if self._pin_out is None or self._pin_out.shape != out.shape:
            self._pin_out = torch.empty(out.shape, dtype=torch.float32).pin_memory()
        self._pin_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.h2d_bytes = words.nbytes
        self.d2h_bytes = self._pin_out.numel() * 4
        return self._pin_out.numpy().copy()
