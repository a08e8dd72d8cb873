"""ORACLE (test infrastructure only): the background-averaged coalition game of ``shap.KernelExplainer(f, data)``.

Restated from memory of shap's KernelExplainer (unpinned, like ``kernelshap_ref.py``): with a background ``data`` [B, L]
every coalition is evaluated once per background row, each dropped segment taking that row's samples, and the outputs
are averaged with the background weights.  The forward underneath is the transformers-pinned one of ``callback.evaluate``.
"""
from __future__ import annotations

import numpy as np
import torch

from .callback import evaluate


def materialize_background(x: np.ndarray, Z: np.ndarray, bounds: np.ndarray, bg: np.ndarray) -> np.ndarray:
    """Coalition matrix Z[K, M] (1 = keep) and background bg[B, L] -> waveforms [K * B, L], row k * B + b =
    keep ? x : bg[b] (the device's row order)."""
    Z = np.atleast_2d(np.asarray(Z))
    bg = np.atleast_2d(np.asarray(bg, dtype=np.float32))
    keep = np.repeat(Z.astype(bool), np.diff(bounds), axis=1)                     # [K, L]
    out = np.where(keep[:, None, :], np.asarray(x, dtype=np.float32)[None, None, :], bg[None, :, :])
    return out.reshape(-1, bg.shape[1]).astype(np.float32)


@torch.no_grad()
def evaluate_coalitions_background(sd, cfg, x, Z, bounds, bg, weights=None, **kw) -> np.ndarray:
    """Background-averaged game: y[k] = sum_b w_b f(row (k, b)) with w normalised to sum 1 (uniform by default), the
    rows evaluated by the transformers-pinned forward in fp32 and averaged in fp64 -> [K, D] float64."""
    Z = np.atleast_2d(np.asarray(Z))
    bg = np.atleast_2d(np.asarray(bg, dtype=np.float32))
    B = bg.shape[0]
    w = np.ones(B) if weights is None else np.asarray(weights, dtype=np.float64)
    w = w / w.sum()
    batch = kw.pop("batch", 32)
    per = max(1, batch // B)
    outs = []
    for s in range(0, Z.shape[0], per):
        rows = evaluate(sd, cfg, materialize_background(x, Z[s:s + per], bounds, bg), batch=batch, **kw)
        outs.append(np.einsum("kbd,b->kd", rows.reshape(-1, B, rows.shape[-1]).astype(np.float64), w))
    return np.concatenate(outs)
