"""ORACLE (test infrastructure only): the time-frequency cell game of KernelSHAP over (segment, frequency band) cells.

Independent of the product package: the band filters are restated here from the semantics in include/w2s.h and the
components computed with numpy's float64 ``rfft``.  A coalition keeps or drops each cell (s, b), bit s * F + b; sample i
of its waveform is the fp32 sum, in band order from +0.0, of the kept cells' components.  The forward underneath is the
transformers-pinned one of ``callback.evaluate``.
"""
from __future__ import annotations

import numpy as np
import torch

from .callback import evaluate


def band_filters(num_samples: int, edges, sr: int = 16000) -> np.ndarray:
    """H_b(f_k) on the rfft bins f_k = k sr / L -> float64 [F, L // 2 + 1].  Interior edge e: crossover c_e(f) = 1 below
    e - 50 Hz, 0 above e + 50 Hz, cos^2(pi (f - e + 50) / 200) between; H_b = c_(e_(b+1)) - c_(e_b), c_(e_0) = 0, c_(e_F) = 1."""
    e = np.asarray(edges, dtype=np.float64)
    f = np.fft.rfftfreq(int(num_samples), d=1.0 / sr)
    lows = [np.zeros_like(f)]
    for edge in e[1:-1]:
        c = np.cos(np.pi * (f - edge + 50.0) / 200.0) ** 2
        c[f <= edge - 50.0] = 1.0
        c[f >= edge + 50.0] = 0.0
        lows.append(c)
    lows.append(np.ones_like(f))
    return np.stack([lows[b + 1] - lows[b] for b in range(len(e) - 1)])


def band_components(x, edges, sr: int = 16000) -> np.ndarray:
    """x_b = irfft(rfft(x) H_b, n = L) in float64, cast to float32 -> [F, L]."""
    x = np.asarray(x, dtype=np.float64)
    X = np.fft.rfft(x)
    H = band_filters(x.size, edges, sr)
    return np.fft.irfft(X[None, :] * H, n=x.size, axis=-1).astype(np.float32)


def materialize_cells(components: np.ndarray, Z: np.ndarray, bounds: np.ndarray) -> np.ndarray:
    """Components [F, L] and cell coalitions Z[K, M_t * F] (1 = keep, bit s * F + b) -> waveforms [K, L] float32:
    row_k[i] = sum_b (keep(k, seg(i) * F + b) ? x_b[i] : 0), fp32 adds in the order b = 0 .. F-1 from +0.0."""
    comp = np.asarray(components, dtype=np.float32)
    F = comp.shape[0]
    Z = np.atleast_2d(np.asarray(Z)).astype(bool)
    M = len(bounds) - 1
    cells = Z.reshape(Z.shape[0], M, F)
    lens = np.diff(bounds)
    out = np.zeros((Z.shape[0], comp.shape[1]), dtype=np.float32)
    for b in range(F):
        keep = np.repeat(cells[:, :, b], lens, axis=1)                    # [K, L]
        out = out + np.where(keep, comp[b][None, :], np.float32(0.0)).astype(np.float32)
    return out


@torch.no_grad()
def evaluate_coalitions_cells(sd, cfg, components, Z, bounds, **kw) -> np.ndarray:
    """f(Z[K, M_t * F]) -> [K, D]: the cell game, rows materialised by ``materialize_cells`` and evaluated by the fp32
    forward."""
    Z = np.atleast_2d(np.asarray(Z))
    batch = kw.pop("batch", 32)
    outs = []
    for s in range(0, Z.shape[0], batch):
        outs.append(evaluate(sd, cfg, materialize_cells(components, Z[s:s + batch], bounds), batch=batch, **kw))
    return np.concatenate(outs)
