"""Clip pre-processing and segmentation (host side, once per clip).

* ``normalize_clip`` -- the processor's zero-mean / unit-variance step the reference applies once to
  the clean clip before any explanation (shap_calculation.py:117; HF
  wav2vec2/feature_extraction_wav2vec2.py:78-97).  Masking is applied AFTER it, so the 0.0 baseline
  is the clip mean.
* ``segment_bounds`` -- contiguous near-equal blocks, bounds[i] = floor(i L / M).  The reference has
  no segmentation precedent; when M divides L this is the equal-block rule of the BASELINE configs.
* ``synthetic_clip`` -- the seeded synthetic 16 kHz audio used by tests and bench (SURVEY.md 8d).
* ``mel_band_edges`` / ``band_components`` -- the frequency bands of time-frequency cells (w2s_set_bands): the clip split
  into F zero-phase band components that sum to it.
"""
from __future__ import annotations

import numpy as np
import torch

MAX_BANDS = 16            # W2S_MAX_BANDS
MIN_BAND_WIDTH = 100.0    # Hz between neighbouring edges: the 100 Hz crossovers of two edges never overlap
CROSSOVER_HALF_WIDTH = 50.0


def normalize_clip(x) -> np.ndarray:
    x = np.asarray(x)
    return ((x - x.mean()) / np.sqrt(x.var() + 1e-7)).astype(np.float32)


def segment_bounds(num_samples: int, num_segments: int) -> np.ndarray:
    i = np.arange(num_segments + 1, dtype=np.int64)
    return ((i * int(num_samples)) // int(num_segments)).astype(np.int32)


def synthetic_clip(num_samples: int, seed: int = 1234, sr: int = 16000) -> np.ndarray:
    """A few drifting sinusoids plus noise, then processor-normalised."""
    rng = np.random.default_rng(seed)
    t = np.arange(num_samples, dtype=np.float64) / sr
    x = 0.3 * rng.standard_normal(num_samples)
    for f0 in (140.0, 410.0, 1270.0, 2900.0):
        amp = 0.5 + 0.5 * np.sin(2 * np.pi * rng.uniform(0.5, 3.0) * t + rng.uniform(0, 6.28))
        x += amp * np.sin(2 * np.pi * f0 * t + rng.uniform(0, 6.28))
    return normalize_clip(x)


def pack_coalitions(Z) -> np.ndarray:
    """Z[K, M] in {0,1} -> uint32 words [K, ceil(M/32)], bit m of row k = Z[k, m] (1 = keep)."""
    Z = np.atleast_2d(np.asarray(Z))
    K, M = Z.shape
    words = (M + 31) // 32
    pad = np.zeros((K, words * 32), dtype=np.uint8)
    pad[:, :M] = Z != 0
    b = np.packbits(pad.reshape(K, words, 4, 8), axis=-1, bitorder="little").reshape(K, words, 4)
    return (b[..., 0].astype(np.uint32) | (b[..., 1].astype(np.uint32) << 8) |
            (b[..., 2].astype(np.uint32) << 16) | (b[..., 3].astype(np.uint32) << 24))


def mel_band_edges(num_bands: int, sr: int = 16000) -> np.ndarray:
    """F + 1 band edges in Hz, equally spaced on the HTK mel scale (mel = 2595 log10(1 + f / 700)) from 0 to sr / 2;
    float64 [F + 1].  At sr = 16000 every F <= 16 keeps neighbouring edges >= 100 Hz apart."""
    F = int(num_bands)
    if F < 1 or F > MAX_BANDS:
        raise ValueError(f"{F} bands; need 1 <= F <= {MAX_BANDS}")
    top = 2595.0 * np.log10(1.0 + (sr / 2.0) / 700.0)
    edges = 700.0 * (10.0 ** (np.linspace(0.0, top, F + 1) / 2595.0) - 1.0)
    edges[0], edges[-1] = 0.0, sr / 2.0
    return check_band_edges(edges, sr)


def check_band_edges(edges, sr: int = 16000) -> np.ndarray:
    """Validated band edges -> float64 [F + 1]: 0 = e_0 < e_1 < ... < e_F = sr / 2, 1 <= F <= 16, neighbouring edges
    >= 100 Hz apart.  Raises ValueError naming the problem."""
    e = np.asarray(edges, dtype=np.float64).reshape(-1)
    F = e.size - 1
    if F < 1 or F > MAX_BANDS:
        raise ValueError(f"{F} bands ({e.size} edges); need 1 <= F <= {MAX_BANDS}")
    if not np.all(np.isfinite(e)):
        raise ValueError("band edges must be finite")
    if e[0] != 0.0 or e[-1] != sr / 2.0:
        raise ValueError(f"band edges must run from 0 to sr / 2 = {sr / 2.0:g} Hz, got {e[0]:g} .. {e[-1]:g}")
    gap = np.diff(e)
    if np.any(gap < MIN_BAND_WIDTH):
        i = int(np.argmin(gap))
        raise ValueError(f"band edges {e[i]:g} and {e[i + 1]:g} Hz are less than {MIN_BAND_WIDTH:g} Hz apart")
    return e


def band_filters(num_samples: int, edges, sr: int = 16000) -> np.ndarray:
    """Real, zero-phase band filters on the rfft bins f_k = k sr / L: float64 [F, L // 2 + 1].  Each interior edge e has
    the crossover c_e(f) = 1 for f <= e - 50, 0 for f >= e + 50, cos^2(pi (f - e + 50) / 200) between; H_b = c_(e_(b+1)) -
    c_(e_b) with c_(e_0) = 0 and c_(e_F) = 1, so the filters sum to 1 at every bin and each is >= 0."""
    e = check_band_edges(edges, sr)
    f = np.arange(int(num_samples) // 2 + 1, dtype=np.float64) * (sr / float(num_samples))
    w = CROSSOVER_HALF_WIDTH
    c = [np.zeros_like(f)]
    for edge in e[1:-1]:
        t = np.clip((f - edge + w) / (2.0 * w), 0.0, 1.0)
        c.append(np.where(f <= edge - w, 1.0, np.where(f >= edge + w, 0.0, np.cos(np.pi * t / 2.0) ** 2)))
    c.append(np.ones_like(f))
    return np.stack([c[b + 1] - c[b] for b in range(len(e) - 1)])


def band_components(x, edges, sr: int = 16000) -> np.ndarray:
    """The clip's band components x_b = irfft(rfft(x) H_b, n = L), in float64 then cast: float32 [F, L].  The filtering is
    circular over the clip.  Their fp32 sum is the clip within rounding; w2s_set_bands takes them."""
    xt = torch.as_tensor(x).detach().reshape(-1).to(device="cpu", dtype=torch.float64)
    L = xt.numel()
    H = torch.from_numpy(band_filters(L, edges, sr))
    comp = torch.fft.irfft(torch.fft.rfft(xt)[None, :] * H, n=L, dim=-1)
    return comp.to(torch.float32).numpy()
