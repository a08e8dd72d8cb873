"""CPU: the frequency-band pieces of time-frequency cells that run without a GPU -- the band filters and components, the
mel edges, argument validation before any device call, and the oracle's cell order."""
import os
import re

import numpy as np
import pytest

from oracle import bands_ref as BD
from oracle import callback as CB
from shap_transformer_asr_b200 import (KernelShapExplainer, _lib, band_arrays, band_components, band_filters,
                                       mel_band_edges, synthetic_clip)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SR = 16000


@pytest.mark.parametrize("L,F", [(16000, 4), (12001, 8), (4000, 1), (80000, 16), (999, 2)])
def test_filters_sum_to_one_and_are_nonnegative(L, F):
    H = band_filters(L, mel_band_edges(F), SR)
    assert H.shape == (F, L // 2 + 1)
    assert np.abs(H.sum(0) - 1.0).max() <= 1e-12
    assert H.min() >= 0.0
    assert np.abs(H - BD.band_filters(L, mel_band_edges(F), SR)).max() <= 1e-12


@pytest.mark.parametrize("L,F", [(16000, 4), (12001, 8), (80000, 16)])
def test_components_sum_to_the_clip_and_match_the_oracle(L, F):
    x = synthetic_clip(L)
    edges = mel_band_edges(F)
    comp = band_components(x, edges)
    assert comp.shape == (F, L) and comp.dtype == np.float32
    scale = np.abs(x).max()
    total = np.zeros(L, np.float32)
    for b in range(F):
        total = total + comp[b]
    assert np.abs(total.astype(np.float64) - x).max() <= F * 2.0 ** -24 * scale
    assert np.abs(comp.astype(np.float64) - BD.band_components(x, edges)).max() <= 1e-6 * scale


@pytest.mark.parametrize("freq", [440.0, 3000.0])
def test_a_tone_lands_in_its_band(freq):
    L, F = 16000, 8
    t = np.arange(L) / SR
    x = np.sin(2 * np.pi * freq * t).astype(np.float32)
    edges = mel_band_edges(F)
    comp = band_components(x, edges).astype(np.float64)
    energy = (comp ** 2).sum(1)
    b = int(np.searchsorted(edges, freq) - 1)
    assert edges[b] < freq < edges[b + 1]
    assert energy[b] >= 0.99 * energy.sum()


def test_mel_band_edges_are_valid_for_every_band_count():
    for F in range(1, _lib.MAX_BANDS + 1):
        e = mel_band_edges(F)
        assert e.shape == (F + 1,) and e[0] == 0.0 and e[-1] == SR / 2
        assert np.all(np.diff(e) >= 100.0)
    for bad in (0, _lib.MAX_BANDS + 1):
        with pytest.raises(ValueError, match="bands"):
            mel_band_edges(bad)


@pytest.mark.parametrize("edges,match", [
    ([0.0, 1000.0, 8000.0 - 1], "sr / 2"),
    ([10.0, 1000.0, 8000.0], "sr / 2"),
    ([0.0, 1000.0, 1050.0, 8000.0], "100 Hz"),
    ([0.0, 8000.0, 1000.0, 8000.0], "100 Hz"),
    ([0.0], "bands"),
    (list(np.linspace(0.0, 8000.0, 18)), "bands"),
    ([0.0, np.nan, 8000.0], "finite"),
])
def test_bad_band_edges_are_refused(edges, match):
    with pytest.raises(ValueError, match=match):
        band_filters(1000, edges, SR)


def test_band_arrays_validation():
    comp = np.zeros((4, 100), np.float32)
    assert band_arrays(comp, num_samples=100, num_segments=25).shape == (4, 100)
    with pytest.raises(ValueError, match=r"\[F, L\]"):
        band_arrays(np.zeros(100, np.float32))
    with pytest.raises(ValueError, match="bands"):
        band_arrays(np.zeros((0, 100), np.float32))
    with pytest.raises(ValueError, match="bands"):
        band_arrays(np.zeros((_lib.MAX_BANDS + 1, 100), np.float32))
    with pytest.raises(ValueError, match="samples"):
        band_arrays(comp, num_samples=99)
    with pytest.raises(ValueError, match="2048"):
        band_arrays(comp, num_samples=100, num_segments=513)
    with pytest.raises(ValueError, match="background"):
        band_arrays(comp, num_samples=100, num_segments=25, background_rows=2)
    with pytest.raises(ValueError, match="None"):
        band_arrays(None)


class _HostEngine:
    """Stands in for Engine up to the first device call: explain must reject bad arguments before that."""
    background_rows = 0
    num_bands = 0

    def set_clip(self, clip, num_segments=1, baseline=0.0):
        self.num_samples, self.num_segments = len(clip), num_segments

    def __getattr__(self, name):
        raise AssertionError(f"explain reached Engine.{name} with invalid band arguments")


@pytest.mark.parametrize("kwargs,match", [
    (dict(band_edges=mel_band_edges(4), background=np.zeros((2, 640), np.float32)), "background"),
    (dict(band_edges=[0.0, 50.0, 8000.0]), "100 Hz"),
    (dict(band_edges=[0.0, 4000.0]), "sr / 2"),
    (dict(band_edges=list(np.linspace(0.0, 8000.0, 18))), "bands"),
    (dict(band_edges=mel_band_edges(16), num_segments=129), "2048"),
])
def test_explain_rejects_bad_band_arguments_before_any_device_call(kwargs, match):
    ex = KernelShapExplainer(_HostEngine(), nsamples=8, seed=0)
    kwargs.setdefault("num_segments", 4)
    with pytest.raises(ValueError, match=match):
        ex.explain(np.zeros(640, np.float32), **kwargs)


def _cells(L=24, M=3, F=2, seed=0):
    rng = np.random.default_rng(seed)
    comp = rng.standard_normal((F, L)).astype(np.float32)
    return comp, CB.segment_bounds(L, M)


def test_materialize_cells_all_kept_and_all_dropped():
    comp, bounds = _cells(L=30, M=3, F=3)
    K = 2
    Z = np.stack([np.ones(9, np.uint8), np.zeros(9, np.uint8)])
    X = BD.materialize_cells(comp, Z, bounds)
    assert X.shape == (K, 30) and X.dtype == np.float32
    assert np.array_equal(X[0], (comp[0] + comp[1]) + comp[2])           # fp32 adds in band order
    assert np.array_equal(X[1], np.zeros(30, np.float32))
    assert not np.signbit(X[1]).any()                                    # +0.0, not -0.0


def test_materialize_cells_bit_order_is_segment_major():
    comp, bounds = _cells(L=24, M=3, F=2)
    for s in range(3):
        for b in range(2):
            Z = np.zeros((1, 6), np.uint8)
            Z[0, s * 2 + b] = 1
            X = BD.materialize_cells(comp, Z, bounds)[0]
            want = np.zeros(24, np.float32)
            want[bounds[s]:bounds[s + 1]] = comp[b, bounds[s]:bounds[s + 1]]
            assert np.array_equal(X, want), (s, b)
    # with F = 1 the cell game is the time-only masker on the one component
    Z = np.array([[1, 0, 1], [0, 1, 1]], np.uint8)
    assert np.array_equal(BD.materialize_cells(comp[:1], Z, bounds), CB.materialize(comp[0], Z, bounds))


def test_header_band_bound_matches_the_binding():
    text = open(os.path.join(ROOT, "include", "w2s.h")).read()
    assert int(re.search(r"#define W2S_MAX_BANDS (\d+)", text).group(1)) == _lib.MAX_BANDS
