"""CPU: the background-dataset pieces that run without a GPU -- kmeans_background (shap.kmeans restated), the argument
validation of Engine.set_background / KernelShapExplainer.explain, the oracle's row order, and the ABI constant."""
import os
import re

import numpy as np
import pytest

from oracle import background_ref as BR
from oracle import callback as CB
from shap_transformer_asr_b200 import KernelShapExplainer, _lib, background_arrays, kmeans_background

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pool(n=40, L=9, seed=0):
    rng = np.random.default_rng(seed)
    centres = rng.standard_normal((4, L)) * 3
    return (centres[rng.integers(0, 4, n)] + 0.1 * rng.standard_normal((n, L))).astype(np.float32)


def test_kmeans_background_is_deterministic_and_rounds_to_column_values():
    X = _pool()
    d1, w1 = kmeans_background(X, 4)
    d2, w2 = kmeans_background(X, 4)
    assert np.array_equal(d1, d2) and np.array_equal(w1, w2)
    assert d1.shape == (4, X.shape[1]) and d1.dtype == np.float32 and w1.dtype == np.float64
    for j in range(X.shape[1]):
        assert np.all(np.isin(d1[:, j], X[:, j])), f"column {j}: a centre coordinate the column never takes"
    unrounded, _ = kmeans_background(X, 4, round_values=False)
    assert not np.all(np.isin(unrounded[:, 0], X[:, 0]))


def test_kmeans_background_weights_are_cluster_sizes():
    from sklearn.cluster import KMeans
    X = _pool(n=37)
    _, w = kmeans_background(X, 3)
    labels = KMeans(n_clusters=3, random_state=0).fit(X.astype(np.float64)).labels_
    assert np.array_equal(w, np.bincount(labels, minlength=3).astype(np.float64))
    assert w.sum() == len(X)


def test_kmeans_with_one_cluster_per_row_gives_back_the_rows():
    X = _pool(n=6, L=5, seed=3)
    d, w = kmeans_background(X, len(X))
    assert np.array_equal(w, np.ones(len(X)))
    assert sorted(map(tuple, d)) == sorted(map(tuple, X))


def test_kmeans_background_rejects_bad_k():
    with pytest.raises(ValueError):
        kmeans_background(_pool(n=5), 6)
    with pytest.raises(ValueError):
        kmeans_background(_pool(n=5), 0)


def test_background_arrays_validation():
    bg = np.zeros((3, 100), np.float32)
    data, w = background_arrays(bg)
    assert data.shape == (3, 100) and np.array_equal(w, np.ones(3))
    assert background_arrays(np.zeros(100, np.float32))[0].shape == (1, 100)     # one row [L]
    with pytest.raises(ValueError, match="rows"):
        background_arrays(np.zeros((0, 100), np.float32))
    with pytest.raises(ValueError, match="rows"):
        background_arrays(np.zeros((_lib.MAX_BACKGROUND + 1, 4), np.float32))
    with pytest.raises(ValueError, match="samples"):
        background_arrays(bg, num_samples=99)
    with pytest.raises(ValueError, match="weights"):
        background_arrays(bg, [1.0, 2.0])
    for bad in ([1.0, -0.5, 1.0], [1.0, np.nan, 1.0], [np.inf, 1.0, 1.0]):
        with pytest.raises(ValueError, match="finite and >= 0"):
            background_arrays(bg, bad)
    with pytest.raises(ValueError, match="sum to zero"):
        background_arrays(bg, [0.0, 0.0, 0.0])


class _HostEngine:
    """Stands in for Engine up to the first device call: explain must reject bad arguments before that."""
    background_rows = 0

    def set_clip(self, clip, num_segments=1, baseline=0.0):
        self.num_samples, self.num_segments = len(clip), num_segments

    def __getattr__(self, name):
        raise AssertionError(f"explain reached Engine.{name} with invalid background arguments")


@pytest.mark.parametrize("kwargs,match", [
    (dict(background=np.zeros((0, 64), np.float32)), "rows"),
    (dict(background=np.zeros((2, 63), np.float32)), "samples"),
    (dict(background=np.zeros((2, 64), np.float32), background_weights=[1.0, -1.0]), "weights"),
    (dict(background=(np.zeros((2, 64), np.float32), [1.0, 1.0]), background_weights=[1.0, 1.0]), "either"),
    (dict(background_weights=[1.0]), "without a background"),
])
def test_explain_rejects_bad_background_arguments_before_any_device_call(kwargs, match):
    ex = KernelShapExplainer(_HostEngine(), nsamples=8, seed=0)
    with pytest.raises(ValueError, match=match):
        ex.explain(np.zeros(64, np.float32), num_segments=4, **kwargs)


def test_oracle_background_rows_are_coalition_major():
    rng = np.random.default_rng(0)
    L, M = 12, 3
    x = rng.standard_normal(L).astype(np.float32)
    bg = rng.standard_normal((2, L)).astype(np.float32)
    Z = np.array([[1, 0, 1], [0, 0, 0], [1, 1, 1]], np.uint8)
    bounds = CB.segment_bounds(L, M)
    X = BR.materialize_background(x, Z, bounds, bg)
    assert X.shape == (6, L)
    for k in range(3):
        for b in range(2):
            keep = np.repeat(Z[k].astype(bool), np.diff(bounds))
            assert np.array_equal(X[k * 2 + b], np.where(keep, x, bg[b]))
    # one zero row is the zero-fill masker
    assert np.array_equal(BR.materialize_background(x, Z, bounds, np.zeros((1, L), np.float32)), CB.materialize(x, Z, bounds))


def test_header_background_bound_matches_the_binding():
    text = open(os.path.join(ROOT, "include", "w2s.h")).read()
    assert int(re.search(r"#define W2S_MAX_BACKGROUND (\d+)", text).group(1)) == _lib.MAX_BACKGROUND
