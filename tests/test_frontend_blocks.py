"""Host block table of the feature encoder's constant-frame skip (w2s_frontend_blocks) against a brute-force per-frame
receptive-field check, and a numpy restatement of the live / needed / fill rules of skip_lists_kernel on the benchmark's
own coalitions."""
import ctypes as C

import numpy as np
import pytest

from oracle import callback as CB
from oracle.kernelshap_ref import KernelExplainerRef
from shap_transformer_asr_b200 import MODELS, _lib

KERNEL = MODELS["wav2vec2-base"].conv_kernel
STRIDE = MODELS["wav2vec2-base"].conv_stride


def table(L, bounds):
    lib = _lib.load()
    k = np.asarray(KERNEL, np.int32)
    s = np.asarray(STRIDE, np.int32)
    b = np.asarray(bounds, np.int32)
    M = len(b) - 1
    n = lib.w2s_frontend_blocks(len(k), k.ctypes.data, s.ctypes.data, L, b.ctypes.data, M, None, 0)
    assert n > 0
    out = np.zeros((n, 4), np.int32)
    assert lib.w2s_frontend_blocks(len(k), k.ctypes.data, s.ctypes.data, L, b.ctypes.data, M, out.ctypes.data, n) == n
    return out


def frames_per_layer(L):
    T, n = [], L
    for k, s in zip(KERNEL, STRIDE):
        n = (n - k) // s + 1
        T.append(n)
    return T


def brute(L, bounds):
    """Per frame, the sample interval of its receptive field; per block, the segments and lower-layer rows it touches."""
    seg = np.repeat(np.arange(len(bounds) - 1), np.diff(bounds))
    T = frames_per_layer(L)
    rows = []
    lo = [np.arange(T[0]) * STRIDE[0]]
    hi = [lo[0] + KERNEL[0] - 1]
    for l in range(1, len(KERNEL)):
        f = np.arange(T[l])
        lo.append(lo[l - 1][f * STRIDE[l]])
        hi.append(hi[l - 1][f * STRIDE[l] + KERNEL[l] - 1])
        for j in range(0, T[l], 128):
            f1 = min(j + 127, T[l] - 1)
            rows.append((seg[lo[l][j]], seg[hi[l][f1]], j * STRIDE[l] // 128, (f1 * STRIDE[l] + KERNEL[l] - 1) // 128))
    return np.asarray(rows, np.int32), T


def lists(tab, T, keep):
    """skip_lists_kernel for one coalition: per layer (live, fill) block indices."""
    nb = [(t + 127) // 128 for t in T[1:]]
    off = np.concatenate([[0], np.cumsum(nb)])
    kept = np.concatenate([[0], np.cumsum(keep)])
    nonconst = kept[tab[:, 1] + 1] - kept[tab[:, 0]] > 0
    needed = np.zeros(len(tab), bool)
    res = [None] * len(nb)
    for l in range(len(nb) - 1, -1, -1):
        sl = slice(off[l], off[l + 1])
        if l == len(nb) - 1:
            needed[sl] = True
        live = nonconst[sl].copy()
        cand = np.flatnonzero(needed[sl] & ~nonconst[sl])
        if len(cand):
            live[cand[0]] = True
        res[l] = (np.flatnonzero(live), np.flatnonzero(needed[sl] & ~live))
        if l > 0:
            for j in np.flatnonzero(live):
                needed[off[l - 1] + tab[off[l] + j, 2]: off[l - 1] + tab[off[l] + j, 3] + 1] = True
    return res


@pytest.mark.parametrize("L,M,seed", [(80000, 100, None), (80000, 37, 1), (16000, 300, 2), (3000, 9, 3)])
def test_block_table_matches_receptive_fields(L, M, seed):
    if seed is None:
        bounds = np.asarray(CB.segment_bounds(L, M), np.int32)
    else:
        rng = np.random.default_rng(seed)
        cuts = np.sort(rng.integers(0, L + 1, M - 1))   # arbitrary bounds: empty segments and ones shorter than 400 samples
        bounds = np.concatenate([[0], cuts, [L]]).astype(np.int32)
    ref, _ = brute(L, bounds)
    np.testing.assert_array_equal(table(L, bounds), ref)


def test_block_table_rejects_bad_bounds():
    lib = _lib.load()
    k = np.asarray(KERNEL, np.int32)
    s = np.asarray(STRIDE, np.int32)
    b = np.asarray([0, 50, 40, 100], np.int32)
    assert lib.w2s_frontend_blocks(len(k), k.ctypes.data, s.ctypes.data, 100, b.ctypes.data, 3, None, 0) == -1


def test_lists_cover_what_the_next_layer_reads():
    """Every row a live block reads is in a live or filled block; filled blocks are all constant; on the benchmark's
    coalitions (C2 geometry, oracle sampler, seed 0) about a third of the conv1 blocks are not contracted."""
    L, M = 80000, 100
    bounds = np.asarray(CB.segment_bounds(L, M), np.int32)
    tab, T = brute(L, bounds)
    nb = [(t + 127) // 128 for t in T[1:]]
    off = np.concatenate([[0], np.cumsum(nb)])
    np.random.seed(0)
    Z, _ = KernelExplainerRef(lambda z: z, M).sample(2048)
    live_frac = np.zeros(len(nb))
    for z in Z[:256]:
        keep = z.astype(np.int64)
        kept = np.concatenate([[0], np.cumsum(keep)])
        res = lists(tab, T, keep)
        for l, (live, fill) in enumerate(res):
            rows = tab[off[l]: off[l + 1]]
            assert not np.any(kept[rows[fill, 1] + 1] - kept[rows[fill, 0]])   # filled blocks see only dropped audio
            live_frac[l] += len(live) / nb[l]
            if l > 0:
                have = np.zeros(nb[l - 1], bool)
                have[res[l - 1][0]] = True
                have[res[l - 1][1]] = True
                for j in live:
                    assert have[rows[j, 2]: rows[j, 3] + 1].all()
        assert len(res[-1][0]) + len(res[-1][1]) == nb[-1]
    live_frac /= 256
    print("live block fraction per layer (conv1 .. conv6):", np.round(live_frac, 3))
    assert 0.55 < live_frac[0] < 0.75
