"""GPU: KernelSHAP against a background dataset -- the background-fill conv0 variants, the per-coalition mean and the
explainer on top of them.

Bit-exact checks compare the fused path with the same device forward on materialised rows (w2s_mask / the oracle's
materialize_background -> eval_waveforms) and the background mean with an exact host replay of its documented fp32 fma
order.  Model-level parity uses the tolerances of tests/test_gpu_parity.py."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from helpers import VARIANTS, build_model
from oracle import background_ref as BR
from oracle import callback as CB
from oracle import w2v2_forward as W
from oracle.kernelshap_ref import KernelExplainerRef, brute_force_shapley
from oracle.make_golden_wavlm import VARIANTS as WAVLM_VARIANTS, build as build_wavlm
from shap_transformer_asr_b200.config import MODELS

pytestmark = pytest.mark.gpu

PHI_TOL = 0.02
L_TINY, M_TINY = 12000, 10


@pytest.fixture(scope="module")
def P():
    import shap_transformer_asr_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def _model(name):
    if name in WAVLM_VARIANTS:
        cfg = WAVLM_VARIANTS[name]
        return build_wavlm(cfg), cfg
    cfg = VARIANTS[name]
    return build_model(cfg), cfg


def _fma32(a: np.float32, b: np.float32, c: np.float32) -> np.float32:
    """fp32 fmaf(a, b, c) on the host: the exact a * b + c rounded once to nearest-even fp32."""
    exact = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    r = np.float32(float(exact))            # within one ulp of the correctly rounded value (double rounding)
    best = None
    for cand in (np.nextafter(r, np.float32(-np.inf)), r, np.nextafter(r, np.float32(np.inf))):
        d = abs(Fraction(float(cand)) - exact)
        if best is None or d < best[0] or (d == best[0] and (cand.view(np.uint32) & 1) == 0):
            best = (d, cand)
    return best[1]


def host_bg_mean(rows: np.ndarray, w32: np.ndarray, B: int) -> np.ndarray:
    """The documented reduction: out[k, c] = fmaf(w[B-1], r[k*B+B-1, c], ... fmaf(w[0], r[k*B, c], 0))."""
    r = rows.reshape(-1, B, rows.shape[-1]).astype(np.float32)
    out = np.zeros((r.shape[0], r.shape[2]), dtype=np.float32)
    for k in range(r.shape[0]):
        for c in range(r.shape[2]):
            acc = np.float32(0)
            for b in range(B):
                acc = _fma32(w32[b], r[k, b, c], acc)
            out[k, c] = acc
    return out


def _coalitions(P, M, K, seed=0):
    Z, _, _ = P.sample_coalitions(M, K, seed=seed)
    return np.concatenate([np.zeros((1, M), np.uint8), np.ones((1, M), np.uint8), Z])


def _setup(P, eng, clip, M, mode="logprob"):
    eng.set_clip(clip, num_segments=M)
    eng.set_targets("logits")
    logits = eng.eval_bits(eng.bits_to_device(np.ones((1, M), np.uint8))).view(-1, eng.config.vocab_size).cpu().numpy()
    frames, tokens = P.char_targets(logits)
    eng.set_targets(mode, frames, tokens)
    return frames, tokens


# ---------------------------------------------------------------------------------------------------------------------
# 1 + 2: the default path is untouched
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,max_batch", [("tiny_group", 16), ("wav2vec2-base", 0)])
def test_zero_fill_is_unchanged_before_and_after_a_background(P, name, max_batch):
    if name in VARIANTS:
        model, cfg = _model(name)
        L, M, K = L_TINY, M_TINY, 40
    else:
        cfg = MODELS[name]
        model, L, M, K = build_model(cfg), 16000, 32, 200
    eng = P.Engine(model, cfg, max_batch=max_batch)
    clip = P.synthetic_clip(L)
    _setup(P, eng, clip, M)
    bits = eng.bits_to_device(_coalitions(P, M, K))
    before = eng.eval_bits(bits).clone()
    eng.set_background(P.make_background(L, 3, seed=1), [1.0, 2.0, 0.5])
    with_bg = eng.eval_bits(bits).clone()
    eng.clear_background()
    after = eng.eval_bits(bits).clone()
    eng.set_clip(clip, num_segments=M, baseline=0.0)        # explicit baseline 0: the same path
    again = eng.eval_bits(bits)
    # the degenerate background: one all-zero row of weight 1 is the zero fill, bit for bit
    eng.set_background(np.zeros((1, L), np.float32), [1.0])
    zero_row = eng.eval_bits(bits)
    torch.cuda.synchronize()
    assert torch.equal(before, after) and torch.equal(before, again)
    assert torch.equal(before, zero_row)
    assert not torch.equal(before, with_bg)
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3: fused == materialised, and the mean == the documented fp32 fma order
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["tiny_group", "tiny_layer_stable", "tiny_conformer_rel", "tiny_wavlm"])
def test_fused_background_equals_materialised_rows(P, name):
    model, cfg = _model(name)
    eng = P.Engine(model, cfg, max_batch=16)
    clip = P.synthetic_clip(L_TINY)
    _setup(P, eng, clip, M_TINY)
    Z = _coalitions(P, M_TINY, 30)
    bits = eng.bits_to_device(Z)
    B = 4
    bg = P.make_background(L_TINY, B, seed=5)
    bg[1] += 0.3 * P.synthetic_clip(L_TINY)[::-1]        # a row with speech-like content, not only noise
    bounds = CB.segment_bounds(L_TINY, M_TINY)
    # each row alone: the fused fill equals the device forward of the materialised waveforms, bit for bit
    per_row = []
    for b in range(B):
        eng.set_background(bg[b:b + 1])
        fused = eng.eval_bits(bits).clone()
        X = torch.from_numpy(BR.materialize_background(clip, Z, bounds, bg[b:b + 1])).cuda()
        assert torch.equal(eng.mask(bits), X)                      # w2s_mask selects what the oracle selects
        explicit = eng.eval_waveforms(X)
        torch.cuda.synchronize()
        assert torch.equal(fused, explicit), f"{name}: background row {b}"
        per_row.append(explicit.cpu().numpy())
    # all rows: the reported mean is the documented fp32 fma order over the per-row outputs
    w = np.array([0.5, 2.0, 1.0, 0.25])
    eng.set_background(bg, w)
    y = eng.eval_bits(bits).cpu().numpy()
    w32 = (w / w.sum()).astype(np.float32)
    rows = np.stack(per_row, axis=1).reshape(-1, y.shape[1])      # [K * B, D], row k * B + b
    assert np.array_equal(eng.mask(bits).cpu().numpy(), BR.materialize_background(clip, Z, bounds, bg))
    assert np.array_equal(y, host_bg_mean(rows, w32, B))
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4: tiling independence (coalitions straddling tiles, ragged last tile)
# ---------------------------------------------------------------------------------------------------------------------
def test_background_result_does_not_depend_on_the_tile(P):
    model, cfg = _model("tiny_group")
    clip = P.synthetic_clip(L_TINY)
    Z = _coalitions(P, M_TINY, 61)           # 63 coalitions x 5 rows = 315 rows: tiles of 7 split coalitions
    bg = P.make_background(L_TINY, 5, seed=2)
    w = [1.0, 3.0, 0.5, 2.0, 1.5]
    outs = []
    for mb in (7, 32, 0):
        eng = P.Engine(model, cfg, max_batch=mb)
        _setup(P, eng, clip, M_TINY)
        eng.set_background(bg, w)
        outs.append(eng.eval_bits(eng.bits_to_device(Z)).cpu())
        eng.close()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


# ---------------------------------------------------------------------------------------------------------------------
# 5: parity with the fp32 forward at C1 size
# ---------------------------------------------------------------------------------------------------------------------
def test_c1_background_kernelshap_matches_oracle(P):
    cfg = MODELS["wav2vec2-base"]
    model = build_model(cfg)
    sd, d = W.state_dict_of(model), cfg.to_dict()
    eng = P.Engine(model, cfg, max_batch=32)
    L, M, K = 16000, 32, 256
    clip = P.synthetic_clip(L)
    bg = P.make_background(L, 5, seed=3)
    wts = np.array([1.0, 2.0, 0.5, 1.5, 3.0])
    res = P.KernelShapExplainer(eng, nsamples=K, seed=0).explain(clip, num_segments=M, background=bg,
                                                                  background_weights=wts)
    assert np.allclose(res["background_weights"], wts / wts.sum())
    bounds = CB.segment_bounds(L, M)
    frames, tokens = res["frames"], res["tokens"]
    f = lambda Z: BR.evaluate_coalitions_background(sd, d, clip, np.atleast_2d(Z), bounds, bg, wts, mode="logprob",
                                                    frames=frames, tokens=tokens, batch=40)
    ref = KernelExplainerRef(f, M)
    np.random.seed(0)
    Zr, wr = ref.sample(K)
    assert np.array_equal(res["Z"], Zr.astype(np.uint8)) and np.array_equal(res["weights"], wr)   # bit-exact coalitions
    y_ref = f(Zr)
    fx, fnull = f(np.ones((1, M)))[0], f(np.zeros((1, M)))[0]
    phi_ref = ref.solve(y_ref, fx, fnull)
    phi = res["phi"].cpu().numpy()
    e_y = np.abs(res["y"].cpu().numpy() - y_ref).max()
    e_phi = np.abs(phi - phi_ref).max() / np.abs(phi_ref).max()
    print(f"C1 background KernelSHAP (B=5): y max abs err {e_y:.3e}; phi max rel err {e_phi:.3e}; D={len(frames)}")
    assert int(res["status"].item()) == 0
    assert e_phi < PHI_TOL
    assert np.abs(phi.sum(0) - (res["fx"] - res["fnull"]).cpu().numpy()).max() < 1e-6
    # the engine is left on the zero fill
    assert eng.background_rows == 0
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6: exact Shapley values of the background-averaged game under full enumeration
# ---------------------------------------------------------------------------------------------------------------------
def test_full_enumeration_with_kmeans_background_equals_brute_force(P):
    cfg = VARIANTS["tiny_group"]
    model = build_model(cfg)
    sd, d = W.state_dict_of(model), cfg.to_dict()
    clip = P.synthetic_clip(L_TINY)
    M = 10
    pool = np.concatenate([P.make_background(L_TINY, 6, seed=7),
                           0.2 * np.stack([P.synthetic_clip(L_TINY)[::-1], np.roll(P.synthetic_clip(L_TINY), 999)])])
    data, weights = P.kmeans_background(pool.astype(np.float32), 3)
    eng = P.Engine(model, cfg, max_batch=64)
    res = P.KernelShapExplainer(eng, nsamples=2 ** M, seed=0).explain(clip, num_segments=M, background=(data, weights))
    assert res["Z"].shape[0] == 2 ** M - 2 and int(res["status"].item()) == 0
    bounds = CB.segment_bounds(L_TINY, M)
    f = lambda Zm: BR.evaluate_coalitions_background(sd, d, clip, np.atleast_2d(Zm), bounds, data, weights,
                                                     mode="logprob", frames=res["frames"], tokens=res["tokens"], batch=63)
    shap_exact = brute_force_shapley(f, M)
    phi = res["phi"].cpu().numpy()
    err = np.abs(phi - shap_exact).max() / np.abs(shap_exact).max()
    print(f"full enumeration M={M}, B=3 kmeans rows: GPU KernelSHAP vs brute-force Shapley max rel err {err:.3e}")
    assert err < 2e-2
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# 7: errors fail before anything is launched, and the handle stays usable
# ---------------------------------------------------------------------------------------------------------------------
def test_background_errors_are_raised_before_launch(P):
    model, cfg = _model("tiny_group")
    eng = P.Engine(model, cfg, max_batch=16)
    clip = P.synthetic_clip(L_TINY)
    _setup(P, eng, clip, M_TINY)
    bits = eng.bits_to_device(_coalitions(P, M_TINY, 20))
    ref = eng.eval_bits(bits).clone()
    bg = P.make_background(L_TINY, 2, seed=0)
    launches = eng.launch_count()
    lib, h = eng.lib, eng._h
    # the library's own checks (the Python wrapper validates first; call the C ABI directly)
    t = torch.from_numpy(P.make_background(L_TINY + 8, 2, seed=0)).cuda()
    w = np.ones(2)
    import ctypes as C
    wp = w.ctypes.data_as(C.POINTER(C.c_double))
    assert lib.w2s_set_background(h, t.data_ptr(), 2, L_TINY + 8, L_TINY + 8, wp, eng._stream()) != 0
    assert b"samples" in lib.w2s_last_error(h)
    assert lib.w2s_set_background(h, t.data_ptr(), 257, L_TINY, L_TINY, wp, eng._stream()) != 0
    assert b"257" in lib.w2s_last_error(h)
    for bad in ([-1.0, 2.0], [np.nan, 1.0], [0.0, 0.0], [np.inf, 1.0]):
        wb = np.asarray(bad, dtype=np.float64)
        assert lib.w2s_set_background(h, t.data_ptr(), 2, L_TINY, L_TINY, wb.ctypes.data_as(C.POINTER(C.c_double)),
                                      eng._stream()) != 0
        assert b"weight" in lib.w2s_last_error(h)
    # through the wrappers
    with pytest.raises(ValueError, match="samples"):
        eng.set_background(P.make_background(L_TINY - 1, 2, seed=0))
    for bad in ([-1.0, 1.0], [np.nan, 1.0], [0.0, 0.0]):
        with pytest.raises(ValueError, match="weights"):
            eng.set_background(bg, bad)
    ex = P.KernelShapExplainer(eng, nsamples=32, seed=0)
    with pytest.raises(ValueError, match="rows"):
        ex.explain(clip, num_segments=M_TINY, background=np.zeros((0, L_TINY), np.float32))
    with pytest.raises(ValueError, match="samples"):
        ex.explain(clip, num_segments=M_TINY, background=P.make_background(L_TINY + 1, 2, seed=0))
    # a later set_clip with a new length: eval and mask refuse the stale background
    eng.set_background(bg)
    eng.set_clip(P.synthetic_clip(L_TINY + 320), num_segments=M_TINY)
    with pytest.raises(RuntimeError, match="background rows have"):
        eng.eval_bits(bits)
    with pytest.raises(RuntimeError, match="background rows have"):
        eng.mask(bits)
    torch.cuda.synchronize()
    assert eng.launch_count() == launches            # nothing was launched by any failing call
    # the handle is still usable: back to the first clip, zero fill, same outputs
    eng.clear_background()
    _setup(P, eng, clip, M_TINY)
    assert torch.equal(eng.eval_bits(bits), ref)
    eng.close()
