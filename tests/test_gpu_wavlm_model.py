"""GPU: WavLMForCTC through the whole evaluation path -- the tiny goldens in every mode, long clips past the bucket clamp,
KernelSHAP at C1 size on wavlm-base-plus, the callback shapes, the C2-style invariants on the C6 workload, and the
gradient path's refusal.  Tolerances are those of tests/test_gpu_parity.py."""
import os

import numpy as np
import pytest
import torch

from helpers import rel_err
from oracle import callback as CB
from oracle import wavlm_forward as WL
from oracle.kernelshap_ref import KernelExplainerRef
from oracle.make_golden_wavlm import VARIANTS as WAVLM_VARIANTS, build
from shap_transformer_asr_b200.config import MODELS, WORKLOADS

pytestmark = pytest.mark.gpu

LOGIT_TOL = 0.025
PHI_TOL = 0.02


@pytest.fixture(scope="module")
def P():
    import shap_transformer_asr_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


@torch.no_grad()
def oracle_eval(sd, cfg, X, mode, frames=None, tokens=None, batch=32):
    """CB.evaluate with the WavLM oracle: waveforms [n, L] -> reduced outputs [n, D]."""
    X = np.atleast_2d(np.asarray(X, dtype=np.float32))
    outs = [CB.reduce_logits(WL.ctc_logits(sd, cfg, torch.from_numpy(np.ascontiguousarray(X[s:s + batch]))), mode,
                             frames, tokens).float() for s in range(0, X.shape[0], batch)]
    return torch.cat(outs).numpy()


@pytest.mark.parametrize("name", list(WAVLM_VARIANTS))
@pytest.mark.parametrize("mode", ["validate", "tcgen05", "fp32_preln"])
def test_tiny_wavlm_logits_match_golden(P, golden_dir, name, mode):
    g = np.load(os.path.join(golden_dir, f"{name}.npz"))
    cfg = WAVLM_VARIANTS[name]
    eng = P.Engine(build(cfg), cfg, max_batch=2, validate_gemm=mode == "validate", validate_attn=mode == "validate",
                   preln_fp32=mode == "fp32_preln")
    eng.set_targets("logits")
    out = eng.eval_waveforms(torch.from_numpy(g["x"]).cuda()).view(g["logits"].shape).cpu().numpy()   # ragged last tile
    err = rel_err(out, g["logits"])
    print(f"{name} [{mode}] logits rel err {err:.3e}")
    assert err < LOGIT_TOL
    eng.close()


@pytest.mark.parametrize("name,L", [("tiny_wavlm_stable", 47000), ("tiny_wavlm", 100000), ("tiny_wavlm", 330000)])
def test_long_wavlm_clips_match_oracle(P, name, L):
    """T' = 146 / 312 / 1031: two key blocks, streaming, and relative distances past the bucket clamp (|j - i| >= 778)."""
    cfg = WAVLM_VARIANTS[name]
    model = build(cfg)
    x = np.random.default_rng(L).standard_normal((2, L)).astype(np.float32)
    with torch.no_grad():
        ref = WL.ctc_logits(WL.state_dict_of(model), cfg.to_dict(), torch.from_numpy(x)).numpy()
    assert ref.shape[1] == {47000: 146, 100000: 312, 330000: 1031}[L]
    eng = P.Engine(model, cfg, max_batch=2)
    eng.set_targets("logits")
    out = eng.eval_waveforms(torch.from_numpy(x).cuda()).view(ref.shape).cpu().numpy()
    err = rel_err(out, ref)
    print(f"{name} L={L} T'={ref.shape[1]} logits rel err {err:.3e}")
    assert err < LOGIT_TOL
    eng.close()


@pytest.fixture(scope="module")
def base_engine(P):
    cfg = MODELS["wavlm-base-plus"]
    model = build(cfg)
    eng = P.Engine(model, cfg, max_batch=32)
    yield eng, model, cfg
    eng.close()


def test_c1_size_kernelshap_matches_oracle(P, base_engine):
    eng, model, cfg = base_engine
    sd, d = WL.state_dict_of(model), cfg.to_dict()
    clip = P.synthetic_clip(16000)
    M, K = 32, 256
    res = P.KernelShapExplainer(eng, nsamples=K, seed=0).explain(clip, num_segments=M)
    bounds = CB.segment_bounds(16000, M)
    frames, tokens = res["frames"], res["tokens"]
    f = lambda Z: oracle_eval(sd, d, CB.materialize(clip, np.atleast_2d(Z), bounds), "logprob", frames, tokens)
    ref = KernelExplainerRef(f, M)
    np.random.seed(0)
    Zr, wr = ref.sample(K)
    assert np.array_equal(res["Z"], Zr.astype(np.uint8)) and np.array_equal(res["weights"], wr)   # bit-exact coalitions
    y_ref = f(Zr)
    phi_ref = ref.solve(y_ref, f(np.ones((1, M)))[0], f(np.zeros((1, M)))[0])
    phi = res["phi"].cpu().numpy()
    e_y = np.abs(res["y"].cpu().numpy() - y_ref).max()
    e_phi = np.abs(phi - phi_ref).max() / np.abs(phi_ref).max()
    print(f"wavlm-base-plus C1 KernelSHAP: y max abs err {e_y:.3e}; phi max rel err {e_phi:.3e}; D={len(frames)}")
    assert int(res["status"].item()) == 0
    assert e_phi < PHI_TOL


def test_callback_shapes(P, base_engine):
    eng, model, cfg = base_engine
    sd, d = WL.state_dict_of(model), cfg.to_dict()
    x = np.random.default_rng(5).standard_normal((3, 16000)).astype(np.float32)
    with torch.no_grad():
        ref_logits = WL.ctc_logits(sd, d, torch.from_numpy(x))
    wrap = P.ModelWrapper(eng)
    xt = torch.from_numpy(x).cuda()
    for inp in (xt, xt[:, None, :], xt[:, None, None, :]):
        out = wrap(inp)
        assert out.shape == (3, 49)
        assert rel_err(out.cpu().numpy(), ref_logits.max(-1).values.numpy()) < LOGIT_TOL
    fn = P.make_predict_function(eng, 7, 11)
    o = fn(x.astype(np.float64))
    assert o.shape == (3,) and o.dtype == np.float32
    assert np.abs(o - ref_logits[:, 7, 11].numpy()).max() < LOGIT_TOL * ref_logits.abs().max().item()
    assert fn(x[0].astype(np.float64)).shape == (1,)
    o = P.make_lime_predict_fn(eng)(x)
    assert o.shape == (3, 1)
    assert np.abs(o - ref_logits.mean(-1).mean(1, keepdim=True).numpy()).max() < LOGIT_TOL * ref_logits.abs().max().item()


def test_c6_invariants(P, base_engine):
    """C6 (wavlm-base-plus, 5 s clip, 100 segments): batch-position independence, all-ones row = explicit waveform,
    masked rows = host-materialised rows, bit for bit."""
    eng, model, cfg = base_engine
    wl = WORKLOADS["C6"]
    clip = P.synthetic_clip(wl.num_samples)
    M = wl.num_segments
    eng.set_clip(clip, num_segments=M)
    Z, kw, _ = P.sample_coalitions(M, wl.num_coalitions, seed=0)
    rows = np.concatenate([np.ones((1, M), np.uint8), np.zeros((1, M), np.uint8), Z[:94]])
    T = cfg.num_frames(wl.num_samples)
    frames = np.arange(0, T, 3, dtype=np.int32)
    tokens = (frames * 7 % 32).astype(np.int32)
    eng.set_targets("logprob", frames, tokens)
    bits = eng.bits_to_device(rows)
    y1 = eng.eval_bits(bits)
    assert torch.equal(y1, eng.eval_bits(bits.flip(0).contiguous()).flip(0))
    assert torch.equal(y1[:1], eng.eval_waveforms(torch.from_numpy(clip).cuda()[None]))
    Xm = torch.from_numpy(CB.materialize(clip, rows[2:6], CB.segment_bounds(wl.num_samples, M))).cuda()
    assert torch.equal(y1[2:6], eng.eval_waveforms(Xm))
    assert torch.isfinite(y1).all() and (y1 <= 0).all()


def test_gradient_path_refuses_wavlm(P):
    """The gradient path has no backward of the gated bias: expected gradients and ModelWrapper autograd fail with an
    error that names WavLM, while the forward without gradients still runs."""
    cfg = WAVLM_VARIANTS["tiny_wavlm"]
    model = build(cfg)
    eng = P.Engine(model, cfg, max_batch=8)
    L = 4000
    x = P.synthetic_clip(L)
    ex = P.ExpectedGradientsExplainer(eng, P.make_background(L, 5, seed=1), nsamples=8, seed=3, batch=8)
    with pytest.raises(RuntimeError, match="WavLM"):
        ex.shap_values(x, np.array([2], dtype=np.int32))
    wrap = P.ModelWrapper(eng)
    xg = torch.from_numpy(np.stack([x, x[::-1].copy()])).cuda().requires_grad_(True)
    with pytest.raises(RuntimeError, match="WavLM"):
        out = wrap(xg)
        torch.autograd.grad(out[:, 3].sum(), xg)
    with torch.no_grad():
        ref = WL.ctc_logits(WL.state_dict_of(model), cfg.to_dict(), xg.detach().cpu()).max(-1).values.numpy()
    out = wrap(xg.detach())
    assert not out.requires_grad
    assert rel_err(out.cpu().numpy(), ref) < LOGIT_TOL
    eng.close()
