"""GPU: the input-gradient path (expected gradients, the reference's production explainer: shap_calculation.py:125-162)
through the C ABI against torch autograd on the `transformers` model -- stage by stage, then end to end.

Tolerance: gradients travel through ~60 bf16-rounded stages (bf16 operands, fp32 accumulation, fp32 LayerNorm / softmax
arithmetic), so they are compared as max |g_gpu - g_ref| <= GRAD_TOL * max |g_ref| per row batch, plus a cosine similarity.
"""
import numpy as np
import pytest
import torch

from helpers import VARIANTS, build_model
from shap_transformer_asr_b200.config import MODELS

pytestmark = pytest.mark.gpu

GRAD_TOL = 0.06


@pytest.fixture(scope="module")
def P():
    import shap_transformer_asr_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def reference_grads(model, x, frames):
    """torch autograd on the transformers model: d max_v logits[r, frames[r], v] / d (x and the intermediate activations)."""
    grabs, hooks = {}, []

    def keep(name):
        def hook(mod, inp, out):
            t = out[0] if isinstance(out, tuple) else out
            t.retain_grad()
            grabs[name] = t
        return hook

    conformer = hasattr(model, "wav2vec2_conformer")
    w = model.wav2vec2_conformer if conformer else model.wav2vec2
    NL = len(w.encoder.layers)
    stable = conformer or bool(model.config.do_stable_layer_norm)
    # input of encoder layer 0: the LayerNorm'ed sum (post-LN encoders) / the un-normalised stream after dropout (stable-LN
    # encoders and the conformer, whose layers end in their own final_layer_norm)
    hooks.append((w.encoder.dropout if stable else w.encoder.layer_norm).register_forward_hook(keep("layer0")))
    for l, layer in enumerate(w.encoder.layers):
        hooks.append(layer.register_forward_hook(keep(f"layer{l + 1}")))
    hooks.append(w.feature_projection.register_forward_hook(keep("h0")))
    convs = w.feature_extractor.conv_layers
    layer_norm_front = model.config.feat_extract_norm == "layer"
    # "convu<l>": the pre-activation of conv layer l (after its norm, if it has one)
    hooks.append(convs[0].layer_norm.register_forward_hook(keep("convu0")))
    for l in range(1, len(convs)):
        hooks.append((convs[l].layer_norm if layer_norm_front else convs[l].conv).register_forward_hook(keep(f"convu{l}")))
    hooks.append(convs[-1].register_forward_hook(keep(f"conv{len(convs) - 1}")))
    xt = torch.tensor(x, requires_grad=True)
    logits = model(xt).logits
    out = logits.max(-1).values[torch.arange(len(x)), torch.as_tensor(frames, dtype=torch.long)]
    out.sum().backward()
    for h in hooks:
        h.remove()
    g = {k: v.grad.detach() for k, v in grabs.items()}
    g.update({"f." + k: v.detach() for k, v in grabs.items()})      # the forward activations at the same points
    g["f.logits"] = logits.detach()
    return xt.grad.detach().numpy(), g, out.detach().numpy(), NL


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def cosine(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30))


def _chan_last(t, T_l):
    """HF conv activations are [n, C, T] (LayerNorm'ed ones [n, T, C]); the path keeps [n, T, C]."""
    a = t.numpy()
    return a if a.shape[1] == T_l else a.transpose(0, 2, 1)


@pytest.mark.parametrize("variant,attn", [("tiny_group", "fused"), ("tiny_group", "contractions"), ("tiny_group", "cuda_core"),
                                          ("tiny_layer_stable", "fused"), ("tiny_conformer_rel", "contractions"),
                                          ("tiny_conformer_rotary", "fused"), ("tiny_conformer_rotary", "contractions")])
def test_gradient_stages_match_autograd_tiny(P, variant, attn):
    """Every stage of the backward pass against autograd (tiny model): localises a wrong kernel to its stage.  Attention
    backward as the fused tcgen05 kernel (the product path), as batched tensor-core contractions + row kernels (the product
    path of the relative-position conformer) and on the CUDA-core cross-check kernels."""
    cfg = VARIANTS[variant]
    model = build_model(cfg)
    stable = cfg.do_stable_layer_norm
    conformer = cfg.kind == "conformer"
    rng = np.random.default_rng(0)
    x = rng.standard_normal((3, 6000)).astype(np.float32)
    T = cfg.num_frames(6000)
    frames = np.array([0, 5, T - 1], dtype=np.int32)
    gx, g, out, NL = reference_grads(model, x, frames)
    eng = P.Engine(model, cfg, max_batch=4)
    eng.grad_debug(True, simt_attention=attn == "cuda_core", unfused_attention=attn == "contractions")
    grad, val = eng.grad_waveforms(torch.from_numpy(x).cuda(), frames)
    torch.cuda.synchronize()
    H = cfg.hidden_size
    lens = cfg.conv_lengths(6000)
    NC = len(lens)
    # forward activations saved by the gradient path, at the points autograd's hooks see them
    fwd = []
    for l in range(NC):
        mine = eng.grad_peek(f"f.convu{l}", (3, lens[l], cfg.conv_dim[l]), torch.bfloat16).float().cpu().numpy()
        fwd.append((f"convu{l}", rel(mine, _chan_last(g[f"f.convu{l}"], lens[l]))))
    if conformer:          # the projection is the fp32 stream itself; every layer's output (after final_layer_norm) is saved
        fwd.append(("h0", rel(eng.grad_peek("f.h0", (3, T, H)).cpu().numpy(), g["f.h0"].numpy())))
        for l in range(1, NL + 1):
            fwd.append((f"layer{l}", rel(eng.grad_peek(f"f.layer{l}", (3, T, H)).cpu().numpy(), g[f"f.layer{l}"].numpy())))
    else:
        fwd.append(("h0", rel(eng.grad_peek("f.h0", (3, T, H), torch.bfloat16).float().cpu().numpy(), g["f.h0"].numpy())))
    for l in range(NL + 1):
        if stable or conformer:
            break          # the stable-LN forward keeps the fp32 residual stream, not a normalised bf16 copy per layer
        mine = eng.grad_peek(f"f.layer{l}", (3, T, H), torch.bfloat16).float().cpu().numpy()
        fwd.append((f"layer{l}", rel(mine, g[f"f.layer{l}"].numpy())))
    lg = eng.grad_peek("f.logits", (3, T, 32)).cpu().numpy()
    fwd.append(("logits", rel(lg, g["f.logits"].numpy())))
    print("forward stages (max rel err vs transformers): " + "; ".join(f"{k} {v:.2e}" for k, v in fwd))
    report = []
    for l in range(NL, -1, -1):
        mine = eng.grad_peek(f"layer{l}", (3, T, H)).cpu().numpy()
        report.append((f"layer{l}", rel(mine, g[f"layer{l}"].numpy())))
    report.append(("h0", rel(eng.grad_peek("h0", (3, T, H)).cpu().numpy(), g["h0"].numpy())))
    mine = eng.grad_peek(f"conv{NC - 1}", (3, lens[-1], cfg.conv_dim[-1]), torch.bfloat16).float().cpu().numpy()
    report.append((f"conv{NC - 1}", rel(mine, _chan_last(g[f"conv{NC - 1}"], lens[-1]))))
    for l in range(NC - 2, -1, -1):
        mine = eng.grad_peek(f"convu{l}", (3, lens[l], cfg.conv_dim[l]), torch.bfloat16).float().cpu().numpy()
        report.append((f"convu{l}", rel(mine, _chan_last(g[f"convu{l}"], lens[l]))))
    report.append(("x", rel(grad.cpu().numpy(), gx)))
    print("gradient stages (max rel err vs autograd): " + "; ".join(f"{k} {v:.2e}" for k, v in report))
    assert max(v for _, v in fwd) < 0.03, fwd
    assert np.abs(val.cpu().numpy() - out).max() < 0.025 * np.abs(out).max() + 1e-3
    worst = max(v for _, v in report)
    assert worst < GRAD_TOL, report
    assert cosine(grad.cpu().numpy(), gx) > 0.999
    eng.close()


@pytest.mark.parametrize("name,n,L", [("tiny_group", 35, 9000), ("wav2vec2-base", 32, 16000), ("tiny_group", 3, 183600),
                                      ("wav2vec2-large", 4, 16000), ("tiny_layer_stable", 34, 9000),
                                      ("wav2vec2-large-lv60", 3, 16000), ("tiny_conformer_rel", 34, 9000),
                                      ("tiny_conformer_rotary", 33, 9000), ("wav2vec2-conformer-large", 3, 16000),
                                      ("tiny_group", 2, 330000),       # T' = 1031: nine key blocks in the fused attention backward
                                      # T' = 312 and 573 (the reference's clip): the relative-position conformer's unfused
                                      # attention backward with the rel-shift in the softmax row kernel; rotary on the fused one
                                      ("tiny_conformer_rel", 4, 100000), ("tiny_conformer_rotary", 4, 100000),
                                      ("tiny_conformer_rel", 3, 183600), ("tiny_conformer_rotary", 3, 183600)])
def test_input_gradients_match_autograd_at_batch_32(P, name, n, L):
    """d (max logit of frame j) / d waveform for >= 32 rows with different target frames (one ragged tile for the tiny
    model: 32 + 3) against torch autograd on the transformers model."""
    if name == "wav2vec2-large-lv60":      # layer-norm front end with conv bias + stable-LN encoder at full width
        import dataclasses
        cfg = dataclasses.replace(MODELS["wav2vec2-large"], feat_extract_norm="layer", conv_bias=True,
                                  do_stable_layer_norm=True, num_hidden_layers=6)
    elif name == "wav2vec2-conformer-large":   # the C4 model (w2v2conformer.py:57) at full width, 6 of its 24 layers
        import dataclasses
        cfg = dataclasses.replace(MODELS[name], num_hidden_layers=6)
    else:
        cfg = VARIANTS[name] if name in VARIANTS else MODELS[name]
    model = build_model(cfg)
    rng = np.random.default_rng(n)
    x = rng.standard_normal((n, L)).astype(np.float32)
    T = cfg.num_frames(L)
    frames = rng.integers(0, T, size=n).astype(np.int32)
    gx, _, out, _ = reference_grads(model, x, frames)
    eng = P.Engine(model, cfg, max_batch=4)
    grad, val = eng.grad_waveforms(torch.from_numpy(x).cuda(), frames)
    grad = grad.cpu().numpy()
    e, c = rel(grad, gx), cosine(grad, gx)
    per_row = [cosine(grad[i], gx[i]) for i in range(n)]
    print(f"{name} n={n} L={L}: input-gradient max rel err {e:.3e}; cosine {c:.5f}; worst row cosine {min(per_row):.5f}")
    assert np.abs(val.cpu().numpy() - out).max() < 0.025 * np.abs(out).max() + 1e-3
    assert e < GRAD_TOL and min(per_row) > 0.995
    # the same rows, one at a time, give the same gradients (no dependence on the position in the batch)
    r = min(5, n - 1)
    g1, _ = eng.grad_waveforms(torch.from_numpy(x[r:r + 1]).cuda(), frames[r:r + 1])
    assert np.abs(g1.cpu().numpy()[0] - grad[r]).max() <= 1e-6 * np.abs(grad[r]).max() + 1e-12
    eng.close()


def test_expected_gradients_explainer_properties(P):
    """ExpectedGradientsExplainer on the tiny model: layout [1, L, D] (shap_calculation.py:200-210), agreement with the
    same estimator evaluated with autograd gradients on the same (background, alpha) draws, and approximate
    completeness (sum of attributions ~ f(x) - E f(background))."""
    cfg = VARIANTS["tiny_group"]
    model = build_model(cfg)
    L = 4000
    x = P.synthetic_clip(L)
    bg = P.make_background(L, 5, seed=1)
    eng = P.Engine(model, cfg, max_batch=8)
    frames = np.array([2, 7], dtype=np.int32)
    ex = P.ExpectedGradientsExplainer(eng, bg, nsamples=64, seed=3, batch=32)
    phi = ex.shap_values(x, frames)
    assert phi.shape == (1, L, 2)
    # reference: identical draws, autograd gradients
    ref = np.zeros((L, 2))
    for d, j in enumerate(frames):
        rng = np.random.default_rng([3, int(j)])
        rind = rng.integers(0, 5, 64)
        alpha = rng.uniform(size=64).astype(np.float32)
        xs = bg[rind] + alpha[:, None] * (x[None] - bg[rind])
        gx, _, _, _ = reference_grads(model, xs.astype(np.float32), np.full(64, j, np.int32))
        ref[:, d] = (gx.astype(np.float64) * (x[None] - bg[rind])).mean(0)
    e, c = rel(phi[0], ref), cosine(phi[0], ref)
    print(f"expected gradients (64 samples, 2 outputs): max rel err vs autograd estimator {e:.3e}; cosine {c:.5f}")
    # The model is invariant to the input scale (GroupNorm over time), so d f / d x grows like 1 / alpha along the path
    # x_s = bg + alpha (x - bg) and the small-alpha draws dominate the mean with heavy cancellation (x . grad f = 0 for a
    # scale-invariant f): the estimator amplifies the per-gradient rounding (1.5e-2, tests above) several times.
    assert c > 0.98 and e < 0.25
    with torch.no_grad():
        fx = model(torch.from_numpy(x)[None]).logits.max(-1).values[0, frames].numpy()
        fb = model(torch.from_numpy(bg)).logits.max(-1).values[:, frames].mean(0).numpy()
    gap = np.abs(phi[0].sum(0) - (fx - fb)) / (np.abs(fx - fb) + 1e-6)
    print(f"completeness gap (64 samples): {gap}")
    eng.close()


def test_gradient_path_rejects_unbuilt_configurations(P):
    """What the gradient path does not cover fails loudly: the conformer's CUDA-core attention cross-check, a target
    frame outside the clip, and the relative-position conformer on clips past the 1024 frames its attention backward
    takes (T' = 1031), before anything is launched."""
    cfg = VARIANTS["tiny_conformer_rel"]
    eng = P.Engine(build_model(cfg), cfg, max_batch=2)
    eng.grad_debug(False, simt_attention=True)
    with pytest.raises(RuntimeError, match="gradient path"):
        eng.grad_waveforms(torch.zeros((1, 4000), device="cuda"), [0])
    eng.grad_debug(False, simt_attention=False)
    with pytest.raises(RuntimeError, match="target frame"):
        eng.grad_waveforms(torch.zeros((1, 4000), device="cuda"), [10 ** 6])
    assert cfg.num_frames(330000) == 1031
    with pytest.raises(RuntimeError, match="at most 1024 frames"):
        eng.grad_waveforms(torch.zeros((1, 330000), device="cuda"), [0])
    # the handle stays usable
    g, _ = eng.grad_waveforms(torch.randn((1, 4000), device="cuda"), [0])
    assert torch.isfinite(g).all()
    eng.close()


def test_model_wrapper_output_is_differentiable_as_in_the_reference(P):
    """B1 of SURVEY.md 8b: shap.GradientExplainer calls `outputs = self.model(*X); selected = outputs[:, idx]` and then
    autograd.grad(selected, X) (conformer_test.ipynb:95).  callbacks.ModelWrapper serves exactly that: its output carries
    an autograd node whose backward is the device vector-Jacobian product -- one-hot (one output index) and general
    (a weighted sum over frames) upstream gradients against torch autograd on the transformers model."""
    cfg = VARIANTS["tiny_group"]
    model = build_model(cfg)
    rng = np.random.default_rng(11)
    x = rng.standard_normal((5, 7000)).astype(np.float32)
    T = cfg.num_frames(7000)
    eng = P.Engine(model, cfg, max_batch=8)
    wrap = P.ModelWrapper(eng)
    xg = torch.from_numpy(x).cuda().requires_grad_(True)
    out = wrap(xg[:, None, :])                                   # [B, 1, L] as shap hands it over (shap_calculation.py:33-36)
    assert out.shape == (5, T) and out.requires_grad
    idx = 9
    (g_one,) = torch.autograd.grad(out[:, idx].sum(), xg, retain_graph=True)
    xr = torch.tensor(x, requires_grad=True)
    ref_logits = model(xr).logits
    ref_out = ref_logits.max(-1).values
    # max over the vocabulary is not differentiable across a tie: weight only the frames whose top-2 margin is clear of
    # the bf16 logit error (random-init logits are nearly flat, so several frames are within it)
    top2 = ref_logits.detach().topk(2, -1).values
    clear = ((top2[..., 0] - top2[..., 1]) > 0.05).float()
    assert clear.sum() >= 10
    w = (torch.from_numpy(rng.standard_normal((5, T)).astype(np.float32)) * clear).cuda()
    (g_gen,) = torch.autograd.grad((out * w).sum(), xg)
    (r_one,) = torch.autograd.grad(ref_out[:, idx].sum(), xr, retain_graph=True)
    (r_gen,) = torch.autograd.grad((ref_out * w.cpu()).sum(), xr)
    e1, e2 = rel(g_one.cpu().numpy(), r_one.numpy()), rel(g_gen.cpu().numpy(), r_gen.numpy())
    print(f"ModelWrapper autograd: one-hot max rel err {e1:.3e}; weighted-sum max rel err {e2:.3e}")
    assert np.abs(out.detach().cpu().numpy() - ref_out.detach().numpy()).max() < 0.025 * ref_out.abs().max().item()
    assert e1 < GRAD_TOL and e2 < GRAD_TOL
    # without requires_grad the wrapper stays on the evaluation path (no autograd node, no saved activations)
    assert not wrap(torch.from_numpy(x).cuda()).requires_grad
    eng.close()


def deeplift_reference_grads(model, rows, frames, rescale_silu=True, glu_placeholder=False):
    """The handler rules of feasability_tests/custom_shap_handlers.py:35-80 as torch backward hooks on the transformers
    model (what shap's PyTorchDeep does with them): `rows` = [explained | reference] halves; SiLU modules use the rescale
    multiplier (nonlinear_1d), GLU the reference's placeholder, everything else the ordinary gradient (linear_1d /
    no handler).  Returns the rule-modified input gradients of the explained half."""
    saved, hooks = {}, []

    def keep(mod, inp, out):
        saved[mod] = (inp[0].detach(), out.detach())

    def silu_rule(mod, grad_in, grad_out):
        xin, y = saved[mod]
        h = xin.shape[0] // 2
        dx, dy = xin[:h] - xin[h:], y[:h] - y[h:]
        rep = [2] + [1] * (dx.dim() - 1)
        safe = torch.where(dx.abs() < 1e-6, torch.ones_like(dx), dx)
        return (torch.where(dx.abs().repeat(rep) < 1e-6, grad_in[0], grad_out[0] * (dy / safe).repeat(rep)),)

    def glu_rule(mod, grad_in, grad_out):
        xin, _ = saved[mod]
        h = xin.shape[0] // 2
        dx = xin[:h] - xin[h:]
        rep0 = [2] + [1] * (dx.dim() - 1)
        rep1 = [1, 2] + [1] * (grad_out[0].dim() - 2)
        return (torch.where(dx.abs().repeat(rep0) < 1e-6, grad_in[0], grad_out[0].repeat(rep1) * 5e-6),)

    for mod in model.modules():
        if rescale_silu and isinstance(mod, torch.nn.SiLU):
            hooks += [mod.register_forward_hook(keep), mod.register_full_backward_hook(silu_rule)]
        if glu_placeholder and isinstance(mod, torch.nn.GLU):
            hooks += [mod.register_forward_hook(keep), mod.register_full_backward_hook(glu_rule)]
    xt = torch.tensor(rows, requires_grad=True)
    n = len(rows) // 2
    logits = model(xt).logits
    out = logits.max(-1).values[torch.arange(n), torch.as_tensor(frames[:n], dtype=torch.long)]   # explained half only
    out.sum().backward()
    for h in hooks:
        h.remove()
    return xt.grad.detach().numpy()[:n], out.detach().numpy()


@pytest.mark.parametrize("variant,glu", [("tiny_conformer_rel", False), ("tiny_conformer_rotary", False),
                                         ("tiny_conformer_rel", True), ("tiny_group", False)])
def test_deeplift_handler_rules_match_torch_hooks(P, variant, glu):
    """f4 of SURVEY.md 8: the reference's DeepLIFT handler rules (rescale on SiLU, linear pass-through on the norms, the GLU
    placeholder as an option) on the device backward pass, against the same rules as torch backward hooks; then the
    explainer built on them (mean over the background of modified-gradient x (input - reference), layout [1, L, D]).
    For the GELU-only Wav2Vec2ForCTC the rules must change nothing."""
    cfg = VARIANTS[variant]
    model = build_model(cfg)
    rng = np.random.default_rng(5)
    L, B = 6000, 5
    x = rng.standard_normal(L).astype(np.float32)
    bg = P.make_background(L, B, seed=4) + 0.3 * rng.standard_normal((B, L)).astype(np.float32)   # references far from zero too
    T = cfg.num_frames(L)
    frames = np.array([3, T - 2], dtype=np.int32)
    rows = np.concatenate([np.repeat(x[None], 2 * B, 0), np.tile(bg, (2, 1))]).astype(np.float32)   # 10 explained | 10 references
    row_frames = np.concatenate([np.repeat(frames, B)] * 2).astype(np.int32)
    ref_g, ref_out = deeplift_reference_grads(model, rows, row_frames, True, glu)
    plain_g, _ = deeplift_reference_grads(model, rows, row_frames, False, False)
    eng = P.Engine(model, cfg, max_batch=4)
    eng.grad_rules(True, glu)
    g, val = eng.grad_waveforms(torch.from_numpy(rows).cuda(), row_frames)
    eng.grad_rules(False, False)
    g = g.cpu().numpy()
    assert np.all(g[2 * B:] == 0)                       # reference rows carry no seed
    e = rel(g[:2 * B], ref_g)
    changed = rel(ref_g, plain_g)                       # how much the rules move the gradient at all
    print(f"{variant} glu_placeholder={glu}: rule-modified gradient max rel err {e:.3e} "
          f"(the rules change the plain gradient by {changed:.3e} of its maximum)")
    assert e < GRAD_TOL and cosine(g[:2 * B], ref_g) > 0.998
    if variant == "tiny_group":
        assert changed == 0.0                           # GELU-only model: nothing to rescale
    else:
        assert changed > 0.02                           # the test would not notice a missing rule otherwise
    assert np.abs(val.cpu().numpy()[:2 * B] - ref_out).max() < 0.025 * np.abs(ref_out).max() + 1e-3
    phi = P.DeepLiftExplainer(eng, bg, rescale_silu=True, glu_placeholder=glu).shap_values(x, frames)
    assert phi.shape == (1, L, 2)
    want = (ref_g.reshape(2, B, L) * (x[None, None] - bg[None])).mean(1).T
    assert rel(phi[0], want) < 2 * GRAD_TOL and cosine(phi[0], want) > 0.995
    eng.close()
