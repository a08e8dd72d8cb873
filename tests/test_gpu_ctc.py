"""GPU: the transcript-level output W2S_OUT_CTC, out = log p_CTC(y | x) = -WavXForCTC(x, labels=y).loss (reduction "sum"),
and its input gradient.

Kernel level: w2s_debug_ctc (the head reduction's CTC code and the gradient seed) against float64 F.ctc_loss and its
autograd gradient on the same fp32 logits.  Error analysis: every alpha step rounds at most 2^-24 |alpha| (plus the
one-ulp error of expf / logf), over T' steps, so |d log p| <= 2e-4 max(1, |ref|) for T' <= 1031; the measured maximum
is below 2e-6, and the test holds it to 1e-5.  The seed is a difference of probabilities in [0, 1], compared absolutely.

Model level: two references, so a failure can be attributed -- (a) the float64 CTC of the engine's own W2S_OUT_LOGITS
output, at the kernel tolerance; (b) the HF loss of the fp32 transformers model.  For (b): d log p / d z_t,v = gamma_t(v)
- softmax(z_t)_v sums to at most 2 in absolute value over v, so |d log p| <= 2 T' max |d z|, and the logits themselves
are within LOGIT_TOL * max |z| (tests/test_gpu_parity.py): the tolerance is 2 T' LOGIT_TOL max |z|.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import VARIANTS, build_model
from oracle import background_ref as BR
from oracle import callback as CB
from oracle import ctc_ref
from oracle import w2v2_forward as W
from oracle.kernelshap_ref import brute_force_shapley
from oracle.make_golden_wavlm import VARIANTS as WAVLM_VARIANTS, build as build_wavlm
from shap_transformer_asr_b200.config import MODELS
from shap_transformer_asr_b200.targets import frames_needed, greedy_transcript
from test_gpu_background import host_bg_mean

pytestmark = pytest.mark.gpu

LOGP_TOL = 1e-5       # |d log p| <= LOGP_TOL * max(1, |ref|)  (2e-4 by the error analysis; measured <= 1.6e-6)
SEED_TOL = 2e-3       # max |d (d log p / d logits)|, typical and peaky logits
LOGIT_TOL = 0.025     # tests/test_gpu_parity.py
GRAD_TOL = 0.06       # tests/test_gpu_grad.py


@pytest.fixture(scope="module")
def P():
    import shap_transformer_asr_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


# ---------------------------------------------------------------------------------------------------------------------
# kernel level
# ---------------------------------------------------------------------------------------------------------------------
def ref_ctc(logits32: torch.Tensor, ys, blank, which):
    """float64 F.ctc_loss: out [n, D] and d out[r, which[r]] / d logits[r] [n, T, V]."""
    z = logits32.double().cpu().requires_grad_(True)
    out = ctc_ref.ctc_logp(z, ys, blank)
    sel = out[torch.arange(z.shape[0]), torch.as_tensor(which)]
    sel.sum().backward()
    return out.detach().numpy(), z.grad.numpy()


def make_transcript(rng, T, U, V, blank, alphabet):
    """U labels from `alphabet` non-blank symbols (repeats likely); None if it needs more than T frames."""
    pool = [v for v in range(V) if v != blank][:alphabet]
    y = [int(v) for v in rng.choice(pool, U)] if U else []
    return y if frames_needed(y) <= T else None


def tight_transcript(rng, T, V, blank):
    """U + repeats = T exactly, with repeated labels.  Past T' = 2 * 512 - 1 no transcript within the cap is tight (512
    equal labels need 1023 frames, the most any 512 labels need); there the tightest one at the cap is returned."""
    if T >= 2 * 512 - 1:
        return [[v for v in range(V) if v != blank][2]] * 512
    pool = [v for v in range(V) if v != blank][:3]
    y, need = [], 0
    while need < T:
        v = int(rng.choice(pool))
        extra = 1 + (bool(y) and y[-1] == v)
        if need + extra > T:
            v = next(p for p in pool if p != y[-1])
            extra = 1
        y.append(v)
        need += extra
    assert frames_needed(y) == T and len(y) <= 512
    return y


def alignment(y, T, blank, rng, late=False):
    """One valid frame labelling for y over T frames (blanks spread at random, or all blanks first when `late`)."""
    seq = []
    for u, v in enumerate(y):
        if u and y[u - 1] == v:
            seq.append(blank)
        seq.append(v)
    spare = T - len(seq)
    if late:
        return [blank] * spare + seq
    cuts = np.sort(rng.integers(0, len(seq) + 1, spare))
    out, j = [], 0
    for i, v in enumerate(seq + [None]):
        while j < spare and cuts[j] == i:
            out.append(blank)
            j += 1
        if v is not None:
            out.append(v)
    return out


def family_logits(family, rng, n, T, V, y, blank):
    z = rng.standard_normal((n, T, V)).astype(np.float32)
    if family == "peaky":          # +-30-nat margins along one alignment of y
        for r in range(n):
            a = alignment(y, T, blank, rng)
            z[r] *= 0.5
            z[r, np.arange(T), a] += 30.0
    elif family == "forced":       # blank dominates early; y must be emitted tightly at the end through states that are
        for r in range(n):         # negligible (~ -30 nats) for most of the clip
            a = alignment(y, T, blank, rng, late=True)
            z[r, np.arange(T), a] += 30.0
            z[r, :T // 2, blank] += 30.0
    elif family == "low":          # log p near -1e4
        z *= 1e4 / (2.0 * T)
        z[:, :, blank] -= 2e4 / T
    return z


KERNEL_T = [1, 31, 32, 33, 249, 573, 1031]


@pytest.mark.parametrize("T", KERNEL_T)
@pytest.mark.parametrize("V,blank", [(32, 0), (128, 77)])
@pytest.mark.parametrize("family", ["typical", "peaky", "forced", "low"])
def test_debug_ctc_matches_float64_ctc_loss(P, T, V, blank, family):
    rng = np.random.default_rng([T, V, blank, len(family)])
    ys = [[], [int([v for v in range(V) if v != blank][5])], tight_transcript(rng, T, V, blank)]
    cap = make_transcript(rng, T, 512, V, blank, 24)
    if cap is not None:
        ys.append(cap)
    mid = make_transcript(rng, T, max(1, T // 3), V, blank, 4)     # repeats from a 4-letter alphabet
    if mid is not None:
        ys.append(mid)
    n = 2 * len(ys)
    which = [i % len(ys) for i in range(n)]
    z = np.concatenate([family_logits(family, rng, 2, T, V, ys[i], blank) for i in range(len(ys))])
    zt = torch.from_numpy(z).cuda()
    out, dl = P.debug_ctc(zt, ys, blank=blank, which=which, grad=True)
    out, dl = out.cpu().numpy(), dl.cpu().numpy()
    ref, gref = ref_ctc(torch.from_numpy(z), ys, blank, which)
    assert np.all(np.isfinite(out)) and np.all(np.isfinite(dl)), "NaN or inf in the output or the seed"
    e = np.abs(out - ref) / np.maximum(1.0, np.abs(ref))
    eg = float(np.abs(dl - gref).max())
    print(f"T={T} V={V} blank={blank} {family} U={[len(y) for y in ys]}: max |d log p|/max(1,|ref|) {e.max():.2e}; "
          f"max |d seed| {eg:.2e}; log p range [{ref.min():.4g}, {ref.max():.4g}]")
    assert e.max() <= LOGP_TOL, (e.max(), np.unravel_index(e.argmax(), e.shape))
    if family in ("typical", "peaky"):
        assert eg <= SEED_TOL
    # the value of a row does not depend on its position: row 0 alone
    one = P.debug_ctc(zt[:1].contiguous(), ys, blank=blank)
    assert torch.equal(one.cpu(), torch.from_numpy(out[:1]))


def test_debug_ctc_refuses_infeasible_transcripts(P):
    z = torch.zeros((1, 4, 32), device="cuda")
    P.debug_ctc(z, [[5, 5, 6]], blank=0)                               # needs 4 frames: fine
    with pytest.raises(RuntimeError, match="transcript 1 needs 6 frames, T = 4"):
        P.debug_ctc(z, [[5], [5, 5, 6, 6]], blank=0)


# ---------------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------------
def _model(name):
    if name in WAVLM_VARIANTS:
        cfg = WAVLM_VARIANTS[name]
        return build_wavlm(cfg), cfg
    cfg = VARIANTS[name] if name in VARIANTS else MODELS[name]
    return build_model(cfg), cfg


def hf_logp(model, x, ys):
    """-WavXForCTC(x, labels=y).loss, reduction "sum", blank = pad_token_id = 0, fp32 on the CPU: [n, D]."""
    model.config.ctc_loss_reduction = "sum"
    model.config.ctc_zero_infinity = False
    out = np.zeros((len(x), len(ys)))
    with torch.no_grad():
        for r in range(len(x)):
            for d, y in enumerate(ys):
                lab = torch.as_tensor(y, dtype=torch.long)[None] if len(y) else torch.full((1, 1), -100)
                out[r, d] = -float(model(torch.from_numpy(x[r:r + 1]), labels=lab).loss)
    return out


def _transcripts(rng, logits, T, V):
    """the greedy transcript, a random feasible one with repeats, and the empty one"""
    return [greedy_transcript(logits).tolist(), make_transcript(rng, T, min(T // 2, 40), V, 0, 6), []]


@pytest.mark.parametrize("name,mode", [(n, m) for n in ["tiny_group", "tiny_layer_stable", "tiny_conformer_rel",
                                                         "tiny_conformer_rotary", "tiny_wavlm"]
                                       for m in ["validate", "tcgen05", "fp32_preln"]] + [("wav2vec2-base", "tcgen05")])
def test_eval_waveforms_transcripts_match_the_hf_loss(P, name, mode):
    model, cfg = _model(name)
    L, n = (16000, 3) if name == "wav2vec2-base" else (9000, 5)
    eng = P.Engine(model, cfg, max_batch=0 if name == "wav2vec2-base" else 4, validate_gemm=mode == "validate",
                   validate_attn=mode == "validate", preln_fp32=mode == "fp32_preln")
    rng = np.random.default_rng(7)
    x = rng.standard_normal((n, L)).astype(np.float32)
    T, V = cfg.num_frames(L), cfg.vocab_size
    with torch.no_grad():
        ref_logits = model(torch.from_numpy(x)).logits
    ys = _transcripts(rng, ref_logits[0].numpy(), T, V)
    xt = torch.from_numpy(x).cuda()
    eng.set_targets("logits")
    own = eng.eval_waveforms(xt).view(n, T, V).cpu()
    eng.set_transcripts(ys)
    assert eng.out_width(L) == len(ys)
    out = eng.eval_waveforms(xt).cpu().numpy()
    assert np.all(np.isfinite(out))
    # (a) the float64 CTC of the engine's own logits: the kernel tolerance
    ea = np.abs(out - ctc_ref.ctc_logp(own, ys, 0).numpy()) / np.maximum(1.0, np.abs(ctc_ref.ctc_logp(own, ys, 0).numpy()))
    # (b) the HF loss of the fp32 model: 2 T' LOGIT_TOL max |z|
    ref = hf_logp(model, x, ys)
    tol_b = 2 * T * LOGIT_TOL * float(ref_logits.abs().max())
    eb = np.abs(out - ref).max()
    print(f"{name} {mode}: (a) max rel {ea.max():.2e}; (b) max |d log p| {eb:.3e} (tolerance {tol_b:.3g}); "
          f"log p range [{ref.min():.4g}, {ref.max():.4g}]; U = {[len(y) for y in ys]}")
    assert ea.max() <= LOGP_TOL
    assert eb <= tol_b
    eng.close()


def test_transcript_outputs_are_bit_reproducible(P):
    model, cfg = _model("tiny_group")
    L = 9000
    x = torch.from_numpy(np.random.default_rng(1).standard_normal((37, L)).astype(np.float32)).cuda()
    T = cfg.num_frames(L)
    ys = [[5, 6, 6, 7, 8], make_transcript(np.random.default_rng(2), T, T // 2, cfg.vocab_size, 0, 5), []]
    outs = []
    for mb in (7, 32, 0):
        eng = P.Engine(model, cfg, max_batch=mb)
        eng.set_transcripts(ys)
        a = eng.eval_waveforms(x).clone()
        b = eng.eval_waveforms(x).clone()               # repeated call
        alone = eng.eval_waveforms(x[11:12].contiguous())   # one row alone
        torch.cuda.synchronize()
        assert torch.equal(a, b) and torch.equal(alone[0], a[11])
        outs.append(a.cpu())
        eng.close()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def test_background_transcript_mean_equals_materialised_rows(P):
    model, cfg = _model("tiny_group")
    L, M = 12000, 10
    eng = P.Engine(model, cfg, max_batch=16)
    clip = P.synthetic_clip(L)
    eng.set_clip(clip, num_segments=M)
    eng.set_targets("logits")
    lg = eng.eval_bits(eng.bits_to_device(np.ones((1, M), np.uint8))).view(-1, cfg.vocab_size).cpu().numpy()
    ys = [greedy_transcript(lg).tolist(), [5, 6, 6, 7]]
    eng.set_transcripts(ys)
    Z, _, _ = P.sample_coalitions(M, 30, seed=0)
    bits = eng.bits_to_device(Z)
    B = 3
    bg = P.make_background(L, B, seed=5)
    bounds = CB.segment_bounds(L, M)
    per_row = []
    for b in range(B):
        eng.set_background(bg[b:b + 1])
        fused = eng.eval_bits(bits).clone()
        explicit = eng.eval_waveforms(torch.from_numpy(BR.materialize_background(clip, Z, bounds, bg[b:b + 1])).cuda())
        torch.cuda.synchronize()
        assert torch.equal(fused, explicit)
        per_row.append(explicit.cpu().numpy())
    w = np.array([0.5, 2.0, 1.0])
    eng.set_background(bg, w)
    y = eng.eval_bits(bits).cpu().numpy()
    rows = np.stack(per_row, axis=1).reshape(-1, y.shape[1])
    assert np.array_equal(y, host_bg_mean(rows, (w / w.sum()).astype(np.float32), B))
    eng.close()


def test_full_enumeration_transcript_kernelshap_equals_brute_force(P):
    cfg = VARIANTS["tiny_group"]
    model = build_model(cfg)
    sd, d = W.state_dict_of(model), cfg.to_dict()
    L, M = 12000, 10
    clip = P.synthetic_clip(L)
    eng = P.Engine(model, cfg, max_batch=64)
    res = P.KernelShapExplainer(eng, nsamples=2 ** M, seed=0).explain(clip, num_segments=M, mode="transcript")
    assert res["Z"].shape[0] == 2 ** M - 2 and int(res["status"].item()) == 0
    ys = res["transcripts"]
    assert len(ys) == 1
    bounds = CB.segment_bounds(L, M)
    f = lambda Zm: ctc_ref.evaluate_coalitions(sd, d, clip, np.atleast_2d(Zm), bounds, transcripts=ys, blank=0, batch=64)
    exact = brute_force_shapley(f, M)
    phi = res["phi"].cpu().numpy()
    err = np.abs(phi - exact).max() / np.abs(exact).max()
    fx, fnull = res["fx"].cpu().numpy(), res["fnull"].cpu().numpy()
    print(f"transcript KernelSHAP, full enumeration M={M}, U={len(ys[0])}: max rel err vs brute force {err:.3e}")
    assert err < 2e-2
    assert np.abs(phi.sum(0) - (fx - fnull)).max() <= 1e-6 * max(1.0, np.abs(fx - fnull).max())
    eng.close()


def test_transcript_errors_are_raised_before_launch(P):
    model, cfg = _model("tiny_group")
    eng = P.Engine(model, cfg, max_batch=8)
    L = 9000
    T = cfg.num_frames(L)
    x = torch.from_numpy(np.random.default_rng(0).standard_normal((2, L)).astype(np.float32)).cuda()
    eng.set_transcripts([[5, 6]])
    eng.eval_waveforms(x)
    launches = eng.launch_count()
    long_y = [5, 5] * T                                  # needs 4T - 1 frames
    eng.set_transcripts([[5], long_y])
    with pytest.raises(RuntimeError, match=f"transcript 1 needs {frames_needed(long_y)} frames, the clip has {T}"):
        eng.eval_waveforms(x)
    with pytest.raises(RuntimeError, match="transcript 1 needs"):
        eng.grad_transcripts(x, [1, 0])
    eng.set_transcripts([[5], [6, 7]])
    with pytest.raises(RuntimeError, match="transcript index 2"):
        eng.grad_transcripts(x, [0, 2])
    eng.grad_rules(rescale_silu=True)
    with pytest.raises(RuntimeError, match="DeepLIFT"):
        eng.grad_transcripts(x, [0, 1])
    eng.grad_rules()
    # w2s_set_targets still refuses the CTC mode, and the library checks its own arguments
    lib, h = eng.lib, eng._h
    assert lib.w2s_set_targets(h, None, None, 0, 5, eng._stream()) != 0
    lab = np.array([5, 0], np.int32)
    off = np.array([0, 2], np.int32)
    P32 = C.POINTER(C.c_int32)
    assert lib.w2s_set_transcripts(h, lab.ctypes.data_as(P32), off.ctypes.data_as(P32), 1, 0, eng._stream()) != 0
    assert b"blank" in lib.w2s_last_error(h)
    assert eng.launch_count() == launches
    eng.close()
    # a fresh handle without transcripts
    eng = P.Engine(model, cfg, max_batch=8)
    with pytest.raises(RuntimeError, match="no transcripts set"):
        eng.grad_transcripts(x, [0, 0])
    assert eng.launch_count() == 0
    eng.close()


def test_wavlm_gradients_are_refused(P):
    model, cfg = _model("tiny_wavlm")
    eng = P.Engine(model, cfg, max_batch=4)
    eng.set_transcripts([[5, 6]])
    x = torch.zeros((1, 9000), device="cuda")
    with pytest.raises(RuntimeError, match="WavLM"):
        eng.grad_transcripts(x, [0])
    assert eng.launch_count() == 0
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# gradients
# ---------------------------------------------------------------------------------------------------------------------
def autograd_logp(model, x, ys, which):
    """d (-loss) / d input_values of the HF model, reduction "sum", per row with its own transcript."""
    model.config.ctc_loss_reduction = "sum"
    model.config.ctc_zero_infinity = False
    g = np.zeros_like(x)
    out = np.zeros(len(x))
    for r in range(len(x)):
        xt = torch.tensor(x[r:r + 1], requires_grad=True)
        y = ys[which[r]]
        lab = torch.as_tensor(y, dtype=torch.long)[None]
        loss = model(xt, labels=lab).loss
        (-loss).backward()
        g[r] = xt.grad[0].numpy()
        out[r] = -float(loss)
    return g, out


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def cosine(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30))


@pytest.mark.parametrize("name,n,L", [("tiny_group", 5, 9000), ("tiny_layer_stable", 4, 9000),
                                      ("tiny_conformer_rel", 4, 9000), ("tiny_conformer_rotary", 4, 9000),
                                      ("wav2vec2-base", 2, 183600)])
def test_grad_transcripts_match_autograd_of_the_hf_loss(P, name, n, L):
    model, cfg = _model(name)
    rng = np.random.default_rng(n)
    x = rng.standard_normal((n, L)).astype(np.float32)
    T, V = cfg.num_frames(L), cfg.vocab_size
    with torch.no_grad():
        lg = model(torch.from_numpy(x[:1])).logits[0].numpy()
    ys = [greedy_transcript(lg).tolist() or [5], make_transcript(rng, T, min(T // 3, 60), V, 0, 6)]
    which = [r % 2 for r in range(n)]
    gx, out_ref = autograd_logp(model, x, ys, which)
    eng = P.Engine(model, cfg, max_batch=4)
    eng.set_transcripts(ys)
    grad, val = eng.grad_transcripts(torch.from_numpy(x).cuda(), which)
    grad, val = grad.cpu().numpy(), val.cpu().numpy()
    e, c = rel(grad, gx), cosine(grad, gx)
    per_row = [cosine(grad[i], gx[i]) for i in range(n)]
    with torch.no_grad():
        zmax = float(model(torch.from_numpy(x)).logits.abs().max())
    tol_b = 2 * T * LOGIT_TOL * zmax
    print(f"{name} n={n} L={L} T'={T}: transcript input-gradient max rel err {e:.3e}; cosine {c:.5f}; worst row cosine "
          f"{min(per_row):.5f}; max |d log p| {np.abs(val - out_ref).max():.3e} (tolerance {tol_b:.3g})")
    assert np.all(np.isfinite(grad)) and np.all(np.isfinite(val))
    assert np.abs(val - out_ref).max() <= tol_b
    assert e < GRAD_TOL and min(per_row) > 0.995
    eng.close()


def test_expected_gradients_on_transcripts_match_the_autograd_estimator(P):
    cfg = VARIANTS["tiny_group"]
    model = build_model(cfg)
    L = 4000
    x = P.synthetic_clip(L)
    bg = P.make_background(L, 5, seed=1)
    eng = P.Engine(model, cfg, max_batch=8)
    T = cfg.num_frames(L)
    ys = [[5, 6, 6], make_transcript(np.random.default_rng(0), T, T // 3, cfg.vocab_size, 0, 5)]
    ex = P.ExpectedGradientsExplainer(eng, bg, nsamples=64, seed=3, batch=32)
    phi = ex.shap_values(x, transcripts=ys)
    assert phi.shape == (1, L, 2)
    with pytest.raises(ValueError, match="mutually exclusive"):
        ex.shap_values(x, frames=[0], transcripts=ys)
    ref = np.zeros((L, 2))
    for d in range(2):
        rng = np.random.default_rng([3, d])
        rind = rng.integers(0, 5, 64)
        alpha = rng.uniform(size=64).astype(np.float32)
        xs = (bg[rind] + alpha[:, None] * (x[None] - bg[rind])).astype(np.float32)
        gx, _ = autograd_logp(model, xs, ys, [d] * 64)
        ref[:, d] = (gx.astype(np.float64) * (x[None] - bg[rind])).mean(0)
    e, c = rel(phi[0], ref), cosine(phi[0], ref)
    print(f"expected gradients on transcripts (64 samples, 2 outputs): max rel err vs autograd estimator {e:.3e}; "
          f"cosine {c:.5f}")
    assert c > 0.98 and e < 0.25
    eng.close()


def test_grad_transcripts_without_out_and_its_launch_count(P):
    """out may be NULL (as for w2s_grad_waveforms); the CTC seed step launches two kernels and is counted as two."""
    model, cfg = _model("tiny_group")
    eng = P.Engine(model, cfg, max_batch=4)
    L = 9000
    x = torch.from_numpy(np.random.default_rng(4).standard_normal((3, L)).astype(np.float32)).cuda()
    eng.set_transcripts([[5, 6, 6], [7]])
    which = np.array([0, 1, 0], np.int32)
    n0 = eng.launch_count()
    g_ref, _ = eng.grad_transcripts(x, which)
    n1 = eng.launch_count()
    eng.grad_waveforms(x, [0, 1, 2])
    n2 = eng.launch_count()
    assert n1 - n0 == (n2 - n1) + 1            # one tile: the same steps, one more kernel in head_bwd
    g = torch.empty_like(g_ref)
    rc = eng.lib.w2s_grad_transcripts(eng._h, x.data_ptr(), 3, L, L, which.ctypes.data_as(C.POINTER(C.c_int32)),
                                      g.data_ptr(), None, eng._stream())
    assert rc == 0, eng.lib.w2s_last_error(eng._h)
    torch.cuda.synchronize()
    assert torch.equal(g, g_ref)
    eng.close()
