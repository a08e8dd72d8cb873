"""GPU: the attention kernels on their own (w2s_debug_attention / w2s_debug_attention_bwd) against float64 references
computed on exactly the bf16 values handed to them -- the tcgen05 forward (attention_fa: its one-block, two-block and
streaming variants, and the log-sum-exp it saves for the backward), the relative-position forward (attention_rel), the
fused tcgen05 backward, and the CUDA-core kernels the model tests use as cross-checks.

Model-level tests dilute an attention error past detection (one zero-filled padding key let into a near-uniform softmax
at T' = 573 moves the output by 0.17 %), so each input family here magnifies one failure mode instead:
  typical   q, k, v ~ N(0, 1)
  sharp     a nearly one-hot softmax whose argmax key sits in the first block, a middle block, the last block and at the
            last valid key: checks which value row is paired with which key
  padding   every valid key scores about -100 after scaling and v is offset from 0: a zero-filled padding key (score 0)
            would take all the weight, and in the backward its exp2(-LSE) overflows, so dQ turns NaN
  blockmax  one head-dim column biases whole 128-key blocks by -30 / -60 / -100 around one peak block (the first, a middle
            or the last one, per (row, head)): exercises the merge factors of independent key blocks and their underflow
  relonly   (relative positions) the position term dominates and peaks at offset +3: ctx[i] = v[min(i + 3, T' - 1)],
            a check of the shift that does not depend on any fp64 formula

Errors are max |kernel - reference| over max |reference| of the same tensor (the log-sum-exp: max abs error in log2
units).  Measured maxima over all frame counts and families on one B200 are in each test's docstring; the tolerances
leave 3-4x headroom.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

SCALE = 0.125   # 1 / sqrt(head_dim 64), as the models use
DEV = "cuda"

# T' -> (heads, B).  Work items of the persistent kernels = B * heads * ceil(T' / 128): below the 148 SMs, exactly 148
# (T' = 127, 129), and above with a remainder (T' = 257, 300, 385, 573, 1031), so CTAs run several items -- with an odd
# number of key blocks the softmax-group ownership carries over from one item to the next.
SHAPES = {1: (12, 3), 2: (2, 5), 33: (16, 2), 127: (2, 74), 128: (12, 3), 129: (2, 37), 255: (12, 2), 256: (16, 3),
          257: (2, 33), 300: (16, 4), 384: (12, 2), 385: (2, 19), 573: (12, 3), 1031: (16, 2)}
FAMILIES = ["typical", "sharp", "padding", "blockmax"]
SIMT_MAX_T = 1024

FWD_TOL = 1.5e-2      # measured <= 4.4e-3 (every kernel)
LSE_TOL = 1e-4        # measured <= 3.2e-5 (log2 units)
# the fused backward rounds P and dS to bf16 and takes D = dO . O from the bf16 forward output; the CUDA-core kernels keep
# P and dS in fp32
GRAD_TOL = {"fused": 5e-2, "cuda_core": 1.2e-2}    # measured <= 1.6e-2 / 3.6e-3
COS_MIN = 0.998       # measured >= 0.9995


@pytest.fixture(scope="module")
def P():
    import shap_transformer_asr_b200 as pkg
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return pkg


def applicable(family, T):
    if family == "padding":
        return T % 128 != 0          # needs padding keys in the last block
    if family == "blockmax":
        return T > 128               # needs two key blocks or more
    return True


class Inputs:
    """bf16 operands of one attention call and their float64 copies ([B, heads, T, 64]; pp: [heads, 2T - 1, 64])."""

    def __init__(self, family, T, B, heads, seed):
        g = torch.Generator(device=DEV).manual_seed(seed)
        dev, f64 = DEV, torch.float64

        def randn(*shape):
            return torch.randn(*shape, generator=g, device=dev, dtype=f64)

        self.T, self.B, self.heads, self.H = T, B, heads, 64 * heads
        q, k, v = randn(B, heads, T, 64), randn(B, heads, T, 64), randn(B, heads, T, 64)
        qv, pp = 0.3 * randn(B, heads, T, 64), 0.3 * randn(heads, 2 * T - 1, 64)
        nb = (T + 127) // 128
        if family == "sharp":
            khat = k / k.norm(dim=-1, keepdim=True)
            k = 8.0 * khat
            targets = torch.tensor(sorted({min(5, T - 1), min((nb // 2) * 128 + 17, T - 1), (nb - 1) * 128, T - 1}),
                                   device=dev)
            q = 64.0 * khat[:, :, targets[torch.arange(T, device=dev) % len(targets)]]   # scaled score 64 vs <= ~26
        elif family == "padding":
            # q . k = -800 (scaled: -100) from q = 800 u, k = -u + noise: the large component sits in q, so dQ = scale dS K
            # does not cancel a large common component of K (which the fused kernel's bf16 dS would not reproduce)
            u = randn(heads, 64)
            u = (u / u.norm(dim=-1, keepdim=True))[None, :, None]
            kn = 0.3 * randn(B, heads, T, 64)
            kn = kn - (kn * u).sum(-1, keepdim=True) * u
            q = 100.0 / SCALE * u + 0.3 * randn(B, heads, T, 64)
            k = -u + kn + 0.01 * randn(B, heads, T, 1) * u      # scaled scores -100 +- 1
            v = 0.75 + randn(B, heads, T, 64)   # outputs near 0.75: a collapse to 0 shows; bf16 O keeps 2^-8 steps
        elif family == "blockmax":
            q, k = 0.5 * q, 0.5 * k
            cyc = torch.tensor([-30.0, -60.0, -100.0], device=dev, dtype=f64)
            blk = torch.arange(T, device=dev) // 128
            peak = torch.tensor([0, nb // 2, nb - 1], device=dev)[torch.arange(B * heads, device=dev) % 3].view(B, heads, 1)
            bias = torch.where(blk == peak, 0.0, cyc[blk % 3])          # [B, heads, T]: scaled score offset of each key
            q[..., 63] = 8.0
            k[..., 63] = bias / (8.0 * SCALE)
        elif family == "relonly":
            q, k = 0.1 * q, 0.1 * k
            qv = 0.05 * qv
            qv[..., 0] = 16.0
            r = torch.arange(2 * T - 1, device=dev, dtype=f64)
            pp = 0.05 * pp
            pp[:, :, 0] = -16.0 * (r - (T + 2)).abs().clamp(max=8.0)   # row T-1-i+j peaks at j = i + 3: gap 32 (scaled)
        b16 = lambda t: t.bfloat16()
        self.q16, self.k16, self.v16, self.qv16, self.pp16 = b16(q), b16(k), b16(v), b16(qv), b16(pp)
        self.q, self.k, self.v, self.qv, self.pp = (t.double() for t in (self.q16, self.k16, self.v16, self.qv16, self.pp16))

    @staticmethod
    def rows(t):     # [B, heads, T, 64] -> [B*T, heads*64]
        B, h, T, d = t.shape
        return t.permute(0, 2, 1, 3).reshape(B * T, h * d)

    def qkv(self, rel=False):
        parts = [self.q16, self.qv16, self.k16, self.v16] if rel else [self.q16, self.k16, self.v16]
        return torch.cat([self.rows(t) for t in parts], 1).contiguous()

    def pos_proj(self):
        return self.pp16.permute(1, 0, 2).reshape(2 * self.T - 1, self.H).contiguous()

    def split(self, qkv_rows, n):   # [B*T, n*H] -> n tensors [B, heads, T, 64] (float64)
        t = qkv_rows.double().view(self.B, self.T, n, self.heads, 64)
        return [t[:, :, i].permute(0, 2, 1, 3) for i in range(n)]


def hf_rel_shift(bd):
    """The shift trick of transformers' Wav2Vec2ConformerSelfAttention._apply_relative_embeddings
    (modeling_wav2vec2_conformer.py:553-559): [.., T, 2T-1] scores over relative positions -> [.., T, T]."""
    zero_pad = torch.zeros((*bd.size()[:3], 1), device=bd.device, dtype=bd.dtype)
    padded = torch.cat([zero_pad, bd], dim=-1)
    padded = padded.view(*bd.size()[:2], bd.shape[3] + 1, bd.shape[2])
    return padded[:, :, 1:].view_as(bd)[:, :, :, : bd.size(-1) // 2 + 1]


def reference(x, rel=False, dout=None):
    """float64: ctx = softmax(scale (Q K^T [+ shift((Q+v) PP^T)])) V, LSE = logsumexp(scores) / ln 2; with `dout`
    ([B, heads, T, 64]) also dQ, dK, dV by autograd."""
    q, k, v = (t.clone().requires_grad_(dout is not None) for t in (x.q, x.k, x.v))
    s = q @ k.transpose(-1, -2)
    if rel:
        s = s + hf_rel_shift(x.qv @ x.pp.transpose(-1, -2)[None])
    s = s * SCALE
    o = torch.softmax(s, -1) @ v
    lse = torch.logsumexp(s, -1) / math.log(2.0)
    if dout is None:
        return o.detach(), lse.detach()
    (o * dout).sum().backward()
    return o.detach(), lse.detach(), q.grad, k.grad, v.grad


def err(a, ref, denom=None):
    d = (a.double() - ref).abs().max().item()
    return d / (denom if denom is not None else ref.abs().max().item() + 1e-30)


def min_cosine(a, ref):
    """Smallest cosine similarity over the (row, head) pairs, skipping pairs whose reference all but vanishes (a one-hot
    softmax: the peak in a one-key last block) -- there both sides are rounding noise."""
    a, ref = a.double().flatten(2), ref.flatten(2)
    norms = ref.norm(dim=-1)
    keep = norms > 1e-2 * norms.max()
    return torch.nn.functional.cosine_similarity(a, ref, dim=-1)[keep].min().item()


@pytest.mark.parametrize("family", FAMILIES + ["relonly"])
@pytest.mark.parametrize("T", list(SHAPES))
def test_forward_kernels_match_fp64(P, T, family):
    """attention_fa (ctx and LSE), attention_rel and the CUDA-core validation kernel (with and without relative positions)
    against the float64 reference.  Measured on a B200 (1000 W) over all T' and families: ctx <= 4.4e-3 of its maximum
    (attention_fa 4.4e-3, attention_rel 4.2e-3, CUDA core 3.8e-3), LSE <= 3.2e-5 (log2 units); relonly gives v[i + 3]
    exactly."""
    if family == "relonly":
        rel_modes = [True]
    elif not applicable(family, T):
        pytest.skip(f"{family} needs {'a ragged last block' if family == 'padding' else 'two key blocks'}")
    else:
        rel_modes = [False, True]
    heads, B = SHAPES[T]
    x = Inputs(family, T, B, heads, seed=T * 10 + FAMILIES.index(family) if family in FAMILIES else T * 10 + 7)
    report, fails = [], []
    for rel in rel_modes:
        o_ref, lse_ref = reference(x, rel)
        qkv = x.qkv(rel)
        pp = x.pos_proj() if rel else None
        kernels = [("tcgen05", True)] + ([("cuda_core", False)] if T <= SIMT_MAX_T else [])
        for name, tc in kernels:
            kname = ("attention_rel" if tc else "simt_rel") if rel else ("attention_fa" if tc else "simt")
            ctx, lse = P.debug_attention(qkv, B, heads, pos_proj=pp, scale=SCALE, tcgen05=tc, with_lse=tc and not rel)
            torch.cuda.synchronize()
            (o,) = x.split(ctx, 1)
            e = err(o, o_ref)
            report.append(f"{kname} ctx {e:.2e}")
            if not e < FWD_TOL:
                fails.append((kname, "ctx", e))
            if lse is not None:
                el = (lse.double() - lse_ref).abs().max().item()
                report.append(f"{kname} lse {el:.2e}")
                if not el < LSE_TOL:
                    fails.append((kname, "lse", el))
            if family == "relonly":
                # the position term alone decides: every query attends to key min(i + 3, T' - 1) of its own row and head
                j = torch.clamp(torch.arange(T, device=DEV) + 3, max=T - 1)
                e3 = err(o, x.v[:, :, j])
                report.append(f"{kname} v[i+3] {e3:.2e}")
                if not e3 < FWD_TOL:
                    fails.append((kname, "v[i+3]", e3))
    print(f"forward T'={T} heads={heads} B={B} {family}: " + "; ".join(report))
    assert not fails, fails


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("T", list(SHAPES))
def test_backward_kernels_match_fp64(P, T, family):
    """The fused tcgen05 backward, fed attention_fa's own ctx and LSE as the gradient path does, and the CUDA-core
    cross-check kernels against float64 autograd with the same bf16 dO.  Measured on a B200 (1000 W) over all T' and
    families, as a fraction of each tensor's maximum: fused dQ 1.6e-2 (padding; 6.0e-3 otherwise), dK 7.6e-3, dV 4.7e-3, per-
    (row, head) cosine >= 0.9995; CUDA core <= 3.6e-3, cosine 1.00000."""
    if not applicable(family, T):
        pytest.skip(f"{family} needs {'a ragged last block' if family == 'padding' else 'two key blocks'}")
    heads, B = SHAPES[T]
    x = Inputs(family, T, B, heads, seed=T * 10 + FAMILIES.index(family))
    g = torch.Generator(device=DEV).manual_seed(T + 1)
    dout16 = torch.randn(B, heads, T, 64, generator=g, device=DEV).bfloat16()
    _, _, dq_ref, dk_ref, dv_ref = reference(x, dout=dout16.double())
    refs = {"dq": dq_ref, "dk": dk_ref, "dv": dv_ref}
    qkv, dctx = x.qkv(), Inputs.rows(dout16).contiguous()
    ctx, lse = P.debug_attention(qkv, B, heads, scale=SCALE, with_lse=True)
    report, fails = [], []
    kernels = [("fused", True)] + ([("cuda_core", False)] if T <= SIMT_MAX_T else [])
    for name, tc in kernels:
        dqkv = P.debug_attention_bwd(qkv, dctx, B, heads, ctx=ctx, lse=lse, scale=SCALE, tcgen05=tc)
        torch.cuda.synchronize()
        got = dict(zip(("dq", "dk", "dv"), x.split(dqkv, 3)))
        dv_max = dv_ref.abs().max().item()
        for gname, ref in refs.items():
            # dQ and dK vanish in exact arithmetic when the softmax is one-hot (sharp) or has a single key (T' = 1):
            # measure them against dV's scale then
            tiny = (family == "sharp" and gname != "dv") or ref.abs().max().item() < 1e-3 * dv_max
            e = err(got[gname], ref, dv_max if tiny else None)
            report.append(f"{name} {gname} {e:.2e}")
            if not e < GRAD_TOL[name]:
                fails.append((name, gname, e))
            if not tiny:
                c = min_cosine(got[gname], ref)
                report.append(f"cos {c:.5f}")
                if not c > COS_MIN:
                    fails.append((name, gname, "cosine", c))
    print(f"backward T'={T} heads={heads} B={B} {family}: " + "; ".join(report))
    assert not fails, fails


def test_forward_is_batch_independent_and_repeatable(P):
    """A row's forward output is bit-identical whether it runs alone or inside a batch (and the work items then fall on
    other CTAs), and a repeated call gives the same bits; the fused backward's dK / dV (accumulated in a fixed order inside
    one CTA) repeat bit for bit too."""
    T, (heads, B) = 573, SHAPES[573]
    x = Inputs("typical", T, B, heads, seed=1)
    for rel in (False, True):
        qkv, pp = x.qkv(rel), (x.pos_proj() if rel else None)
        for tc in (True, False):
            want_lse = tc and not rel
            ctx, lse = P.debug_attention(qkv, B, heads, pos_proj=pp, scale=SCALE, tcgen05=tc, with_lse=want_lse)
            ctx2, lse2 = P.debug_attention(qkv, B, heads, pos_proj=pp, scale=SCALE, tcgen05=tc, with_lse=want_lse)
            assert torch.equal(ctx, ctx2) and (lse is None or torch.equal(lse, lse2))
            for b in range(B):
                rows = slice(b * T, (b + 1) * T)
                c1, l1 = P.debug_attention(qkv[rows].contiguous(), 1, heads, pos_proj=pp, scale=SCALE, tcgen05=tc,
                                           with_lse=want_lse)
                assert torch.equal(c1, ctx[rows]), (rel, tc, b)
                assert lse is None or torch.equal(l1[0], lse[b]), (rel, tc, b)
    qkv = x.qkv()
    ctx, lse = P.debug_attention(qkv, B, heads, scale=SCALE, with_lse=True)
    dctx = torch.randn(B * T, 64 * heads, device=DEV).bfloat16()
    d1 = P.debug_attention_bwd(qkv, dctx, B, heads, ctx=ctx, lse=lse, scale=SCALE)
    d2 = P.debug_attention_bwd(qkv, dctx, B, heads, ctx=ctx, lse=lse, scale=SCALE)
    H = 64 * heads
    assert torch.equal(d1[:, H:], d2[:, H:])


@pytest.mark.parametrize("T", [300, 1031])
def test_outputs_cover_every_row_and_nothing_else(P, T):
    """NaN-prefilled outputs with a guard tail: every row < T' of every batch is written (ctx, LSE, dqkv) and nothing past
    the arrays is touched."""
    heads, B = SHAPES[T]
    H, G = 64 * heads, 4096
    x = Inputs("typical", T, B, heads, seed=2)

    def nan_buf(n, dtype):
        return torch.full((n + G,), float("nan"), dtype=dtype, device=DEV)

    for rel in (False, True):
        for tc in (True, False):
            if not tc and T > SIMT_MAX_T:
                continue
            cbuf = nan_buf(B * T * H, torch.bfloat16)
            lbuf = nan_buf(B * heads * T, torch.float32) if tc and not rel else None
            P.debug_attention(x.qkv(rel), B, heads, pos_proj=x.pos_proj() if rel else None, scale=SCALE, tcgen05=tc,
                              ctx=cbuf, lse=lbuf)
            torch.cuda.synchronize()
            assert torch.isfinite(cbuf[:B * T * H]).all() and torch.isnan(cbuf[B * T * H:]).all(), (rel, tc)
            if lbuf is not None:
                assert torch.isfinite(lbuf[:B * heads * T]).all() and torch.isnan(lbuf[B * heads * T:]).all()
    qkv = x.qkv()
    ctx, lse = P.debug_attention(qkv, B, heads, scale=SCALE, with_lse=True)
    dctx = torch.randn(B * T, H, device=DEV).bfloat16()
    for tc in (True, False):
        if not tc and T > SIMT_MAX_T:
            continue
        dbuf = nan_buf(B * T * 3 * H, torch.bfloat16)
        P.debug_attention_bwd(qkv, dctx, B, heads, ctx=ctx, lse=lse, scale=SCALE, tcgen05=tc, dqkv=dbuf)
        torch.cuda.synchronize()
        assert torch.isfinite(dbuf[:B * T * 3 * H]).all() and torch.isnan(dbuf[B * T * 3 * H:]).all(), tc


def test_cuda_core_kernels_at_their_frame_limit(P):
    """The CUDA-core kernels meet the float64 reference at T' = 1024, the most they take, and refuse T' = 1025 with an
    error that names the limit (instead of computing a truncated softmax)."""
    for T in (1024, 1025):
        x = Inputs("typical", T, 1, 2, seed=3)
        qkv = x.qkv()
        dout16 = torch.randn(1, 2, T, 64, device=DEV).bfloat16()
        dctx = Inputs.rows(dout16).contiguous()
        if T > SIMT_MAX_T:
            with pytest.raises(RuntimeError, match="1024"):
                P.debug_attention(qkv, 1, 2, scale=SCALE, tcgen05=False)
            with pytest.raises(RuntimeError, match="1024"):
                P.debug_attention(x.qkv(True), 1, 2, pos_proj=x.pos_proj(), scale=SCALE, tcgen05=False)
            with pytest.raises(RuntimeError, match="1024"):
                P.debug_attention_bwd(qkv, dctx, 1, 2, scale=SCALE, tcgen05=False)
            continue
        o_ref, _, dq, dk, dv = reference(x, dout=dout16.double())
        ctx, _ = P.debug_attention(qkv, 1, 2, scale=SCALE, tcgen05=False)
        assert err(x.split(ctx, 1)[0], o_ref) < FWD_TOL
        o_rel, _ = reference(x, rel=True)
        ctx, _ = P.debug_attention(x.qkv(True), 1, 2, pos_proj=x.pos_proj(), scale=SCALE, tcgen05=False)
        assert err(x.split(ctx, 1)[0], o_rel) < FWD_TOL
        got = x.split(P.debug_attention_bwd(qkv, dctx, 1, 2, scale=SCALE, tcgen05=False), 3)
        for a, ref in zip(got, (dq, dk, dv)):
            assert err(a, ref) < GRAD_TOL["cuda_core"] and min_cosine(a, ref) > COS_MIN
