"""GPU: WavLM's gated relative-position bias inside the attention kernels (w2s_debug_attention_bias), against a float64
reference computed on exactly the bf16 q / k / v and the fp32 table and gate handed to them -- the tcgen05 kernel's
one-block, two-block and streaming variants and the CUDA-core validation kernel.

  score[b, h, i, j] = scale q_i . k_j + gate[b, h, i] * E[bucket(j - i), h]

Input families, each magnifying one failure mode:
  typical    q, k, v ~ N(0, 1), E ~ N(0, 1) through the model's buckets (saturated from |j - i| = 778 on), gates in (1, 3)
  biasonly   q, k nearly 0, the table peaks at j - i = +3 with a gap of 16 and the gates vary in (0.8, 1.2): the gated
             bias alone selects key min(i + 3, T' - 1), a check of the index and of the gate's row that needs no formula
  padding    every valid key scores about -100 (scaled) plus the bias, v is offset from 0: a zero-filled padding key whose
             score was not masked after the bias add would take all the weight
  gates      extreme gates per (b, h, i) from {-3, 0, 5, 20}: negative, vanishing and large multipliers of the table
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

SCALE = 0.125
DEV = "cuda"
FWD_TOL = 1.5e-2      # tests/test_gpu_attention.py
SIMT_MAX_T = 1024

# T' -> (heads, B): one block (1, 77, 128), two blocks (129, 256), streaming (257, 713, 801, 1031); 713 is the bucket
# boundary with the thinnest float margin, 801 and 1031 reach the saturated buckets
SHAPES = {1: (12, 3), 77: (2, 5), 128: (12, 3), 129: (2, 37), 256: (16, 3), 257: (2, 33), 713: (12, 2), 801: (2, 3),
          1031: (16, 2)}
FAMILIES = ["typical", "biasonly", "padding", "gates"]


@pytest.fixture(scope="module")
def P():
    import shap_transformer_asr_b200 as pkg
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return pkg


class Inputs:
    """bf16 q, k, v [B, heads, T, 64], the natural-units table [heads, 2T - 1] (entry r <-> j - i = r - (T - 1)) and the
    gate [B, heads, T] (fp32), with float64 copies."""

    def __init__(self, P, family, T, B, heads, seed):
        g = torch.Generator(device=DEV).manual_seed(seed)
        f64 = torch.float64

        def randn(*shape):
            return torch.randn(*shape, generator=g, device=DEV, dtype=f64)

        def rand(*shape):
            return torch.rand(*shape, generator=g, device=DEV, dtype=f64)

        self.T, self.B, self.heads, self.H = T, B, heads, 64 * heads
        q, k, v = randn(B, heads, T, 64), randn(B, heads, T, 64), randn(B, heads, T, 64)
        bucket = torch.from_numpy(P.relative_buckets(T)).to(DEV).long()
        table = randn(320, heads)[bucket].t().contiguous()                     # [heads, 2T - 1]
        gate = 1.0 + 2.0 * rand(B, heads, T)
        d = torch.arange(2 * T - 1, device=DEV, dtype=f64) - (T - 1)
        if family == "biasonly":
            q, k = 0.1 * q, 0.1 * k
            table = (-16.0 * (d - 3).abs().clamp(max=8.0))[None].repeat(heads, 1) + 0.05 * randn(heads, 2 * T - 1)
            gate = 0.8 + 0.4 * rand(B, heads, T)
        elif family == "padding":
            u = randn(heads, 64)
            u = (u / u.norm(dim=-1, keepdim=True))[None, :, None]
            q = 100.0 / SCALE * u + 0.3 * randn(B, heads, T, 64)
            k = -u + 0.3 * randn(B, heads, T, 64) * 0.1
            v = 0.75 + randn(B, heads, T, 64)
        elif family == "gates":
            gate = torch.tensor([-3.0, 0.0, 5.0, 20.0], device=DEV, dtype=f64)[torch.randint(0, 4, (B, heads, T), generator=g, device=DEV)]
        self.q16, self.k16, self.v16 = q.bfloat16(), k.bfloat16(), v.bfloat16()
        self.table32, self.gate32 = table.float().contiguous(), gate.float().contiguous()
        self.q, self.k, self.v = (t.double() for t in (self.q16, self.k16, self.v16))
        self.table, self.gate = self.table32.double(), self.gate32.double()

    @staticmethod
    def rows(t):
        B, h, T, d = t.shape
        return t.permute(0, 2, 1, 3).reshape(B * T, h * d)

    def qkv(self):
        return torch.cat([self.rows(t) for t in (self.q16, self.k16, self.v16)], 1).contiguous()

    def split(self, ctx):
        return ctx.double().view(self.B, self.T, self.heads, 64).permute(0, 2, 1, 3)

    def reference(self):
        T = self.T
        idx = (T - 1) + torch.arange(T, device=DEV)[None, :] - torch.arange(T, device=DEV)[:, None]     # [i, j]
        bias = self.table[:, idx]                                                                       # [heads, T, T]
        s = self.q @ self.k.transpose(-1, -2) * SCALE + self.gate[..., None] * bias[None]
        return torch.softmax(s, -1) @ self.v


def err(a, ref):
    return (a - ref).abs().max().item() / (ref.abs().max().item() + 1e-30)


def run(P, x, tc, ctx=None):
    return P.debug_attention_bias(x.qkv(), x.B, x.heads, x.table32, x.gate32, scale=SCALE, tcgen05=tc, ctx=ctx)


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("T", list(SHAPES))
def test_bias_attention_matches_fp64(P, T, family):
    if family == "padding" and T % 128 == 0:
        pytest.skip("padding needs a ragged last key block")
    heads, B = SHAPES[T]
    x = Inputs(P, family, T, B, heads, seed=T * 10 + FAMILIES.index(family))
    o_ref = x.reference()
    report, fails = [], []
    for name, tc in [("tcgen05", True)] + ([("cuda_core", False)] if T <= SIMT_MAX_T else []):
        o = x.split(run(P, x, tc))
        torch.cuda.synchronize()
        e = err(o, o_ref)
        report.append(f"{name} {e:.2e}")
        if not e < FWD_TOL:
            fails.append((name, e))
        if family == "biasonly":
            j = torch.clamp(torch.arange(T, device=DEV) + 3, max=T - 1)
            e3 = err(o, x.v[:, :, j])
            report.append(f"{name} v[i+3] {e3:.2e}")
            if not e3 < FWD_TOL:
                fails.append((name, "v[i+3]", e3))
    print(f"bias attention T'={T} heads={heads} B={B} {family}: " + "; ".join(report))
    assert not fails, fails


def test_bias_attention_is_batch_independent_and_repeatable(P):
    T, (heads, B) = 713, SHAPES[713]
    x = Inputs(P, "typical", T, B, heads, seed=1)
    qkv = x.qkv()
    for tc in (True, False):
        c1 = P.debug_attention_bias(qkv, B, heads, x.table32, x.gate32, scale=SCALE, tcgen05=tc)
        c2 = P.debug_attention_bias(qkv, B, heads, x.table32, x.gate32, scale=SCALE, tcgen05=tc)
        assert torch.equal(c1, c2), tc
        for b in range(B):
            rows = slice(b * T, (b + 1) * T)
            one = P.debug_attention_bias(qkv[rows].contiguous(), 1, heads, x.table32, x.gate32[b:b + 1].contiguous(),
                                         scale=SCALE, tcgen05=tc)
            assert torch.equal(one, c1[rows]), (tc, b)


@pytest.mark.parametrize("T", [300, 1031])
def test_bias_attention_writes_every_row_and_nothing_else(P, T):
    heads, B = (16, 4) if T == 300 else SHAPES[T]
    x = Inputs(P, "typical", T, B, heads, seed=2)
    n, G = B * T * 64 * heads, 4096
    for tc in (True, False):
        if not tc and T > SIMT_MAX_T:
            continue
        buf = torch.full((n + G,), float("nan"), dtype=torch.bfloat16, device=DEV)
        run(P, x, tc, ctx=buf)
        torch.cuda.synchronize()
        assert torch.isfinite(buf[:n]).all() and torch.isnan(buf[n:]).all(), tc


def test_bias_attention_refuses_the_log_sum_exp(P):
    x = Inputs(P, "typical", 129, 1, 2, seed=3)
    lse = torch.empty(2 * 129, dtype=torch.float32, device=DEV)
    for tc in (True, False):
        with pytest.raises(RuntimeError, match="log-sum-exp"):
            P.debug_attention_bias(x.qkv(), 1, 2, x.table32, x.gate32, scale=SCALE, tcgen05=tc, lse=lse)


def test_cuda_core_bias_kernel_keeps_its_frame_limit(P):
    x = Inputs(P, "typical", 1025, 1, 2, seed=4)
    with pytest.raises(RuntimeError, match="1024"):
        run(P, x, False)
