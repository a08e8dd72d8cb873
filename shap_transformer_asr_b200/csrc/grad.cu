// Backward (input-gradient) kernels of the expected-gradients path -- the reference's production explainer
// (shap.GradientExplainer, shap_calculation.py:125-162; loop structure feasability_tests/conformer_test.ipynb:95).
// Expected gradients need d(output)/d(input) only: no weight gradients.  The dense contractions of the backward pass
// (dX = dY W) run on the same tcgen05 contraction kernels as the forward pass, on pre-transposed weights; this file
// holds what is left: the element-wise / normalisation / softmax backward steps and the data movement around the
// strided convolutions.  First slice: Wav2Vec2 with a group-norm front end and a post-LN encoder (wav2vec2-base /
// -large, the model family the reference runs).
//
// Conventions: activations saved by the forward pass are bf16 unless stated; gradients between contractions are bf16
// (they feed a tensor-core A operand), gradients that are accumulated across a residual branch are fp32.
#include "kernels.cuh"
#include "ctc.cuh"

namespace w2s {

// exact-erf GELU and its derivative (HF ACT2FN["gelu"]): gelu'(u) = Phi(u) + u phi(u)
__device__ __forceinline__ float gelu_grad(float u) {
  const float cdf = 0.5f * (1.0f + erff(u * 0.70710678118654752f));
  const float pdf = 0.39894228040143268f * __expf(-0.5f * u * u);
  return fmaf(u, pdf, cdf);
}

// y = gelu(u)   (the forward pass of the gradient path stores the pre-activation u and applies GELU separately)
__global__ void __launch_bounds__(256) gelu_fwd_kernel(const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ y,
                                                        long long n8) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 a = reinterpret_cast<const uint4*>(u)[i];
    uint4 o;
    o.x = pack_bf16x2(gelu_erf(bf16_lo(a.x)), gelu_erf(bf16_hi(a.x)));
    o.y = pack_bf16x2(gelu_erf(bf16_lo(a.y)), gelu_erf(bf16_hi(a.y)));
    o.z = pack_bf16x2(gelu_erf(bf16_lo(a.z)), gelu_erf(bf16_hi(a.z)));
    o.w = pack_bf16x2(gelu_erf(bf16_lo(a.w)), gelu_erf(bf16_hi(a.w)));
    reinterpret_cast<uint4*>(y)[i] = o;
  }
}
std::string launch_gelu_fwd(const __nv_bfloat16* u, __nv_bfloat16* y, long long n, cudaStream_t s) {
  if (n % 8) return "gelu_fwd: element count must be a multiple of 8";
  if (n == 0) return "";
  const long long n8 = n / 8;
  gelu_fwd_kernel<<<(unsigned)((n8 + 255) / 256 > 148 * 16 ? 148 * 16 : (n8 + 255) / 256), 256, 0, s>>>(u, y, n8);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// d <- d * gelu'(u)
__global__ void __launch_bounds__(256) gelu_bwd_kernel(const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ d,
                                                        long long n8) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 a = reinterpret_cast<const uint4*>(u)[i];
    const uint4 g = reinterpret_cast<const uint4*>(d)[i];
    uint4 o;
    o.x = pack_bf16x2(bf16_lo(g.x) * gelu_grad(bf16_lo(a.x)), bf16_hi(g.x) * gelu_grad(bf16_hi(a.x)));
    o.y = pack_bf16x2(bf16_lo(g.y) * gelu_grad(bf16_lo(a.y)), bf16_hi(g.y) * gelu_grad(bf16_hi(a.y)));
    o.z = pack_bf16x2(bf16_lo(g.z) * gelu_grad(bf16_lo(a.z)), bf16_hi(g.z) * gelu_grad(bf16_hi(a.z)));
    o.w = pack_bf16x2(bf16_lo(g.w) * gelu_grad(bf16_lo(a.w)), bf16_hi(g.w) * gelu_grad(bf16_hi(a.w)));
    reinterpret_cast<uint4*>(d)[i] = o;
  }
}
std::string launch_gelu_bwd(const __nv_bfloat16* u, __nv_bfloat16* d, long long n, cudaStream_t s) {
  if (n % 8) return "gelu_bwd: element count must be a multiple of 8";
  if (n == 0) return "";
  const long long n8 = n / 8;
  gelu_bwd_kernel<<<(unsigned)((n8 + 255) / 256 > 148 * 16 ? 148 * 16 : (n8 + 255) / 256), 256, 0, s>>>(u, d, n8);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// pre0 = h0 + gelu(upos)   (positional-conv branch + residual of the gradient-path forward, fp32 out)
__global__ void __launch_bounds__(256) add_gelu_kernel(const __nv_bfloat16* __restrict__ h0, const __nv_bfloat16* __restrict__ up,
                                                        float* __restrict__ out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = __bfloat162float(h0[i]) + gelu_erf(__bfloat162float(up[i]));
}
std::string launch_add_gelu(const __nv_bfloat16* h0, const __nv_bfloat16* up, float* out, long long n, cudaStream_t s) {
  if (n == 0) return "";
  add_gelu_kernel<<<(unsigned)((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256), 256, 0, s>>>(h0, up, out, n);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// fp32 -> bf16 copy of a gradient (A operand of the next contraction), optionally scaled element-wise by gelu'(u)
__global__ void __launch_bounds__(256) grad_cast_kernel(const float* __restrict__ g, const __nv_bfloat16* __restrict__ u,
                                                         __nv_bfloat16* __restrict__ out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float v = g[i];
    if (u) v *= gelu_grad(__bfloat162float(u[i]));
    out[i] = __float2bfloat16_rn(v);
  }
}
std::string launch_grad_cast(const float* g, const __nv_bfloat16* u, __nv_bfloat16* out, long long n, cudaStream_t s) {
  if (n == 0) return "";
  grad_cast_kernel<<<(unsigned)((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256), 256, 0, s>>>(g, u, out, n);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// LayerNorm backward w.r.t. its input, one warp per row:
//   xhat = (x - mean) rstd,  g = dy gamma,  dx = rstd (g - mean(g) - xhat mean(g xhat))  (+ add)
// x is the saved LayerNorm INPUT (fp32 or bf16); statistics are recomputed from it (two-pass, fp32).
template <bool X_F32, bool DY_F32>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const void* dy, const void* __restrict__ x, long long rows,
                                                      int H, const float* __restrict__ gamma, float eps,
                                                      const float* __restrict__ add, float* __restrict__ dx,
                                                      __nv_bfloat16* __restrict__ dx16) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  constexpr int MAXV = 32;   // H <= 1024
  float xv[MAXV], gv[MAXV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    float t = 0.f;
    if (idx < H) {
      if constexpr (X_F32) t = reinterpret_cast<const float*>(x)[row * H + idx];
      else t = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(x)[row * H + idx]);
    }
    xv[i] = t;
    sum += t;
  }
  const float mean = warp_sum(sum) / (float)H;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const float d = xv[i] - mean;
    if (lane + 32 * i < H) sq = fmaf(d, d, sq);
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)H + eps);
  float sg = 0.f, sgx = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    float g = 0.f;
    if (idx < H) {
      if constexpr (DY_F32) g = reinterpret_cast<const float*>(dy)[row * H + idx];
      else g = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(dy)[row * H + idx]);
      g *= __ldg(gamma + idx);
    }
    gv[i] = g;
    xv[i] = (xv[i] - mean) * rstd;   // xhat
    if (idx < H) {
      sg += g;
      sgx = fmaf(g, xv[i], sgx);
    }
  }
  const float mg = warp_sum(sg) / (float)H, mgx = warp_sum(sgx) / (float)H;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    if (idx < H) {
      float v = rstd * (gv[i] - mg - xv[i] * mgx);
      if (add) v += add[row * H + idx];
      if (dx) dx[row * H + idx] = v;
      if (dx16) dx16[row * H + idx] = __float2bfloat16_rn(v);
    }
  }
}
// Same, four consecutive elements per lane and step (16-byte loads / stores of the fp32 streams): H % 4 == 0.
__device__ __forceinline__ float4 ln_ld4(const void* p, long long i, bool f32) {
  if (f32) return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + i);
  const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p) + i);
  return make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
}
template <bool X_F32, bool DY_F32>
__global__ void __launch_bounds__(256) ln_bwd_vec_kernel(const void* dy, const void* __restrict__ x, long long rows,
                                                          int H, const float* __restrict__ gamma, float eps,
                                                          const float* __restrict__ add, float* __restrict__ dx,
                                                          __nv_bfloat16* __restrict__ dx16) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  constexpr int NV = 8;   // H <= 1024
  const long long base = row * H;
  float4 xv[NV], gv[NV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int idx = (lane + 32 * i) * 4;
    xv[i] = idx < H ? ln_ld4(x, base + idx, X_F32) : make_float4(0.f, 0.f, 0.f, 0.f);
    sum += (xv[i].x + xv[i].y) + (xv[i].z + xv[i].w);
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) {   // the gradient loads are independent of the statistics: issue them early
    const int idx = (lane + 32 * i) * 4;
    gv[i] = idx < H ? ln_ld4(dy, base + idx, DY_F32) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float mean = warp_sum(sum) / (float)H;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if ((lane + 32 * i) * 4 < H) {
      const float a = xv[i].x - mean, b = xv[i].y - mean, c = xv[i].z - mean, d = xv[i].w - mean;
      sq += (a * a + b * b) + (c * c + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)H + eps);
  float sg = 0.f, sgx = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int idx = (lane + 32 * i) * 4;
    if (idx < H) {
      const float4 gm = *reinterpret_cast<const float4*>(gamma + idx);
      gv[i] = make_float4(gv[i].x * gm.x, gv[i].y * gm.y, gv[i].z * gm.z, gv[i].w * gm.w);
      xv[i] = make_float4((xv[i].x - mean) * rstd, (xv[i].y - mean) * rstd, (xv[i].z - mean) * rstd, (xv[i].w - mean) * rstd);
      sg += (gv[i].x + gv[i].y) + (gv[i].z + gv[i].w);
      sgx += (gv[i].x * xv[i].x + gv[i].y * xv[i].y) + (gv[i].z * xv[i].z + gv[i].w * xv[i].w);
    }
  }
  const float mg = warp_sum(sg) / (float)H, mgx = warp_sum(sgx) / (float)H;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int idx = (lane + 32 * i) * 4;
    if (idx < H) {
      float4 v = make_float4(rstd * (gv[i].x - mg - xv[i].x * mgx), rstd * (gv[i].y - mg - xv[i].y * mgx),
                             rstd * (gv[i].z - mg - xv[i].z * mgx), rstd * (gv[i].w - mg - xv[i].w * mgx));
      if (add) {
        const float4 a = *reinterpret_cast<const float4*>(add + base + idx);
        v = make_float4(v.x + a.x, v.y + a.y, v.z + a.z, v.w + a.w);
      }
      if (dx) *reinterpret_cast<float4*>(dx + base + idx) = v;
      if (dx16) *reinterpret_cast<uint2*>(dx16 + base + idx) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
    }
  }
}

std::string launch_ln_bwd(const void* dy, const void* x, int x_fp32, long long rows, int H, const float* gamma, float eps,
                          const float* add, float* dx, __nv_bfloat16* dx16, cudaStream_t s, int dy_fp32) {
  if (H > 1024) return "ln_bwd: H > 1024 not supported";
  if (rows == 0) return "";
  const unsigned grid = (unsigned)((rows + 7) / 8);
  if (H % 4 == 0) {
    if (x_fp32 && dy_fp32) ln_bwd_vec_kernel<true, true><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
    else if (x_fp32) ln_bwd_vec_kernel<true, false><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
    else if (dy_fp32) ln_bwd_vec_kernel<false, true><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
    else ln_bwd_vec_kernel<false, false><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
    W2S_CUDA_OK(cudaGetLastError());
    return "";
  }
  if (x_fp32 && dy_fp32) ln_bwd_kernel<true, true><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
  else if (x_fp32) ln_bwd_kernel<true, false><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
  else if (dy_fp32) ln_bwd_kernel<false, true><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
  else ln_bwd_kernel<false, false><<<grid, 256, 0, s>>>(dy, x, rows, H, gamma, eps, add, dx, dx16);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// Start of the backward pass for the ModelWrapper output (max logit of frame `frames[b]`, shap_calculation.py:50):
// d out / d logits is one-hot at (frames[b], argmax token), so d h[b, frames[b], :] = W_head[argmax, :] and zero elsewhere.
// Also returns the selected output value.  logits: [n*T, ldl] fp32 from the forward pass.
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ logits, int ldl, int V,
                                                        const __nv_bfloat16* __restrict__ w_head, int n, int T, int H,
                                                        const int* __restrict__ frames, float* __restrict__ dh,
                                                        float* __restrict__ out_val, int active) {
  const int b = blockIdx.x;
  const int t = frames[b];
  __shared__ int s_arg;
  if (threadIdx.x < 32) {
    const float* row = logits + ((long long)b * T + t) * ldl;
    float best = -INFINITY;
    int arg = 0;
    for (int v = threadIdx.x; v < V; v += 32) {
      const float x = row[v];
      if (x > best) {
        best = x;
        arg = v;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ob > best || (ob == best && oa < arg)) {   // first maximum, as torch.max
        best = ob;
        arg = oa;
      }
    }
    if (threadIdx.x == 0) {
      s_arg = arg;
      if (out_val) out_val[b] = best;
    }
  }
  __syncthreads();
  const int arg = s_arg;
  float* dst = dh + (long long)b * T * H;
  for (long long i = threadIdx.x; i < (long long)T * H; i += blockDim.x) {
    const int tt = (int)(i / H), k = (int)(i - (long long)tt * H);
    dst[i] = (tt == t && b < active) ? __bfloat162float(w_head[(long long)arg * H + k]) : 0.f;   // reference rows: no seed
  }
}
// General vector-Jacobian seed for the same output: out[b, t] = max_v logits[b, t, v] for EVERY frame and an upstream
// gradient gout[b, t] (what autograd hands to ModelWrapper's backward): d h[b, t, :] = gout[b, t] W_head[argmax(b, t), :].
// One warp per (row, frame).
__global__ void __launch_bounds__(256) head_vjp_kernel(const float* __restrict__ logits, int ldl, int V,
                                                        const __nv_bfloat16* __restrict__ w_head, long long items, int H,
                                                        const float* __restrict__ gout, float* __restrict__ dh,
                                                        float* __restrict__ out_all) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long it = (long long)blockIdx.x * 8 + warp; it < items; it += (long long)gridDim.x * 8) {
    const float* row = logits + it * ldl;
    float best = -INFINITY;
    int arg = 0;
    for (int v = lane; v < V; v += 32) {
      const float x = row[v];
      if (x > best) {
        best = x;
        arg = v;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ob > best || (ob == best && oa < arg)) {
        best = ob;
        arg = oa;
      }
    }
    if (lane == 0 && out_all) out_all[it] = best;
    const float g = gout[it];
    for (int k = lane; k < H; k += 32) dh[it * H + k] = g * __bfloat162float(w_head[(long long)arg * H + k]);
  }
}
std::string launch_head_vjp(const float* logits, int ldl, int V, const __nv_bfloat16* w_head, int n, int T, int H,
                            const float* gout, float* dh, float* out_all, cudaStream_t s) {
  const long long items = (long long)n * T;
  if (items == 0) return "";
  long long blocks = (items + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  head_vjp_kernel<<<(unsigned)blocks, 256, 0, s>>>(logits, ldl, V, w_head, items, H, gout, dh, out_all);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// Start of the backward pass for the transcript-level output W2S_OUT_CTC (ctc.cuh), one warp per row r: the forward
// recursion stores alpha_t(s) and lse_t; the backward one carries beta_t(s) = log of the paths from (t, s) to the end,
// emissions after t only.  At every frame the state occupation q_s = exp(alpha_t(s) + beta_t(s) - log p) is summed per
// vocabulary entry -- blank over the even states, label v over the positions u with y_u = v in ascending u (a per-label
// list built once) -- so no atomics and a fixed order: gamma_t(v).  dz[r, t, v] = gamma_t(v) - softmax(z_t)_v.
__global__ void __launch_bounds__(32) ctc_grad_kernel(const float* __restrict__ logits, int ldl, int V, int T,
                                                      const int* __restrict__ labels, const int* __restrict__ offsets,
                                                      const int* __restrict__ which, int blank, int s_max,
                                                      float* __restrict__ alpha_all, float* __restrict__ lse_all,
                                                      float* __restrict__ dz, int ldz, float* __restrict__ out_val) {
  extern __shared__ float ctc_smem[];
  float* alpha = ctc_smem;                 // [s_max] working row of the forward recursion
  float* beta = alpha + s_max;             // [s_max]
  float* q = beta + s_max;                 // [s_max] occupation, then beta + emission
  int* pos = reinterpret_cast<int*>(q + s_max);   // [CTC_MAX_U] label positions grouped by label
  int* start = pos + CTC_MAX_U;            // [V + 1]
  int* cur = start + V + 1;                // [V] fill cursors
  const int b = blockIdx.x, lane = threadIdx.x;
  const int d = which[b];
  const int* lab = labels + offsets[d];
  const int U = offsets[d + 1] - offsets[d], S = 2 * U + 1;
  const int k = (S + 31) >> 5, s0 = lane * k, s1 = min(S, s0 + k);
  const float* rows = logits + (long long)b * T * ldl;
  float* alpha_row = alpha_all + (long long)b * T * s_max;
  float* lse = lse_all + (long long)b * T;
  const float logp = ctc_forward_warp<4>(
      T, V, lab, U, blank, lane, alpha,
      [&](int t, float(&lg)[4]) { return ctc_row_frame(rows + (long long)t * ldl, V, lane, lg); }, alpha_row, lse);
  if (lane == 0) {
    if (out_val) out_val[b] = logp;
    for (int v = 0; v <= V; ++v) start[v] = 0;
    for (int u = 0; u < U; ++u) ++start[lab[u] + 1];
    for (int v = 0; v < V; ++v) start[v + 1] += start[v];
    for (int v = 0; v < V; ++v) cur[v] = start[v];
    for (int u = 0; u < U; ++u) pos[cur[lab[u]]++] = u;
  }
  __syncwarp();
  for (int s = s0; s < s1; ++s) beta[s] = s >= S - 2 ? 0.f : -INFINITY;
  __syncwarp();
  for (int t = T - 1; t >= 0; --t) {
    const float* z = rows + (long long)t * ldl;
    const float* a = alpha_row + (long long)t * S;
    const float lt = lse[t];
    // occupation normalised per frame: sum_s q_s = 1 exactly in exact arithmetic (every path passes through one state
    // at t), so dividing by the computed sum instead of exp(log p) removes the rounding that alpha_t + beta_t and log p
    // accumulate in common over the frames (a nats-scale error of log p at |log p| ~ 1e4 would otherwise scale every q)
    float m = -INFINITY;
    for (int s = s0; s < s1; ++s) m = fmaxf(m, a[s] + beta[s]);   // -inf when either is; never (-inf) - (-inf)
    m = warp_max(m);
    float zs = 0.f;
    for (int s = s0; s < s1; ++s) {
      const float e = a[s] + beta[s];
      const float o = e == -INFINITY ? 0.f : expf(e - m);
      q[s] = o;
      zs += o;
    }
    const float inv = 1.f / warp_sum(zs);
    float gb = 0.f;
    for (int s = s0; s < s1; ++s) {
      q[s] *= inv;
      if (!(s & 1)) gb += q[s];
    }
    gb = warp_sum(gb);
    __syncwarp();
    for (int v = lane; v < V; v += 32) {
      float g = 0.f;
      if (v == blank) {
        g = gb;
      } else {
        for (int i = start[v]; i < start[v + 1]; ++i) g += q[2 * pos[i] + 1];
      }
      dz[((long long)b * T + t) * ldz + v] = g - expf(z[v] - lt);
    }
    __syncwarp();
    if (t == 0) break;
    // beta_{t-1}(s) = logsumexp over s' in {s, s + 1, s + 2 (skip)} of beta_t(s') + y_t(s')
    for (int s = s0; s < s1; ++s)
      q[s] = beta[s] == -INFINITY ? -INFINITY : beta[s] + (z[ctc_label(lab, blank, s)] - lt);
    __syncwarp();
    for (int s = s0; s < s1; ++s) {
      const float w1 = s + 1 < S ? q[s + 1] : -INFINITY;
      const float w2 = s + 2 < S && ctc_skip(lab, s + 2) ? q[s + 2] : -INFINITY;
      beta[s] = ctc_lae3(q[s], w1, w2);
    }
    __syncwarp();
  }
}

// dh[r, t, :] = dz[r, t, :] W_head (W_head [V, H] bf16): one block per (row, frame), the V terms added in order
__global__ void __launch_bounds__(256) ctc_seed_dh_kernel(const float* __restrict__ dz, int ldz, int V,
                                                          const __nv_bfloat16* __restrict__ w_head, int H, float* __restrict__ dh) {
  __shared__ float g[128];
  const long long rt = blockIdx.x;
  for (int v = threadIdx.x; v < V; v += blockDim.x) g[v] = dz[rt * ldz + v];
  __syncthreads();
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    float acc = 0.f;
    for (int v = 0; v < V; ++v) acc = fmaf(g[v], __bfloat162float(w_head[(long long)v * H + c]), acc);
    dh[rt * H + c] = acc;
  }
}

std::string launch_ctc_seed(const float* logits, int ldl, int V, const __nv_bfloat16* w_head, int n, int T, int H,
                            const int* labels, const int* offsets, const int* which, int blank, int s_max, float* alpha,
                            float* lse, float* dz, int ldz, float* dh, float* out_val, cudaStream_t s) {
  if (n == 0) return "";
  if (V > 128) return "ctc: vocab_size > 128 not supported";
  const size_t smem = sizeof(float) * 3 * (size_t)s_max + sizeof(int) * (CTC_MAX_U + 2 * V + 1);
  ctc_grad_kernel<<<n, 32, smem, s>>>(logits, ldl, V, T, labels, offsets, which, blank, s_max, alpha, lse, dz, ldz, out_val);
  W2S_CUDA_OK(cudaGetLastError());
  if (dh) {
    ctc_seed_dh_kernel<<<(unsigned)((long long)n * T), 256, 0, s>>>(dz, ldz, V, w_head, H, dh);
    W2S_CUDA_OK(cudaGetLastError());
  }
  return "";
}

std::string launch_head_bwd(const float* logits, int ldl, int V, const __nv_bfloat16* w_head, int n, int T, int H,
                            const int* frames, float* dh, float* out_val, cudaStream_t s, int active) {
  if (n == 0) return "";
  head_bwd_kernel<<<n, 256, 0, s>>>(logits, ldl, V, w_head, n, T, H, frames, dh, out_val, active < 0 ? n : active);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// Self-attention backward (HF wav2vec2/modeling_wav2vec2.py:438-463; no mask, eval mode), CUDA cores, two passes that
// need no atomics:
//   pass 1, one warp per query row i:  S_i. = scale q_i K^T, P = softmax(S_i.), dP_ij = dO_i . v_j,
//           D_i = sum_j P_ij dP_ij,  dS_ij = P_ij (dP_ij - D_i),  dq_i = scale sum_j dS_ij k_j;  saves (m_i, l_i, D_i)
//   pass 2, one warp per key row j:    P_ij recomputed from (m_i, l_i),  dk_j = scale sum_i dS_ij q_i,  dv_j = sum_i P_ij dO_i
// qkv: [B*T, ld] with q | k | v at column offsets 0 / H / 2H (+ head * hd);  dctx, dqkv likewise ([B*T, H], [B*T, 3H]).
constexpr int AB_MAXC = 32;   // key chunks of 32 -> T <= 1024

__global__ void __launch_bounds__(128) attn_bwd_q_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                          const __nv_bfloat16* __restrict__ dctx, int B, int T, int H,
                                                          int heads, float scale, __nv_bfloat16* __restrict__ dqkv,
                                                          float* __restrict__ stats /* [B, heads, T, 3] */) {
  __shared__ float qs[4][64], dos[4][64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long gw = (long long)blockIdx.x * 4 + warp;
  if (gw >= (long long)B * heads * T) return;
  const int i = (int)(gw % T), h = (int)((gw / T) % heads), b = (int)(gw / ((long long)T * heads));
  const int ld = 3 * H;
  const __nv_bfloat16* base = qkv + (long long)b * T * ld + h * 64;
  for (int d = lane; d < 64; d += 32) {
    qs[warp][d] = __bfloat162float(base[(long long)i * ld + d]);
    dos[warp][d] = __bfloat162float(dctx[((long long)b * T + i) * H + h * 64 + d]);
  }
  __syncwarp();
  float sc[AB_MAXC], dp[AB_MAXC];
  float mx = -INFINITY;
#pragma unroll
  for (int c = 0; c < AB_MAXC; ++c) {
    const int j = c * 32 + lane;
    float a = -INFINITY, g = 0.f;
    if (j < T) {
      const __nv_bfloat16* kr = base + (long long)j * ld + H;
      const __nv_bfloat16* vr = base + (long long)j * ld + 2 * H;
      a = 0.f;
      for (int d = 0; d < 64; d += 2) {
        const uint32_t kk = *reinterpret_cast<const uint32_t*>(kr + d);
        const uint32_t vv = *reinterpret_cast<const uint32_t*>(vr + d);
        a = fmaf(qs[warp][d], bf16_lo(kk), a);
        a = fmaf(qs[warp][d + 1], bf16_hi(kk), a);
        g = fmaf(dos[warp][d], bf16_lo(vv), g);
        g = fmaf(dos[warp][d + 1], bf16_hi(vv), g);
      }
      a *= scale;
    }
    sc[c] = a;
    dp[c] = g;
    mx = fmaxf(mx, a);
  }
  mx = warp_max(mx);
  float l = 0.f;
#pragma unroll
  for (int c = 0; c < AB_MAXC; ++c) {
    const float e = (c * 32 + lane < T) ? __expf(sc[c] - mx) : 0.f;
    sc[c] = e;
    l += e;
  }
  l = warp_sum(l);
  const float inv = 1.0f / l;
  float D = 0.f;
#pragma unroll
  for (int c = 0; c < AB_MAXC; ++c) {
    sc[c] *= inv;                // P_ij
    D = fmaf(sc[c], dp[c], D);
  }
  D = warp_sum(D);
  // dq_i = scale sum_j dS_ij k_j: lanes own dims (2 each), dS broadcast by shuffle
  float dq0 = 0.f, dq1 = 0.f;
#pragma unroll
  for (int c = 0; c < AB_MAXC; ++c) {
    if (c * 32 >= T) break;
    const float ds = sc[c] * (dp[c] - D);
    for (int l2 = 0; l2 < 32; ++l2) {
      const int j = c * 32 + l2;
      const float dsj = __shfl_sync(0xffffffffu, ds, l2);
      if (j < T) {
        const uint32_t kk = *reinterpret_cast<const uint32_t*>(base + (long long)j * ld + H + 2 * lane);
        dq0 = fmaf(dsj, bf16_lo(kk), dq0);
        dq1 = fmaf(dsj, bf16_hi(kk), dq1);
      }
    }
  }
  *reinterpret_cast<uint32_t*>(dqkv + ((long long)b * T + i) * ld + h * 64 + 2 * lane) = pack_bf16x2(dq0 * scale, dq1 * scale);
  if (lane == 0) {
    float* st = stats + (((long long)b * heads + h) * T + i) * 3;
    st[0] = mx;
    st[1] = inv;
    st[2] = D;
  }
}

__global__ void __launch_bounds__(128) attn_bwd_kv_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                           const __nv_bfloat16* __restrict__ dctx, int B, int T, int H,
                                                           int heads, float scale, __nv_bfloat16* __restrict__ dqkv,
                                                           const float* __restrict__ stats) {
  __shared__ float ks[4][64], vs[4][64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long gw = (long long)blockIdx.x * 4 + warp;
  if (gw >= (long long)B * heads * T) return;
  const int j = (int)(gw % T), h = (int)((gw / T) % heads), b = (int)(gw / ((long long)T * heads));
  const int ld = 3 * H;
  const __nv_bfloat16* base = qkv + (long long)b * T * ld + h * 64;
  for (int d = lane; d < 64; d += 32) {
    ks[warp][d] = __bfloat162float(base[(long long)j * ld + H + d]);
    vs[warp][d] = __bfloat162float(base[(long long)j * ld + 2 * H + d]);
  }
  __syncwarp();
  const float* st0 = stats + ((long long)b * heads + h) * T * 3;
  float dk0 = 0.f, dk1 = 0.f, dv0 = 0.f, dv1 = 0.f;
  for (int c = 0; c * 32 < T; ++c) {
    const int i = c * 32 + lane;
    float p = 0.f, ds = 0.f;
    if (i < T) {
      const __nv_bfloat16* qr = base + (long long)i * ld;
      const __nv_bfloat16* dor = dctx + ((long long)b * T + i) * H + h * 64;
      float a = 0.f, g = 0.f;
      for (int d = 0; d < 64; d += 2) {
        const uint32_t qq = *reinterpret_cast<const uint32_t*>(qr + d);
        const uint32_t oo = *reinterpret_cast<const uint32_t*>(dor + d);
        a = fmaf(bf16_lo(qq), ks[warp][d], a);
        a = fmaf(bf16_hi(qq), ks[warp][d + 1], a);
        g = fmaf(bf16_lo(oo), vs[warp][d], g);
        g = fmaf(bf16_hi(oo), vs[warp][d + 1], g);
      }
      p = __expf(a * scale - st0[i * 3]) * st0[i * 3 + 1];
      ds = p * (g - st0[i * 3 + 2]);
    }
    for (int l2 = 0; l2 < 32; ++l2) {
      const int ii = c * 32 + l2;
      const float pi = __shfl_sync(0xffffffffu, p, l2);
      const float dsi = __shfl_sync(0xffffffffu, ds, l2);
      if (ii < T) {
        const uint32_t qq = *reinterpret_cast<const uint32_t*>(base + (long long)ii * ld + 2 * lane);
        const uint32_t oo = *reinterpret_cast<const uint32_t*>(dctx + ((long long)b * T + ii) * H + h * 64 + 2 * lane);
        dk0 = fmaf(dsi, bf16_lo(qq), dk0);
        dk1 = fmaf(dsi, bf16_hi(qq), dk1);
        dv0 = fmaf(pi, bf16_lo(oo), dv0);
        dv1 = fmaf(pi, bf16_hi(oo), dv1);
      }
    }
  }
  __nv_bfloat16* orow = dqkv + ((long long)b * T + j) * ld + h * 64 + 2 * lane;
  *reinterpret_cast<uint32_t*>(orow + H) = pack_bf16x2(dk0 * scale, dk1 * scale);
  *reinterpret_cast<uint32_t*>(orow + 2 * H) = pack_bf16x2(dv0, dv1);
}

std::string launch_attn_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* dctx, int B, int T, int H, int heads, float scale,
                            __nv_bfloat16* dqkv, float* stats, cudaStream_t s) {
  if (H != heads * 64) return "attention backward: head_dim must be 64";
  if (T > 32 * AB_MAXC) return "attention backward: more than 1024 frames are not supported yet";
  const long long total = (long long)B * heads * T;
  if (total == 0) return "";
  attn_bwd_q_kernel<<<(unsigned)((total + 3) / 4), 128, 0, s>>>(qkv, dctx, B, T, H, heads, scale, dqkv, stats);
  attn_bwd_kv_kernel<<<(unsigned)((total + 3) / 4), 128, 0, s>>>(qkv, dctx, B, T, H, heads, scale, dqkv, stats);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// ---- attention backward on the tensor cores: the five contractions (S = Q K^T, dP = dO V^T, dV = P^T dO, dQ = dS K,
// dK = dS^T Q) run as batched GEMMs per (coalition, head) on the contraction kernels; what is left are the two row-wise
// passes below and the transposes that give every GEMM a K-major operand.  All [.., T, Tp] buffers are zero in their
// padding (columns T..Tp; cleared once when the plan is built, never written).

// rows of S (already scaled) -> P = softmax(S) as bf16, row-major and transposed.  CTA = 32 query rows of one (b, h):
// a warp holds a whole row in registers (one read of S), the CTA's 32 x T tile of P is staged in shared memory (row pitch
// an odd number of words: conflict-free column reads) and written out a second time as 64-byte runs of P^T.
constexpr int AT_MAXV = 32;   // T <= 1024

template <bool DS>   // false: P = softmax(S);  true: dS = P (dP - sum_j P dP), with `in16` = P and `in32` = dP
__global__ void __launch_bounds__(256) attn_rows_t_kernel(const float* __restrict__ in32, const __nv_bfloat16* __restrict__ in16,
                                                           int T, int Tp, __nv_bfloat16* __restrict__ out,
                                                           __nv_bfloat16* __restrict__ outT, const float* __restrict__ bd,
                                                           int Rp) {
  // bd (softmax only): the conformer's relative-position scores [bh, T, Rp]; S[i, j] += bd[i, T - 1 - i + j] (the HF
  // rel_shift as index arithmetic, modeling_wav2vec2_conformer.py:540-553) while the row is read
  extern __shared__ __nv_bfloat16 tile[];   // [32][Tp + 2]
  const int pitch = Tp + 2;
  const long long bh = blockIdx.y;
  const int i0 = blockIdx.x * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long base = bh * (long long)T * Tp;
  for (int r = warp; r < 32; r += 8) {
    const int i = i0 + r;
    if (i >= T) continue;   // warp-uniform
    const float* row32 = in32 + base + (long long)i * Tp;
    float v[AT_MAXV];
    if constexpr (!DS) {
      float mx = -INFINITY;
      const float* bdrow = bd ? bd + (bh * (long long)T + i) * Rp + (T - 1 - i) : nullptr;
#pragma unroll
      for (int c = 0; c < AT_MAXV; ++c) {
        const int j = c * 32 + lane;
        v[c] = j < T ? row32[j] + (bdrow ? bdrow[j] : 0.f) : -INFINITY;
        mx = fmaxf(mx, v[c]);
      }
      mx = warp_max(mx);
      float l = 0.f;
#pragma unroll
      for (int c = 0; c < AT_MAXV; ++c) {
        v[c] = (c * 32 + lane < T) ? __expf(v[c] - mx) : 0.f;
        l += v[c];
      }
      const float inv = 1.0f / warp_sum(l);
#pragma unroll
      for (int c = 0; c < AT_MAXV; ++c) v[c] *= inv;
    } else {
      const __nv_bfloat16* row16 = in16 + base + (long long)i * Tp;
      float pv[AT_MAXV];
      float D = 0.f;
#pragma unroll
      for (int c = 0; c < AT_MAXV; ++c) {
        const int j = c * 32 + lane;
        pv[c] = j < T ? __bfloat162float(row16[j]) : 0.f;
        v[c] = j < T ? row32[j] : 0.f;
        D = fmaf(pv[c], v[c], D);
      }
      D = warp_sum(D);
#pragma unroll
      for (int c = 0; c < AT_MAXV; ++c) v[c] = pv[c] * (v[c] - D);
    }
#pragma unroll
    for (int c = 0; c < AT_MAXV; ++c) {
      const int j = c * 32 + lane;
      if (j < T) {
        const __nv_bfloat16 q = __float2bfloat16_rn(v[c]);
        out[base + (long long)i * Tp + j] = q;
        tile[r * pitch + j] = q;
      }
    }
  }
  __syncthreads();
  const int nrow = min(32, T - i0);   // valid query rows of this CTA
  for (int j = warp; j < T; j += 8)
    if (lane < nrow) outT[base + (long long)j * Tp + i0 + lane] = tile[lane * pitch + j];
}

std::string launch_attn_softmax_t(const float* S, int BH, int T, int Tp, __nv_bfloat16* P, __nv_bfloat16* PT, cudaStream_t s,
                                  const float* bd, int Rp) {
  if (BH == 0) return "";
  if (T > 32 * AT_MAXV) return "attention backward: more than 1024 frames are not supported yet";
  const size_t smem = (size_t)32 * (Tp + 2) * sizeof(__nv_bfloat16);
  static bool attr = false;
  if (!attr) {
    W2S_CUDA_OK(cudaFuncSetAttribute(attn_rows_t_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    W2S_CUDA_OK(cudaFuncSetAttribute(attn_rows_t_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    attr = true;
  }
  attn_rows_t_kernel<false><<<dim3((T + 31) / 32, BH), 256, smem, s>>>(S, nullptr, T, Tp, P, PT, bd, Rp);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}
std::string launch_attn_ds_t(const __nv_bfloat16* P, const float* dP, int BH, int T, int Tp, __nv_bfloat16* dS,
                             __nv_bfloat16* dST, cudaStream_t s) {
  if (BH == 0) return "";
  if (T > 32 * AT_MAXV) return "attention backward: more than 1024 frames are not supported yet";
  const size_t smem = (size_t)32 * (Tp + 2) * sizeof(__nv_bfloat16);
  attn_rows_t_kernel<true><<<dim3((T + 31) / 32, BH), 256, smem, s>>>(dP, P, T, Tp, dS, dST, nullptr, 0);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// per-head transpose: src[(b T + t) ld + off + h 64 + c] -> dst[((b heads + h) 64 + c) Tp + t]   (t < T; padding untouched)
__global__ void __launch_bounds__(256) head_transpose_kernel(const __nv_bfloat16* __restrict__ src, int ld, int off, int T, int Tp,
                                                              int heads, __nv_bfloat16* __restrict__ dst) {
  __shared__ __nv_bfloat16 tile[64][66];
  const int bh = blockIdx.y, b = bh / heads, h = bh - b * heads;
  const int t0 = blockIdx.x * 64;
  for (int i = threadIdx.x; i < 64 * 64; i += blockDim.x) {
    const int r = i >> 6, c = i & 63;   // r: frame, c: channel
    const int t = t0 + r;
    tile[r][c] = t < T ? src[((long long)b * T + t) * ld + off + h * 64 + c] : __float2bfloat16_rn(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 64 * 64; i += blockDim.x) {
    const int c = i >> 6, r = i & 63;
    const int t = t0 + r;
    if (t < T) dst[((long long)bh * 64 + c) * Tp + t] = tile[r][c];
  }
}
std::string launch_head_transpose(const __nv_bfloat16* src, int ld, int off, int B, int T, int Tp, int heads, __nv_bfloat16* dst,
                                  cudaStream_t s) {
  if (B == 0) return "";
  head_transpose_kernel<<<dim3((T + 63) / 64, B * heads), 256, 0, s>>>(src, ld, off, T, Tp, heads, dst);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// Strided conv, backward w.r.t. its input.  The contraction dcol[t_out, j C + c] = sum_o du[t_out, o] W[o][j C + c] ran on the
// tensor cores; this gathers the <= ceil(kw / stride) taps that reach input frame t_in (t_in = stride t_out + j) and, when
// `u_prev` is given, multiplies by gelu'(u_prev) -- the gradient w.r.t. the previous layer's pre-activation.
__global__ void __launch_bounds__(256) conv_gather_kernel(const __nv_bfloat16* __restrict__ dcol, int T_in, int T_out, int C,
                                                           int kw, int stride, const __nv_bfloat16* __restrict__ u_prev,
                                                           __nv_bfloat16* __restrict__ out) {
  const int b = blockIdx.y;
  const int C8 = C >> 3;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)T_in * C8;
       i += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(i / C8), c = (int)(i - (long long)t * C8) * 8;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int j = t % stride; j < kw; j += stride) {
      const int to = (t - j) / stride;
      if (t - j < 0 || to >= T_out) continue;
      const uint4 v = *reinterpret_cast<const uint4*>(dcol + ((long long)b * T_out + to) * kw * C + (long long)j * C + c);
      acc[0] += bf16_lo(v.x); acc[1] += bf16_hi(v.x); acc[2] += bf16_lo(v.y); acc[3] += bf16_hi(v.y);
      acc[4] += bf16_lo(v.z); acc[5] += bf16_hi(v.z); acc[6] += bf16_lo(v.w); acc[7] += bf16_hi(v.w);
    }
    const long long o = ((long long)b * T_in + t) * C + c;
    if (u_prev) {
      const uint4 u = *reinterpret_cast<const uint4*>(u_prev + o);
      acc[0] *= gelu_grad(bf16_lo(u.x)); acc[1] *= gelu_grad(bf16_hi(u.x));
      acc[2] *= gelu_grad(bf16_lo(u.y)); acc[3] *= gelu_grad(bf16_hi(u.y));
      acc[4] *= gelu_grad(bf16_lo(u.z)); acc[5] *= gelu_grad(bf16_hi(u.z));
      acc[6] *= gelu_grad(bf16_lo(u.w)); acc[7] *= gelu_grad(bf16_hi(u.w));
    }
    uint4 r;
    r.x = pack_bf16x2(acc[0], acc[1]); r.y = pack_bf16x2(acc[2], acc[3]);
    r.z = pack_bf16x2(acc[4], acc[5]); r.w = pack_bf16x2(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(out + o) = r;
  }
}
std::string launch_conv_gather(const __nv_bfloat16* dcol, int n, int T_in, int T_out, int C, int kw, int stride,
                               const __nv_bfloat16* u_prev, __nv_bfloat16* out, cudaStream_t s) {
  if (C % 8) return "conv backward: channel count must be a multiple of 8";
  if (n == 0) return "";
  const long long per = (long long)T_in * (C / 8);
  dim3 grid((unsigned)((per + 255) / 256 > 2048 ? 2048 : (per + 255) / 256), n);
  conv_gather_kernel<<<grid, 256, 0, s>>>(dcol, T_in, T_out, C, kw, stride, u_prev, out);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// conv0 + GroupNorm-over-time, backward to the waveform (HF wav2vec2/modeling_wav2vec2.py:302-323).  With
// u = a_c (c0 - mean_c) + beta_c  (a_c = rstd_c gamma_c per (row, channel), c0 = conv0 output), du given:
//   d c0[t, c] = a_c (du[t, c] - m1_c - xhat[t, c] m2_c),   m1_c = mean_t du,  m2_c = mean_t (du xhat),  xhat = (u - beta_c) / gamma_c
//   d x[i]     = sum_c sum_{t, j: 5 t + j = i} w[c][j] d c0[t, c]
// pass 1: per (row, channel) the two time means (one warp per 32 channels x a slab of frames, fp32 atomics-free: one CTA
//         per (row, 64-channel group) walks all frames);  pass 2: per (row, frame) the 10 tap sums g[t][j] = sum_c w[c][j] d c0[t, c];
// pass 3: gather d x[i] = g[i / 5][i % 5] + g[i / 5 - 1][i % 5 + 5].
constexpr int GN_BWD_CHUNKS = 32;   // time chunks per (row, 64 channels): 8 x n x 32 CTAs instead of 8 x n
__global__ void __launch_bounds__(256) gn_bwd_stats_kernel(const __nv_bfloat16* __restrict__ du, const __nv_bfloat16* __restrict__ u,
                                                            int T0, int C, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            float* __restrict__ part /* [n, GN_BWD_CHUNKS, C, 2] sums */) {
  // CTA = (64 channels, row, time chunk); thread = (channel pair, frame lane): 32 channel pairs x 8 frame lanes
  const int row = blockIdx.y, c0 = blockIdx.x * 64, z = blockIdx.z;
  const int cp = threadIdx.x & 31, fl = threadIdx.x >> 5;
  const int c = c0 + 2 * cp;
  const int per = (T0 + GN_BWD_CHUNKS - 1) / GN_BWD_CHUNKS;
  const int t_lo = z * per, t_hi = min(T0, t_lo + per);
  __shared__ float red[8][32][4];
  float s1a = 0.f, s1b = 0.f, s2a = 0.f, s2b = 0.f;
  if (c < C) {
    const float ga = gamma[c], gb = gamma[c + 1], ba = beta[c], bb = beta[c + 1];
    const float iga = 1.0f / ga, igb = 1.0f / gb;
#pragma unroll 4
    for (int t = t_lo + fl; t < t_hi; t += 8) {
      const long long o = ((long long)row * T0 + t) * C + c;
      const uint32_t dv = *reinterpret_cast<const uint32_t*>(du + o);
      const uint32_t uv = *reinterpret_cast<const uint32_t*>(u + o);
      const float da = bf16_lo(dv), db = bf16_hi(dv);
      s1a += da;
      s1b += db;
      s2a = fmaf(da, (bf16_lo(uv) - ba) * iga, s2a);
      s2b = fmaf(db, (bf16_hi(uv) - bb) * igb, s2b);
    }
  }
  red[fl][cp][0] = s1a; red[fl][cp][1] = s1b; red[fl][cp][2] = s2a; red[fl][cp][3] = s2b;
  __syncthreads();
  if (fl == 0 && c < C) {
    float r[4] = {0.f, 0.f, 0.f, 0.f};
    for (int f = 0; f < 8; ++f)
      for (int q = 0; q < 4; ++q) r[q] += red[f][cp][q];
    float* dst = part + (((long long)row * GN_BWD_CHUNKS + z) * C + c) * 2;
    dst[0] = r[0]; dst[1] = r[2];   // channel c: (sum du, sum du xhat)
    dst[2] = r[1]; dst[3] = r[3];   // channel c + 1
  }
}
// chunk sums -> means m1 = mean(du), m2 = mean(du xhat), in a fixed order (deterministic), folded with the forward scale
// a_c = gamma_c rstd_c into the affine form the tap kernel applies per element:
//   d c0 = a (du - m1 - xhat m2),  xhat = (u - beta) / gamma   =>   d c0 = A du + B u + D
__global__ void gn_bwd_reduce_kernel(const float* __restrict__ part, int n, int C, int T0, const float* __restrict__ gn_a,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     float* __restrict__ coef /* [n, C, 3] */) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // (row, channel)
  if (i >= (long long)n * C) return;
  const long long row = i / C;
  const int c = (int)(i - row * C);
  float s1 = 0.f, s2 = 0.f;
  for (int z = 0; z < GN_BWD_CHUNKS; ++z) {
    const float* p = part + (((long long)row * GN_BWD_CHUNKS + z) * C + c) * 2;
    s1 += p[0];
    s2 += p[1];
  }
  const float m1 = s1 / (float)T0, m2 = s2 / (float)T0;
  const float a = gn_a[i], ig = 1.0f / gamma[c];
  coef[i * 3 + 0] = a;
  coef[i * 3 + 1] = -a * m2 * ig;
  coef[i * 3 + 2] = a * (beta[c] * m2 * ig - m1);
}

// pass 2: g[row, t, j] = sum_c w[c][j] (A_c du + B_c u + D_c).  A warp takes two adjacent frames per step and a lane a
// channel pair (4-byte loads); the filters sit transposed in shared memory ([tap][channel]: conflict-free 8-byte reads)
// and are read once per two frames.
template <int KW>
__global__ void __launch_bounds__(256) conv0_bwd_taps_kernel(const __nv_bfloat16* __restrict__ du, const __nv_bfloat16* __restrict__ u,
                                                              int T0, int C, const float* __restrict__ w /* [C][KW] */,
                                                              const float* __restrict__ coef /* [n, C, 3] */,
                                                              float* __restrict__ g /* [n, T0, KW] */) {
  extern __shared__ float s_w[];   // [KW][C]
  for (int i = threadIdx.x; i < C * KW; i += blockDim.x) s_w[(i % KW) * C + i / KW] = w[i];
  __syncthreads();
  const int row = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* cf_row = coef + (long long)row * C * 3;
  for (int t = 2 * (blockIdx.x * 8 + warp); t < T0; t += 2 * gridDim.x * 8) {
    const bool two = t + 1 < T0;
    float acc0[KW], acc1[KW];
#pragma unroll
    for (int j = 0; j < KW; ++j) acc0[j] = acc1[j] = 0.f;
    const long long o = ((long long)row * T0 + t) * C;
    for (int c = 2 * lane; c < C; c += 64) {
      const float2 k0 = *reinterpret_cast<const float2*>(cf_row + c * 3);       // A_c   B_c
      const float2 k1 = *reinterpret_cast<const float2*>(cf_row + c * 3 + 2);   // D_c   A_c+1
      const float2 k2 = *reinterpret_cast<const float2*>(cf_row + c * 3 + 4);   // B_c+1 D_c+1
      const uint32_t d0 = *reinterpret_cast<const uint32_t*>(du + o + c), u0 = *reinterpret_cast<const uint32_t*>(u + o + c);
      const float x0 = fmaf(k0.x, bf16_lo(d0), fmaf(k0.y, bf16_lo(u0), k1.x));
      const float y0 = fmaf(k1.y, bf16_hi(d0), fmaf(k2.x, bf16_hi(u0), k2.y));
      float x1 = 0.f, y1 = 0.f;
      if (two) {
        const uint32_t d1 = *reinterpret_cast<const uint32_t*>(du + o + C + c), u1 = *reinterpret_cast<const uint32_t*>(u + o + C + c);
        x1 = fmaf(k0.x, bf16_lo(d1), fmaf(k0.y, bf16_lo(u1), k1.x));
        y1 = fmaf(k1.y, bf16_hi(d1), fmaf(k2.x, bf16_hi(u1), k2.y));
      }
#pragma unroll
      for (int j = 0; j < KW; ++j) {
        const float2 wj = *reinterpret_cast<const float2*>(s_w + j * C + c);
        acc0[j] = fmaf(wj.x, x0, fmaf(wj.y, y0, acc0[j]));
        acc1[j] = fmaf(wj.x, x1, fmaf(wj.y, y1, acc1[j]));
      }
    }
#pragma unroll
    for (int j = 0; j < KW; ++j) {
      acc0[j] = warp_sum(acc0[j]);
      acc1[j] = warp_sum(acc1[j]);
    }
    if (lane == 0) {
      float* dst = g + ((long long)row * T0 + t) * KW;
#pragma unroll
      for (int j = 0; j < KW; ++j) dst[j] = acc0[j];
      if (two) {
#pragma unroll
        for (int j = 0; j < KW; ++j) dst[KW + j] = acc1[j];
      }
    }
  }
}

// pass 3: d x[i] = sum over the frames t with 0 <= i - stride t < KW of g[t][i - stride t]
__global__ void __launch_bounds__(256) conv0_bwd_gather_kernel(const float* __restrict__ g, int T0, int KW, int stride, long long L,
                                                                float* __restrict__ dx, long long ld) {
  const int row = blockIdx.y;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += (long long)gridDim.x * blockDim.x) {
    float acc = 0.f;
    const long long thi = i / stride;
    for (long long t = thi; t >= 0 && i - t * stride < KW; --t)
      if (t < T0) acc += g[((long long)row * T0 + t) * KW + (i - t * stride)];
    dx[(long long)row * ld + i] = acc;
  }
}

std::string launch_conv0_bwd(const __nv_bfloat16* du, const __nv_bfloat16* u, int n, long long L, int T0, int C, int kw, int stride,
                             const float* w, const float* gn_a, const float* gamma, const float* beta, float* m12, float* g,
                             float* dx, long long ld, cudaStream_t s) {
  if (kw != 10) return "conv0 backward: only kernel width 10 is implemented";
  if (C % 64) return "conv0 backward: channel count must be a multiple of 64";
  if (n == 0) return "";
  // the caller's scratch buffer `m12` holds the [n, C, 3] coefficients + the [n, 32, C, 2] chunk sums
  float* coef = m12;
  float* part = m12 + (long long)n * C * 3;
  gn_bwd_stats_kernel<<<dim3(C / 64, n, GN_BWD_CHUNKS), 256, 0, s>>>(du, u, T0, C, gamma, beta, part);
  gn_bwd_reduce_kernel<<<(unsigned)(((long long)n * C + 255) / 256), 256, 0, s>>>(part, n, C, T0, gn_a, gamma, beta, coef);
  const unsigned gx = (unsigned)((T0 + 15) / 16 > 1024 ? 1024 : (T0 + 15) / 16);
  conv0_bwd_taps_kernel<10><<<dim3(gx, n), 256, sizeof(float) * C * 10, s>>>(du, u, T0, C, w, coef, g);
  conv0_bwd_gather_kernel<<<dim3((unsigned)((L + 255) / 256 > 1024 ? 1024 : (L + 255) / 256), n), 256, 0, s>>>(g, T0, kw, stride, L, dx, ld);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// conv0 + LayerNorm over channels (feat_extract_norm = "layer", HF wav2vec2/modeling_wav2vec2.py:275-299), backward to the
// waveform.  u = gamma xhat + beta with xhat = (c0 - mean_f) rstd_f per frame f; du given, rstd_f saved by the forward pass:
//   d c0[f, c] = rstd_f (g - mean_c g - xhat mean_c (g xhat)),  g = du gamma,  xhat = (u - beta) / gamma
//   taps[f][j] = sum_c w[c][j] d c0[f, c];  d x[i] = sum of the taps that reach sample i (conv0_bwd_gather_kernel)
template <int KW>
__global__ void __launch_bounds__(256) conv0_ln_bwd_taps_kernel(const __nv_bfloat16* __restrict__ du, const __nv_bfloat16* __restrict__ u,
                                                                 const float* __restrict__ rstd, int T0, int C,
                                                                 const float* __restrict__ w, const float* __restrict__ gamma,
                                                                 const float* __restrict__ beta, float* __restrict__ g) {
  const int row = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = blockIdx.x * 8 + warp; t < T0; t += gridDim.x * 8) {
    const long long o0 = ((long long)row * T0 + t) * C;
    float s1 = 0.f, s2 = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float gc = __bfloat162float(du[o0 + c]) * gamma[c];
      const float xh = (__bfloat162float(u[o0 + c]) - beta[c]) / gamma[c];
      s1 += gc;
      s2 = fmaf(gc, xh, s2);
    }
    const float m1 = warp_sum(s1) / (float)C, m2 = warp_sum(s2) / (float)C;
    const float rs = rstd[(long long)row * T0 + t];
    float acc[KW];
#pragma unroll
    for (int j = 0; j < KW; ++j) acc[j] = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float gc = __bfloat162float(du[o0 + c]) * gamma[c];
      const float xh = (__bfloat162float(u[o0 + c]) - beta[c]) / gamma[c];
      const float dc = rs * (gc - m1 - xh * m2);
#pragma unroll
      for (int j = 0; j < KW; ++j) acc[j] = fmaf(__ldg(w + c * KW + j), dc, acc[j]);
    }
#pragma unroll
    for (int j = 0; j < KW; ++j) acc[j] = warp_sum(acc[j]);
    if (lane == 0) {
      float* dst = g + ((long long)row * T0 + t) * KW;
#pragma unroll
      for (int j = 0; j < KW; ++j) dst[j] = acc[j];
    }
  }
}
std::string launch_conv0_ln_bwd(const __nv_bfloat16* du, const __nv_bfloat16* u, const float* rstd, int n, long long L, int T0, int C,
                                int kw, int stride, const float* w, const float* gamma, const float* beta, float* g, float* dx,
                                long long ld, cudaStream_t s) {
  if (kw != 10) return "conv0 backward: only kernel width 10 is implemented";
  if (n == 0) return "";
  conv0_ln_bwd_taps_kernel<10><<<dim3((unsigned)((T0 + 7) / 8 > 1024 ? 1024 : (T0 + 7) / 8), n), 256, 0, s>>>(du, u, rstd, T0, C, w, gamma, beta, g);
  conv0_bwd_gather_kernel<<<dim3((unsigned)((L + 255) / 256 > 1024 ? 1024 : (L + 255) / 256), n), 256, 0, s>>>(g, T0, kw, stride, L, dx, ld);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// ---- conformer encoder (HF modeling_wav2vec2_conformer.py:568-630): activation, GLU, relative-position shift ----------
// act'(u) for the encoder's activation (ACT2FN[config.hidden_act]): swish'(u) = s (1 + u (1 - s)), s = sigmoid(u)
__device__ __forceinline__ float act_grad(float u, int act) {
  if (act == ACT_SWISH) {
    const float sg = 1.0f / (1.0f + __expf(-u));
    return sg * fmaf(u, 1.0f - sg, 1.0f);
  }
  return gelu_grad(u);
}

// y = act(u)
__global__ void __launch_bounds__(256) act_fwd_kernel(const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ y,
                                                       long long n2, int act) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t a = reinterpret_cast<const uint32_t*>(u)[i];
    reinterpret_cast<uint32_t*>(y)[i] = pack_bf16x2(apply_act(bf16_lo(a), act), apply_act(bf16_hi(a), act));
  }
}
std::string launch_act_fwd(const __nv_bfloat16* u, __nv_bfloat16* y, long long n, int act, cudaStream_t s) {
  if (n % 2) return "act_fwd: element count must be even";
  if (n == 0) return "";
  const long long n2 = n / 2;
  act_fwd_kernel<<<(unsigned)((n2 + 255) / 256 > 148 * 16 ? 148 * 16 : (n2 + 255) / 256), 256, 0, s>>>(u, y, n2, act);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// DeepLIFT "rescale" multiplier of an activation (shap's nonlinear_1d, which custom_shap_handlers.py:45-52 assigns to SiLU):
// (act(x) - act(r)) / (x - r) between the explained row's input x and the paired reference row's r; the ordinary
// derivative where |x - r| < 1e-6
__device__ __forceinline__ float act_rescale(float x, float r, int act) {
  const float dx = x - r;
  return fabsf(dx) < 1e-6f ? act_grad(x, act) : (apply_act(x, act) - apply_act(r, act)) / dx;
}
// d <- d * act'(u) (* chan_scale[column] when given: the folded BatchNorm scale that sits between u's producer and act).
// pair2 > 0: rows come as [explained | reference] halves (pair2 = bf16 PAIRS per half) and the explained half uses the
// rescale multiplier against its reference row.
__global__ void __launch_bounds__(256) act_bwd_kernel(const __nv_bfloat16* __restrict__ u, __nv_bfloat16* __restrict__ d,
                                                       long long n2, int act, const float* __restrict__ chan_scale, int H,
                                                       long long pair2) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t a = reinterpret_cast<const uint32_t*>(u)[i];
    const uint32_t g = reinterpret_cast<const uint32_t*>(d)[i];
    float mlo, mhi;
    if (pair2 > 0 && i < pair2) {
      const uint32_t r = reinterpret_cast<const uint32_t*>(u)[i + pair2];
      mlo = act_rescale(bf16_lo(a), bf16_lo(r), act);
      mhi = act_rescale(bf16_hi(a), bf16_hi(r), act);
    } else {
      mlo = act_grad(bf16_lo(a), act);
      mhi = act_grad(bf16_hi(a), act);
    }
    float lo = bf16_lo(g) * mlo, hi = bf16_hi(g) * mhi;
    if (chan_scale) {
      const int c = (int)((2 * i) % H);
      lo *= chan_scale[c];
      hi *= chan_scale[c + 1];
    }
    reinterpret_cast<uint32_t*>(d)[i] = pack_bf16x2(lo, hi);
  }
}
std::string launch_act_bwd(const __nv_bfloat16* u, __nv_bfloat16* d, long long n, int act, const float* chan_scale, int H,
                           cudaStream_t s, int paired) {
  if (n % 2 || H % 2) return "act_bwd: element and channel counts must be even";
  if (paired && n % 4) return "act_bwd: paired rows need an even row count";
  if (n == 0) return "";
  const long long n2 = n / 2;
  act_bwd_kernel<<<(unsigned)((n2 + 255) / 256 > 148 * 16 ? 148 * 16 : (n2 + 255) / 256), 256, 0, s>>>(u, d, n2, act, chan_scale, H,
                                                                                                     paired ? n2 / 2 : 0);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// GLU over interleaved (value, gate) column pairs: out[r, j] = raw[r, 2j] sigmoid(raw[r, 2j + 1])
__global__ void __launch_bounds__(256) glu_fwd_kernel(const __nv_bfloat16* __restrict__ raw, __nv_bfloat16* __restrict__ out,
                                                       long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t a = reinterpret_cast<const uint32_t*>(raw)[i];
    out[i] = __float2bfloat16_rn(bf16_lo(a) / (1.0f + __expf(-bf16_hi(a))));
  }
}
std::string launch_glu_fwd(const __nv_bfloat16* raw, __nv_bfloat16* out, long long n, cudaStream_t s) {
  if (n == 0) return "";
  glu_fwd_kernel<<<(unsigned)((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256), 256, 0, s>>>(raw, out, n);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}
// d raw[r, 2j] = d out sigmoid(gate);  d raw[r, 2j + 1] = d out value sigmoid(gate) (1 - sigmoid(gate))
// pair > 0 (elements of the explained half): the reference's GLU handler (custom_shap_handlers.py:63-80, a placeholder its
// author left in): every GLU input channel whose explained and reference values differ by >= 1e-6 receives
// grad_output * 5e-6, the others the ordinary gradient
__global__ void __launch_bounds__(256) glu_bwd_kernel(const __nv_bfloat16* __restrict__ raw, const __nv_bfloat16* __restrict__ dout,
                                                       __nv_bfloat16* __restrict__ draw, long long n, long long pair) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t a = reinterpret_cast<const uint32_t*>(raw)[i];
    const float g = __bfloat162float(dout[i]);
    const float sg = 1.0f / (1.0f + __expf(-bf16_hi(a)));
    float dv = g * sg, dg = g * bf16_lo(a) * sg * (1.0f - sg);
    if (pair > 0) {
      const uint32_t r = reinterpret_cast<const uint32_t*>(raw)[i < pair ? i + pair : i - pair];
      // the saved inputs are bf16: two values that round to the same bf16 number of magnitude m may still differ by up to
      // m 2^-8 in the fp32 model, so "differs by < 1e-6" is only certain below m = 2.5e-4
      auto same = [](float x, float y) { return fabsf(x - y) < 1e-6f && fabsf(x) < 2.5e-4f; };
      if (!same(bf16_lo(a), bf16_lo(r))) dv = g * 5e-6f;
      if (!same(bf16_hi(a), bf16_hi(r))) dg = g * 5e-6f;
    }
    reinterpret_cast<uint32_t*>(draw)[i] = pack_bf16x2(dv, dg);
  }
}
std::string launch_glu_bwd(const __nv_bfloat16* raw, const __nv_bfloat16* dout, __nv_bfloat16* draw, long long n, cudaStream_t s,
                           int placeholder_paired) {
  if (n == 0) return "";
  if (placeholder_paired && n % 2) return "glu_bwd: paired rows need an even row count";
  glu_bwd_kernel<<<(unsigned)((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256), 256, 0, s>>>(raw, dout, draw, n,
                                                                                                   placeholder_paired ? n / 2 : 0);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// relative positions: the forward gather S[bh, i, j] += BD[bh, i, T - 1 - i + j] is folded into attn_rows_t_kernel;
// the transpose of that gather: dBD[bh, i, r] = dS[bh, i, r - (T - 1) + i] where that key exists, else 0 (all Rp columns
// written, eight per thread as one 16-byte store)
__global__ void __launch_bounds__(128) rel_unshift_kernel(const __nv_bfloat16* __restrict__ dS, __nv_bfloat16* __restrict__ dBD,
                                                           int T, int Tp, int Rp) {
  const long long row = (long long)blockIdx.y * T + blockIdx.x;
  const int i = blockIdx.x;
  const __nv_bfloat16* src = dS + row * Tp;
  __nv_bfloat16* dst = dBD + row * Rp;
  const int shift = i - (T - 1);
  for (int r0 = threadIdx.x * 8; r0 < Rp; r0 += blockDim.x * 8) {
    __align__(16) __nv_bfloat16 v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int j = r0 + k + shift;
      v[k] = (j >= 0 && j < T) ? src[j] : __float2bfloat16_rn(0.f);
    }
    *reinterpret_cast<uint4*>(dst + r0) = *reinterpret_cast<const uint4*>(v);
  }
}
std::string launch_rel_unshift(const __nv_bfloat16* dS, __nv_bfloat16* dBD, int BH, int T, int Tp, int Rp, cudaStream_t s) {
  if (BH == 0) return "";
  if (Rp % 8) return "rel_unshift: padded relative-position count must be a multiple of 8";
  rel_unshift_kernel<<<dim3(T, BH), 128, 0, s>>>(dS, dBD, T, Tp, Rp);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// depthwise conv backward-data taps: dst[j][c] = src[k - 1 - j][c]  (taps stored [k][H]; "same" padding, odd k)
__global__ void flip_taps_kernel(const float* __restrict__ src, float* __restrict__ dst, int k, int H) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < k * H) {
    const int j = i / H, c = i - j * H;
    dst[i] = src[(k - 1 - j) * H + c];
  }
}
std::string launch_flip_taps(const float* src, float* dst, int k, int H, cudaStream_t s) {
  flip_taps_kernel<<<(k * H + 255) / 256, 256, 0, s>>>(src, dst, k, H);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}
__global__ void fill_f32_kernel(float* dst, float v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = v;
}
std::string launch_fill_f32(float* dst, float v, int n, cudaStream_t s) {
  fill_f32_kernel<<<(n + 255) / 256, 256, 0, s>>>(dst, v, n);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// ---- weight re-layout for the backward contractions (once, at first use) --------------------------------------
// dst[c][r] = src[r][c]  (bf16, R x C -> C x R)
__global__ void transpose_bf16_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int R, int C) {
  __shared__ __nv_bfloat16 tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < C) ? src[(long long)r * C + c] : __float2bfloat16_rn(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < R && c < C) dst[(long long)c * R + r] = tile[threadIdx.x][i];
  }
}
std::string launch_transpose_bf16(const __nv_bfloat16* src, __nv_bfloat16* dst, int R, int C, cudaStream_t s) {
  transpose_bf16_kernel<<<dim3((C + 31) / 32, (R + 31) / 32), dim3(32, 8), 0, s>>>(src, dst, R, C);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// positional conv, backward-data weights: w'[g][ci][j' * 64 + co] = w[g*cpg + co][ci][kw - 1 - j']  (zero for co >= cpg),
// from the HF layout src[H][cpg][kw] (weight-norm already folded)
__global__ void repack_posconv_bwd_kernel(const float* src, __nv_bfloat16* dst, int H, int G, int kw) {
  const int cpg = H / G;
  const long long n = (long long)H * kw * 64;   // [G][cpg (ci)][kw * 64 + co]
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i & 63);
    const int jp = (int)((i >> 6) % kw);
    const int row = (int)(i / ((long long)kw * 64));   // g * cpg + ci
    const int g = row / cpg, ci = row - g * cpg;
    float v = 0.f;
    if (co < cpg) v = src[((long long)(g * cpg + co) * cpg + ci) * kw + (kw - 1 - jp)];
    dst[i] = __float2bfloat16_rn(v);
  }
}
std::string launch_repack_posconv_bwd(const float* src, __nv_bfloat16* dst, int H, int G, int kw, cudaStream_t s) {
  const long long n = (long long)H * kw * 64;
  repack_posconv_bwd_kernel<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, dst, H, G, kw);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

}  // namespace w2s
