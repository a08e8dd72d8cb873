// K9: lm_head (H -> V) fused with the output reduction of the callback.
//   max logit per frame            shap_calculation.py:50
//   logit at (frame, token)        feasability_tests/w2v2conformer.py:40-42
//   log-softmax at (frame, token)  north-star per-character CTC log-probability
//   mean over vocab and time       feasability_tests/lime_shap_wav2vec2_comparison.py:68-70
//   CTC log-likelihood of a transcript over all frames (ctc.cuh), -Wav2Vec2ForCTC(x, labels=y).loss
// One warp per (row, frame) work item: lane = vocabulary entry, so log-softmax and gather are warp
// shuffles (HF wav2vec2/modeling_wav2vec2.py:1705-1708 for the linear layer).
#include "kernels.cuh"
#include "ctc.cuh"
#include "../../include/w2s.h"

namespace w2s {

constexpr int HEAD_MAXJ = 4;  // V <= 128

// Reduction of one frame's logits held one-per-lane (logit[j] = entry lane + 32 j): shared by both kernels.
__device__ __forceinline__ void head_reduce_frame(const float (&logit)[HEAD_MAXJ], int V, int mode, int tok, int lane,
                                                  float* dst) {
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < HEAD_MAXJ; ++j)
    if (lane + 32 * j < V) mx = fmaxf(mx, logit[j]);
  mx = warp_max(mx);
  if (mode == W2S_OUT_MAX) {
    if (lane == 0) *dst = mx;
    return;
  }
  float sel = 0.f;
#pragma unroll
  for (int j = 0; j < HEAD_MAXJ; ++j) {
    const float cand = __shfl_sync(0xffffffffu, logit[j], tok & 31);
    if ((tok >> 5) == j) sel = cand;
  }
  if (mode == W2S_OUT_LOGPROB) {
    float se = 0.f;
#pragma unroll
    for (int j = 0; j < HEAD_MAXJ; ++j)
      if (lane + 32 * j < V) se += __expf(logit[j] - mx);
    se = warp_sum(se);
    sel -= mx + __logf(se);
  }
  if (lane == 0) *dst = sel;
}

// Work items per mode: MAX / LOGITS one per (row, frame); LOGIT / LOGPROB one per (row, target); CTC one per (row,
// transcript); MEAN one per row (the warp walks the frames in order, so the sum is bit-reproducible -- no atomics).
__device__ __forceinline__ long long head_items(const DynArgs& d, int n, int T) {
  if (d.mode == W2S_OUT_LOGIT || d.mode == W2S_OUT_LOGPROB || d.mode == W2S_OUT_CTC) return (long long)n * d.D;
  if (d.mode == W2S_OUT_MEAN) return n;
  return (long long)n * T;
}

// CUDA-core validation variant: lm_head (H -> V) + reduction in one kernel, weights staged in shared memory.
__global__ void __launch_bounds__(256) head_kernel(const HeadParams p) {
  extern __shared__ uint8_t smem[];
  const DynArgs d = *p.dyn;
  // the pointers of the argument block are device allocations: keeps the stores and target loads global (LDG / STG)
  __builtin_assume(__isGlobal(d.out) && __isGlobal(d.frames) && __isGlobal(d.tokens));
  const int ldw = p.H + 2;  // bf16 elements; (H+2)/2 odd -> conflict-free row stride
  __nv_bfloat16* ws = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* hs = ws + (size_t)p.V * ldw;  // 8 warps x H
  float* ctc_alpha = reinterpret_cast<float*>(hs + 8 * (size_t)p.H);   // 8 warps x CTC_MAX_S, then 8 warps x 128 logits
  for (int i = threadIdx.x; i < p.V * p.H; i += blockDim.x) {
    const int v = i / p.H, k = i - v * p.H;
    ws[v * ldw + k] = p.w[i];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __nv_bfloat16* hrow = hs + (size_t)warp * p.H;
  const bool targeted = (d.mode == W2S_OUT_LOGIT || d.mode == W2S_OUT_LOGPROB);
  const long long items = head_items(d, p.n, p.T);
  const int per = targeted ? d.D : p.T;
  auto frame_logits = [&](int b, int t, float (&logit)[HEAD_MAXJ]) {
    const __nv_bfloat16* src = p.h + ((long long)b * p.T + t) * p.H;
    __syncwarp();
    for (int k = lane * 2; k < p.H; k += 64)
      *reinterpret_cast<uint32_t*>(hrow + k) = *reinterpret_cast<const uint32_t*>(src + k);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < HEAD_MAXJ; ++j) {
      const int v = lane + 32 * j;
      float acc = 0.f;
      if (v < p.V) {
        const __nv_bfloat16* wr = ws + (size_t)v * ldw;
        for (int k = 0; k < p.H; k += 2) {
          const uint32_t hh = *reinterpret_cast<const uint32_t*>(hrow + k);
          const uint32_t ww = *reinterpret_cast<const uint32_t*>(wr + k);
          acc = fmaf(bf16_lo(hh), bf16_lo(ww), acc);
          acc = fmaf(bf16_hi(hh), bf16_hi(ww), acc);
        }
        acc += p.bias[v];
      }
      logit[j] = acc;
    }
  };
  for (long long it = (long long)blockIdx.x * 8 + warp; it < items; it += (long long)gridDim.x * 8) {
    float logit[HEAD_MAXJ];
    if (d.mode == W2S_OUT_CTC) {
      const int b = (int)(it / d.D), dd = (int)(it - (long long)b * d.D);
      float* zs = ctc_alpha + 8 * CTC_MAX_S + warp * 32 * HEAD_MAXJ;   // the frame's logits, indexed by vocabulary id
      const float r = ctc_forward_warp<HEAD_MAXJ>(
          p.T, p.V, d.ctc_labels + d.ctc_offsets[dd], d.ctc_offsets[dd + 1] - d.ctc_offsets[dd], d.blank, lane,
          ctc_alpha + warp * CTC_MAX_S, [&](int t, float(&lg)[HEAD_MAXJ]) -> const float* {
            frame_logits(b, t, lg);
#pragma unroll
            for (int j = 0; j < HEAD_MAXJ; ++j)
              if (lane + 32 * j < p.V) zs[lane + 32 * j] = lg[j];
            __syncwarp();
            return zs;
          });
      if (lane == 0) d.out[(long long)b * d.D + dd] = r;
      continue;
    }
    if (d.mode == W2S_OUT_MEAN) {
      float sm = 0.f;
      for (int t = 0; t < p.T; ++t) {
        frame_logits((int)it, t, logit);
#pragma unroll
        for (int j = 0; j < HEAD_MAXJ; ++j)
          if (lane + 32 * j < p.V) sm += logit[j];
      }
      sm = warp_sum(sm);
      if (lane == 0) d.out[it] = sm / ((float)p.V * (float)p.T);
      continue;
    }
    const int b = (int)(it / per);
    const int dd = (int)(it - (long long)b * per);
    const int t = targeted ? d.frames[dd] : dd;
    frame_logits(b, t, logit);
    if (d.mode == W2S_OUT_LOGITS) {
#pragma unroll
      for (int j = 0; j < HEAD_MAXJ; ++j) {
        const int v = lane + 32 * j;
        if (v < p.V) d.out[((long long)b * p.T + t) * p.V + v] = logit[j];
      }
      continue;
    }
    head_reduce_frame(logit, p.V, d.mode, targeted ? d.tokens[dd] : 0, lane,
                      d.out + (targeted ? (long long)b * d.D + dd : (long long)b * p.T + t));
  }
}

// second stage of the tensor-core head: logits[rows, ldl] (fp32, bias included) -> reduction; one warp per work item.
// Six blocks per SM, as before the CTC branch was added: its alpha rows take 32.8 KB of shared memory per block, and the
// bound keeps the register count of every mode at 40.
__global__ void __launch_bounds__(256, 6) head_reduce_kernel(const float* __restrict__ logits, const HeadParams p) {
  __shared__ float ctc_alpha[8][CTC_MAX_S];
  const DynArgs d = *p.dyn;
  __builtin_assume(__isGlobal(d.out) && __isGlobal(d.frames) && __isGlobal(d.tokens));   // as in head_kernel
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool targeted = (d.mode == W2S_OUT_LOGIT || d.mode == W2S_OUT_LOGPROB);
  const long long items = head_items(d, p.n, p.T);
  const int per = targeted ? d.D : p.T;
  for (long long it = (long long)blockIdx.x * 8 + warp; it < items; it += (long long)gridDim.x * 8) {
    float logit[HEAD_MAXJ];
    if (d.mode == W2S_OUT_CTC) {
      const int b = (int)(it / d.D), dd = (int)(it - (long long)b * d.D);
      const float* rows = logits + (long long)b * p.T * p.ldl;
      const float r = ctc_forward_warp<HEAD_MAXJ>(
          p.T, p.V, d.ctc_labels + d.ctc_offsets[dd], d.ctc_offsets[dd + 1] - d.ctc_offsets[dd], d.blank, lane,
          ctc_alpha[warp], [&](int t, float(&lg)[HEAD_MAXJ]) -> const float* {
            const float* row = rows + (long long)t * p.ldl;
#pragma unroll
            for (int j = 0; j < HEAD_MAXJ; ++j) lg[j] = lane + 32 * j < p.V ? row[lane + 32 * j] : -INFINITY;
            return row;
          });
      if (lane == 0) d.out[(long long)b * d.D + dd] = r;
      continue;
    }
    if (d.mode == W2S_OUT_MEAN) {
      const float* row = logits + it * p.T * p.ldl;
      float sm = 0.f;
      for (int t = 0; t < p.T; ++t) {
#pragma unroll
        for (int j = 0; j < HEAD_MAXJ; ++j)
          if (lane + 32 * j < p.V) sm += row[(long long)t * p.ldl + lane + 32 * j];
      }
      sm = warp_sum(sm);
      if (lane == 0) d.out[it] = sm / ((float)p.V * (float)p.T);
      continue;
    }
    const int b = (int)(it / per);
    const int dd = (int)(it - (long long)b * per);
    const int t = targeted ? d.frames[dd] : dd;
    const float* row = logits + ((long long)b * p.T + t) * p.ldl;
#pragma unroll
    for (int j = 0; j < HEAD_MAXJ; ++j) {
      const int v = lane + 32 * j;
      logit[j] = v < p.V ? row[v] : -INFINITY;
    }
    if (d.mode == W2S_OUT_LOGITS) {
#pragma unroll
      for (int j = 0; j < HEAD_MAXJ; ++j) {
        const int v = lane + 32 * j;
        if (v < p.V) d.out[((long long)b * p.T + t) * p.V + v] = logit[j];
      }
      continue;
    }
    head_reduce_frame(logit, p.V, d.mode, targeted ? d.tokens[dd] : 0, lane,
                      d.out + (targeted ? (long long)b * d.D + dd : (long long)b * p.T + t));
  }
}

// The grid is sized for one item per (row, frame) -- the largest item count any mode has, unless more targets than
// frames were set, which the grid-stride loops absorb -- so the launch does not depend on the per-call mode.
static unsigned head_grid(const HeadParams& p, int cap) {
  long long blocks = ((long long)p.n * p.T + 7) / 8;
  if (blocks > cap) blocks = cap;
  return (unsigned)(blocks < 1 ? 1 : blocks);
}

std::string launch_head_reduce(const float* logits, const HeadParams& p, cudaStream_t s) {
  if (p.V > 32 * HEAD_MAXJ) return "head: vocab_size > 128 not supported";
  if (p.n == 0) return "";
  W2S_CUDA_OK(launch_pdl(head_reduce_kernel, dim3(head_grid(p, 148 * 8)), dim3(256), 0, s, 1, logits, p));
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

static bool g_head_attr = false;

std::string launch_head(const HeadParams& p, cudaStream_t s) {
  if (p.V > 32 * HEAD_MAXJ) return "head: vocab_size > 128 not supported";
  if (p.H % 2) return "head: hidden size must be even";
  if (p.n == 0) return "";
  // weights and hidden rows (bf16), then the CTC scratch of every warp: alpha and one frame of logits (fp32)
  const size_t smem = ((size_t)p.V * (p.H + 2) + 8 * (size_t)p.H) * sizeof(__nv_bfloat16) +
                      8 * (size_t)(CTC_MAX_S + 32 * HEAD_MAXJ) * sizeof(float);
  if (!g_head_attr) {
    W2S_CUDA_OK(cudaFuncSetAttribute(head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    g_head_attr = true;
  }
  if (smem > 200 * 1024) return "head: vocab * hidden too large for shared memory";
  head_kernel<<<head_grid(p, 148 * 4), 256, smem, s>>>(p);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// Background mean of a w2s_eval call with a background: the K * B per-row outputs (coalition-major) -> out[K, width].
// One thread per (coalition, column); the terms are added in the documented order b = 0 .. B-1, one fmaf each from 0, so
// the result does not depend on the batch tile or on how the coalitions are spread over GPUs.
__global__ void __launch_bounds__(256) bg_mean_kernel(const float* __restrict__ rows, const float* __restrict__ w, int B,
                                                      long long K, long long width, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K * width) return;
  const long long k = i / width, c = i - k * width;
  const float* r = rows + k * B * width + c;
  float acc = 0.f;
  for (int b = 0; b < B; ++b) acc = fmaf(__ldg(w + b), __ldg(r + (long long)b * width), acc);
  out[i] = acc;
}

std::string launch_bg_mean(const float* rows, const float* w, int B, long long K, long long width, float* out,
                           cudaStream_t s) {
  const long long n = K * width;
  if (n == 0) return "";
  bg_mean_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(rows, w, B, K, width, out);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

}  // namespace w2s
