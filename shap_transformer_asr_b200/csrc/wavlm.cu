// WavLM's gated relative-position bias (HF wavlm/modeling_wavlm.py:147-186, :253-271): the bucket table (host, double
// precision), the per-clip-length bias table the attention kernels read, and the per-layer gate.  The bias term itself is
// added inside the attention kernels (attention_fa.cu, attention.cu).
#include "../../include/w2s.h"
#include "kernels.cuh"

#include <cmath>

namespace w2s {

__global__ void rel_bias_table_kernel(const float* src, const int32_t* bucket, int T, int heads, float* out) {
  const int ld = rel_bias_ld(T);
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)heads * ld) return;
  const int h = (int)(idx / ld), r = (int)(idx % ld) - REL_BIAS_PAD;
  float v = 0.f;
  if (r >= 0 && r < 2 * T - 1) v = (bucket ? src[bucket[r] * heads + h] : src[(long long)h * (2 * T - 1) + r]) * 1.4426950408889634f;
  out[idx] = v;
}

std::string launch_rel_bias_table(const float* src, const int32_t* bucket, int T, int heads, float* out, cudaStream_t s) {
  const long long n = (long long)heads * rel_bias_ld(T);
  rel_bias_table_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, bucket, T, heads, out);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// One thread per (row, head): 64 bf16 inputs (one 128-byte line; the lanes of a warp read consecutive lines), 8 outputs.
__global__ void __launch_bounds__(256) wavlm_gate_kernel(const __nv_bfloat16* x, long long rows, int T, int heads,
                                                         const float* w, const float* bias, const float* c, float* gate) {
  __shared__ float ws[8 * 64];
  __shared__ float bs[8];
  for (int k = threadIdx.x; k < 8 * 64; k += blockDim.x) ws[k] = w[k];
  if (threadIdx.x < 8) bs[threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * heads) return;
  const long long r = t / heads;
  const int h = (int)(t % heads);
  const uint4* xp = reinterpret_cast<const uint4*>(x + r * heads * 64 + h * 64);
  float acc[8];
#pragma unroll
  for (int o = 0; o < 8; ++o) acc[o] = bs[o];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const uint4 u = xp[q];
    const float xv[8] = {bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y),
                         bf16_lo(u.z), bf16_hi(u.z), bf16_lo(u.w), bf16_hi(u.w)};
#pragma unroll
    for (int o = 0; o < 8; ++o)
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[o] = fmaf(ws[o * 64 + q * 8 + e], xv[e], acc[o]);
  }
  // :169-176: the 8 outputs viewed as (2, 4) and summed, sigmoid, gate_a (gate_b c_h - 1) + 2
  const float a = 1.f / (1.f + expf(-((acc[0] + acc[1]) + (acc[2] + acc[3]))));
  const float bp = 1.f / (1.f + expf(-((acc[4] + acc[5]) + (acc[6] + acc[7]))));
  const int b = (int)(r / T), i = (int)(r % T);
  gate[((long long)b * heads + h) * T + i] = a * (bp * c[h] - 1.f) + 2.f;
}

std::string launch_wavlm_gate(const __nv_bfloat16* x, int B, int T, int heads, const float* w, const float* b,
                              const float* c, float* gate, cudaStream_t s) {
  const long long n = (long long)B * T * heads;
  if (n == 0) return "";
  wavlm_gate_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, (long long)B * T, T, heads, w, b, c, gate);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

}  // namespace w2s

// HF :253-271 (_relative_positions_bucket), in double precision: the float32 logarithm of the reference gives the same
// buckets for |d| < 20000, but the margin is thin (d = 713 lands at 75.99996), so no fast-math or device logarithm.
extern "C" int w2s_relative_buckets(int T, int num_buckets, int max_distance, int32_t* out) {
  const int half = num_buckets / 2, max_exact = half / 2;
  if (T < 1 || !out || max_exact < 1 || max_distance <= max_exact) return 1;
  const double denom = std::log((double)max_distance / max_exact);
  for (int r = 0; r < 2 * T - 1; ++r) {
    const int d = r - (T - 1), a = d < 0 ? -d : d;
    int bucket = d > 0 ? half : 0;
    if (a < max_exact) {
      bucket += a;
    } else {
      const long long large = (long long)(max_exact + std::log((double)a / max_exact) / denom * (half - max_exact));
      bucket += (int)(large < half - 1 ? large : half - 1);
    }
    out[r] = bucket;
  }
  return 0;
}
