// Constant-frame skip of the feature encoder (coalition evaluations with the baseline fill, group-norm front end).
//
// A dropped sample holds the baseline and every layer of the encoder is time-invariant (conv0 + per-(coalition, channel)
// GroupNorm + GELU, then bias-free convolutions + GELU), so a frame whose receptive field lies in dropped samples only
// has one value per (coalition, layer).  conv0 stays dense; for conv1 .. conv6 a 128-row block whose receptive field
// holds no kept segment is not contracted, and the blocks the next layer reads (or, for the last layer, every block)
// get that value copied in from one representative block of the same coalition that the contraction does compute.  A
// contraction row does not depend on where the row sits in its tile, so the copy is bit-identical to the dense row.
#include "../../include/w2s.h"
#include "skip.cuh"

#include <algorithm>
#include <climits>
#include <vector>

namespace w2s {

// ---- per (coalition, layer): live blocks, blocks to fill, representative block --------------------------------------
// One CTA per coalition.  Layers are walked from the last down: a block of layer l is needed when the last layer owns it
// or a live block of layer l + 1 reads it; it is live when its receptive field holds a kept segment, when it is the
// coalition's representative (the first needed block that is all constant), or when the layer runs dense.
__device__ __forceinline__ bool any_kept(const uint32_t* z, int lo, int hi) {
  for (int w = lo >> 5; w <= (hi >> 5); ++w) {
    uint32_t m = z[w];
    if (w == (lo >> 5)) m &= ~0u << (lo & 31);
    if (w == (hi >> 5)) m &= ~0u >> (31 - (hi & 31));
    if (m) return true;
  }
  return false;
}

__global__ void __launch_bounds__(256) skip_lists_kernel(const SkipParams p) {
  extern __shared__ uint8_t sm[];
  uint8_t* nonconst = sm;
  uint8_t* needed = nonconst + p.total;
  uint8_t* live = needed + p.total;
  int* pos = reinterpret_cast<int*>(sm + ((3 * p.total + 15) & ~15));
  __shared__ uint32_t z[64];
  __shared__ int s_rep, s_cnt[2], s_base[2];
  const int b = blockIdx.x;
  const DynArgs* dyn = p.dyn;
  const int zw = dyn->zwords;
  for (int i = threadIdx.x; i < zw; i += blockDim.x) z[i] = dyn->zbits[(long long)b * zw + i];
  __syncthreads();
  for (int i = threadIdx.x; i < p.total; i += blockDim.x) {
    const int4 t = p.tab[i];
    nonconst[i] = any_kept(z, t.x, t.y) ? 1 : 0;
    needed[i] = 0;
    live[i] = 0;
  }
  __syncthreads();
  for (int l = p.nl - 1; l >= 0; --l) {
    const int o = p.off[l], nb = p.nb[l];
    if (threadIdx.x == 0) {
      s_rep = INT_MAX;
      s_cnt[0] = s_cnt[1] = 0;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < nb; j += blockDim.x) {
      if (l == p.nl - 1) needed[o + j] = 1;
      if (needed[o + j] && !nonconst[o + j]) atomicMin(&s_rep, j);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < nb; j += blockDim.x) {
      const bool lv = p.dense[l] || nonconst[o + j] || j == s_rep;
      live[o + j] = lv;
      if (p.dense[l]) continue;
      if (lv) pos[j] = atomicAdd(&s_cnt[0], 1);
      else if (needed[o + j]) pos[j] = atomicAdd(&s_cnt[1], 1);
    }
    __syncthreads();
    if (l > 0) {
      for (int j = threadIdx.x; j < nb; j += blockDim.x) {
        if (!live[o + j]) continue;
        const int4 t = p.tab[o + j];
        for (int i = t.z; i <= t.w; ++i) needed[p.off[l - 1] + i] = 1;
      }
    }
    if (p.dense[l]) continue;   // uniform across the CTA
    if (threadIdx.x == 0) {
      s_base[0] = atomicAdd(p.live[l], s_cnt[0]);
      s_base[1] = atomicAdd(p.fill[l], s_cnt[1]);
      if (s_cnt[1]) p.rep[(long long)l * p.n + b] = s_rep;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < nb; j += blockDim.x) {
      if (live[o + j]) p.live[l][1 + s_base[0] + pos[j]] = (b << 16) | j;
      else if (needed[o + j]) p.fill[l][1 + s_base[1] + pos[j]] = (b << 16) | j;
    }
    __syncthreads();
  }
}

__global__ void skip_reset_kernel(const SkipParams p) {
  const int l = threadIdx.x;
  if (l < p.nl) {
    p.live[l][0] = 0;
    p.fill[l][0] = 0;
  }
}

std::string launch_skip_lists(const SkipParams& p, cudaStream_t s) {
  if (p.n == 0) return "";
  skip_reset_kernel<<<1, 32, 0, s>>>(p);
  W2S_CUDA_OK(cudaGetLastError());
  int maxnb = 0;
  for (int l = 0; l < p.nl; ++l) maxnb = std::max(maxnb, p.nb[l]);
  const size_t smem = (size_t)((3 * p.total + 15) & ~15) + sizeof(int) * maxnb;
  if (smem > 200 * 1024) return "frontend skip: clip too long for the block lists";
  if (smem > 48 * 1024) W2S_CUDA_OK(cudaFuncSetAttribute(skip_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  skip_lists_kernel<<<p.n, 256, smem, s>>>(p);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// ---- fill: every row of each listed block of one layer gets the coalition's representative row --------------------
// 16 bytes per thread; the representative rows (one per coalition) stay in L2.
__global__ void __launch_bounds__(256) skip_fill_kernel(const int* __restrict__ fill, const int* __restrict__ rep,
                                                        __nv_bfloat16* buf, int T, int C) {
  const long long cpr = C / 8;   // 16-byte chunks per row
  const long long per = 128 * cpr;
  const long long total = (long long)fill[0] * per;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long e = i / per, rem = i - e * per;
    const int r = (int)(rem / cpr), c = (int)(rem - (long long)r * cpr);
    const int v = fill[1 + e];
    const int b = v >> 16, row = (v & 0xffff) * 128 + r;
    if (row >= T) continue;
    __nv_bfloat16* base = buf + (long long)b * T * C;
    const uint4 x = *reinterpret_cast<const uint4*>(base + (long long)rep[b] * 128 * C + c * 8);
    *reinterpret_cast<uint4*>(base + (long long)row * C + c * 8) = x;
  }
}

std::string launch_skip_fill(const int* fill, const int* rep, __nv_bfloat16* buf, int T, int C, int num_sms, cudaStream_t s) {
  if (C % 8) return "frontend skip: channel count must be a multiple of 8";
  skip_fill_kernel<<<num_sms * 4, 256, 0, s>>>(fill, rep, buf, T, C);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

}  // namespace w2s

// ---- host block table (include/w2s.h) ---------------------------------------------------------------------------------
int64_t w2s_frontend_blocks(int num_layers, const int32_t* kernel, const int32_t* stride, int64_t L,
                            const int32_t* seg_bounds, int M, int32_t* out, int64_t cap) {
  if (num_layers < 2 || num_layers > W2S_MAX_CONV_LAYERS || L <= 0 || M <= 0 || seg_bounds[0] != 0 || seg_bounds[M] != L)
    return -1;
  for (int m = 0; m < M; ++m)
    if (seg_bounds[m + 1] < seg_bounds[m]) return -1;
  // segment of sample i: the last m with seg_bounds[m] <= i (empty segments own no sample)
  auto seg = [&](int64_t i) { return (int32_t)(std::upper_bound(seg_bounds, seg_bounds + M + 1, i) - seg_bounds) - 1; };
  std::vector<int64_t> T(num_layers);
  int64_t n = L, J = 1, R = 0;
  int64_t rows = 0;
  std::vector<int64_t> Jl(num_layers), Rl(num_layers);
  for (int l = 0; l < num_layers; ++l) {
    if (kernel[l] < 1 || stride[l] < 1 || n < kernel[l]) return -1;
    n = (n - kernel[l]) / stride[l] + 1;
    T[l] = n;
    R = l == 0 ? kernel[0] : R + (int64_t)(kernel[l] - 1) * J;   // receptive field in samples
    J *= stride[l];                                              // hop in samples
    Jl[l] = J;
    Rl[l] = R;
    if (l > 0) rows += (n + 127) / 128;
  }
  if (rows > cap || !out) return rows;
  int64_t k = 0;
  for (int l = 1; l < num_layers; ++l) {
    for (int64_t j = 0; j * 128 < T[l]; ++j, ++k) {
      const int64_t f0 = j * 128, f1 = std::min(f0 + 127, T[l] - 1);
      out[4 * k] = seg(f0 * Jl[l]);
      out[4 * k + 1] = seg(f1 * Jl[l] + Rl[l] - 1);
      out[4 * k + 2] = (int32_t)(f0 * stride[l] / 128);
      out[4 * k + 3] = (int32_t)((f1 * stride[l] + kernel[l] - 1) / 128);
    }
  }
  return rows;
}
