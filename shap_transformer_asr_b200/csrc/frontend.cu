// HBM-bound front of the path: coalition materialisation (K0), conv0 + norm + GELU (K1), LayerNorm,
// positional-conv staging and the one-off weight re-layout kernels.
#include "kernels.cuh"

namespace w2s {

// =================================================================================================
// K0  mask + baseline fill.  One thread = 4 consecutive samples (float4 store, 128 B per 8 lanes).
// Follows feasability_tests/conformer_test.ipynb:138-141 (fill value) with keep-bit convention.
// =================================================================================================
// FILL_BG: global row g = row0 + blockIdx.y is coalition g / B filled from background row g % B (w2s_set_background).
// FILL_BANDS: `bg` holds the B = F band components (row stride bg_ld) and bit s * F + b of the row keeps cell (s, b); the
// clip and the baseline are not read.
template <int FILL>
__global__ void __launch_bounds__(256) mask_kernel(const float* __restrict__ x, const uint16_t* __restrict__ seg_id,
                                                    const uint32_t* __restrict__ zbits, int zwords, long long L,
                                                    float baseline, float* __restrict__ out, long long ld,
                                                    const float* __restrict__ bg, int B, long long bg_ld, long long row0) {
  constexpr bool BG = FILL == FILL_BG;
  __shared__ uint32_t z[64];
  const long long g = BG ? row0 + blockIdx.y : blockIdx.y;
  const long long k = BG ? g / B : g;
  if (threadIdx.x < zwords) z[threadIdx.x] = zbits[k * zwords + threadIdx.x];
  __syncthreads();
  const long long i0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i0 >= L) return;
  float* o = out + g * ld + i0;
  if constexpr (FILL == FILL_BANDS) {
    const int F = B;
    auto keep = [&](uint32_t sgm, int b) { const uint32_t c = sgm * F + b; return (z[c >> 5] >> (c & 31)) & 1u; };
    if (i0 + 4 <= L && ((ld & 3) == 0) && (bg_ld & 3) == 0) {
      const ushort4 sv = *reinterpret_cast<const ushort4*>(seg_id + i0);
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int b = 0; b < F; ++b) {
        const float4 cv = *reinterpret_cast<const float4*>(bg + b * bg_ld + i0);
        r.x += keep(sv.x, b) ? cv.x : 0.f;
        r.y += keep(sv.y, b) ? cv.y : 0.f;
        r.z += keep(sv.z, b) ? cv.z : 0.f;
        r.w += keep(sv.w, b) ? cv.w : 0.f;
      }
      *reinterpret_cast<float4*>(o) = r;
    } else {
      for (int j = 0; j < 4 && i0 + j < L; ++j) {
        const uint32_t sgm = seg_id[i0 + j];
        float v = 0.f;
        for (int b = 0; b < F; ++b) v += keep(sgm, b) ? bg[b * bg_ld + i0 + j] : 0.f;
        o[j] = v;
      }
    }
    return;
  }
  const float* f = BG ? bg + (g - k * B) * bg_ld : nullptr;
  if (i0 + 4 <= L && ((ld & 3) == 0) && (!BG || (bg_ld & 3) == 0)) {
    const float4 xv = *reinterpret_cast<const float4*>(x + i0);
    const ushort4 sv = *reinterpret_cast<const ushort4*>(seg_id + i0);
    float4 fv;
    if constexpr (BG) fv = *reinterpret_cast<const float4*>(f + i0);
    else fv = make_float4(baseline, baseline, baseline, baseline);
    float4 r;
    r.x = (z[sv.x >> 5] >> (sv.x & 31)) & 1u ? xv.x : fv.x;
    r.y = (z[sv.y >> 5] >> (sv.y & 31)) & 1u ? xv.y : fv.y;
    r.z = (z[sv.z >> 5] >> (sv.z & 31)) & 1u ? xv.z : fv.z;
    r.w = (z[sv.w >> 5] >> (sv.w & 31)) & 1u ? xv.w : fv.w;
    *reinterpret_cast<float4*>(o) = r;
  } else {
    for (int j = 0; j < 4 && i0 + j < L; ++j) {
      const uint32_t sgm = seg_id[i0 + j];
      o[j] = (z[sgm >> 5] >> (sgm & 31)) & 1u ? x[i0 + j] : (BG ? f[i0 + j] : baseline);
    }
  }
}

std::string launch_mask(const float* x, const uint16_t* seg_id, const uint32_t* zbits, int zwords, long long K,
                        long long L, float baseline, float* out, long long ld, cudaStream_t s) {
  if (zwords > 64) return "mask: more than 2048 segments are not supported";
  if (K == 0) return "";
  dim3 grid((unsigned)((L + 1023) / 1024), (unsigned)K);
  W2S_CUDA_OK(launch_pdl(mask_kernel<FILL_PLAIN>, grid, dim3(256), 0, s, 1, x, seg_id, zbits, zwords, L, baseline, out, ld,
                         (const float*)nullptr, 0, 0LL, 0LL));
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

std::string launch_mask_bg(const float* x, const uint16_t* seg_id, const uint32_t* zbits, int zwords, long long K,
                           long long L, const float* bg, int B, long long bg_ld, float* out, long long ld, cudaStream_t s) {
  if (zwords > 64) return "mask: more than 2048 segments are not supported";
  const long long rows = K * B;
  for (long long r0 = 0; r0 < rows; r0 += 65535) {   // grid.y limit
    const long long n = rows - r0 < 65535 ? rows - r0 : 65535;
    dim3 grid((unsigned)((L + 1023) / 1024), (unsigned)n);
    W2S_CUDA_OK(launch_pdl(mask_kernel<FILL_BG>, grid, dim3(256), 0, s, 1, x, seg_id, zbits, zwords, L, 0.f, out, ld, bg, B,
                           bg_ld, r0));
    W2S_CUDA_OK(cudaGetLastError());
  }
  return "";
}

std::string launch_mask_bands(const uint16_t* seg_id, const uint32_t* zbits, int zwords, long long K, long long L,
                              const float* comp, int F, long long comp_ld, float* out, long long ld, cudaStream_t s) {
  if (zwords > 64) return "mask: more than 2048 cells are not supported";
  for (long long k0 = 0; k0 < K; k0 += 65535) {   // grid.y limit
    const long long n = K - k0 < 65535 ? K - k0 : 65535;
    dim3 grid((unsigned)((L + 1023) / 1024), (unsigned)n);
    W2S_CUDA_OK(launch_pdl(mask_kernel<FILL_BANDS>, grid, dim3(256), 0, s, 1, (const float*)nullptr, seg_id,
                           zbits + k0 * zwords, zwords, L, 0.f, out + k0 * ld, ld, comp, F, comp_ld, 0LL));
    W2S_CUDA_OK(cudaGetLastError());
  }
  return "";
}

// The same selection folded into a consumer's load: `zs` is the coalition's bit row staged in shared memory.  FILL_BG:
// dropped samples come from a background row instead of the constant; FILL_BANDS: sample i is the sum over bands b of
// component b where cell (seg(i), b) is kept (compile-time variants, so that the baseline-fill kernels keep their code).
template <int FILL = FILL_PLAIN>
struct WaveRow {
  const float* x;        // FILL_BANDS: the band components, rows `ld` apart
  const uint16_t* seg;   // null: plain waveform row
  const uint32_t* zs;
  float baseline;
  const float* fill;     // FILL_BG: background row
  long long ld;          // FILL_BANDS
  int F;                 // FILL_BANDS
  __device__ __forceinline__ float at(long long i) const {
    if constexpr (FILL == FILL_BANDS) {
      // one L2-resident load and one shared-memory bit test per band; fp32 adds in band order from +0.0
      const uint32_t c0 = (uint32_t)__ldg(seg + i) * (uint32_t)F;
      float v = 0.f;
      for (int b = 0; b < F; ++b) {
        const uint32_t c = c0 + b;
        const float t = __ldg(x + b * ld + i);
        v += (zs[c >> 5] >> (c & 31)) & 1u ? t : 0.f;
      }
      return v;
    } else {
      const float v = __ldg(x + i);
      if constexpr (FILL == FILL_BG) {
        const uint32_t sgm = __ldg(seg + i);
        return (zs[sgm >> 5] >> (sgm & 31)) & 1u ? v : __ldg(fill + i);
      } else {
        if (!seg) return v;
        const uint32_t sgm = __ldg(seg + i);
        return (zs[sgm >> 5] >> (sgm & 31)) & 1u ? v : baseline;
      }
    }
  }
};
// Row `row` of the tile described by the per-call argument block; ends with a CTA-wide barrier.  FILL_BG: tile row r is
// global row g = row0 + r of the call, coalition g / B with background row g % B.  FILL_BANDS: tile row r is coalition r,
// its bit row has one bit per time-frequency cell.
template <int FILL = FILL_PLAIN>
__device__ __forceinline__ WaveRow<FILL> wave_row(const DynArgs* __restrict__ dyn, int row, uint32_t* zs) {
  WaveRow<FILL> w;
  w.zs = zs;
  if constexpr (FILL == FILL_BG) {
    const long long g = dyn->row0 + row, B = dyn->B, k = g / B;
    const int zw = dyn->zwords;
    for (int i = threadIdx.x; i < zw; i += blockDim.x) zs[i] = dyn->zbits[k * zw + i];
    w.x = dyn->clip; w.seg = dyn->seg_id; w.baseline = 0.f;
    w.fill = dyn->bg + (g - k * B) * dyn->ld;
  } else if constexpr (FILL == FILL_BANDS) {
    const int zw = dyn->zwords;
    for (int i = threadIdx.x; i < zw; i += blockDim.x) zs[i] = dyn->zbits[(long long)row * zw + i];
    w.x = dyn->bands; w.seg = dyn->seg_id; w.ld = dyn->ld; w.F = dyn->F;
  } else if (dyn->clip) {
    const int zw = dyn->zwords;
    for (int i = threadIdx.x; i < zw; i += blockDim.x) zs[i] = dyn->zbits[(long long)row * zw + i];
    w.x = dyn->clip; w.seg = dyn->seg_id; w.baseline = dyn->baseline;
  } else {
    w.x = dyn->x + (long long)row * dyn->ld; w.seg = nullptr; w.baseline = 0.f;
  }
  __syncthreads();
  return w;
}

// =================================================================================================
// K1a  GroupNorm statistics of conv0 output without materialising it.
// conv0 is linear and bias-free under GroupNorm (a conv bias cancels in y - mean), so per waveform row
//   sum_t y[t,c]   = sum_j w[c,j] S[j],        S[j]    = sum_t x[s t + j]
//   sum_t y[t,c]^2 = sum_jj' w[c,j] w[c,j'] R[j,j'],  R[j,j'] = sum_t x[s t + j] x[s t + j']
// (HF wav2vec2/modeling_wav2vec2.py:302-323: GroupNorm(num_groups=C) normalises each channel over time).
// One CTA per waveform row.  The 65 sums are accumulated in fp64 from the first product on (the product of two fp32
// samples is exact in fp64): for low-pass input under a high-pass / band-pass filter the quadratic form w^T R w cancels
// by many orders of magnitude, and fp32 partial sums lose percent-level accuracy in the variance there.
// =================================================================================================
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int KW, int FILL>
__global__ void __launch_bounds__(256, 1) conv0_stats_kernel(const Conv0Params p) {
  constexpr int NR = KW * (KW + 1) / 2;
  constexpr int NACC = KW + NR;
  __shared__ double red[8][NACC];
  __shared__ double tot[NACC];
  __shared__ uint32_t zs[64];
  const int row = blockIdx.x;
  const WaveRow<FILL> x = wave_row<FILL>(p.dyn, row, zs);
  double acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.0;
  for (int t = threadIdx.x; t < p.T0; t += blockDim.x) {
    double xv[KW];
    const long long i0 = (long long)t * p.stride;
#pragma unroll
    for (int j = 0; j < KW; ++j) xv[j] = (double)x.at(i0 + j);
    int r = KW;
#pragma unroll
    for (int j = 0; j < KW; ++j) {
      acc[j] += xv[j];
#pragma unroll
      for (int jj = j; jj < KW; ++jj) {
        acc[r] = fma(xv[j], xv[jj], acc[r]);
        ++r;
      }
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < NACC; ++i) {
    const double v = warp_sum_f64(acc[i]);
    if (lane == 0) red[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < NACC) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
    tot[threadIdx.x] = s;
  }
  __syncthreads();
  const double invT = 1.0 / (double)p.T0;
  for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
    double wj[KW];
#pragma unroll
    for (int j = 0; j < KW; ++j) wj[j] = (double)p.w[c * KW + j];
    double sum = 0.0, sq = 0.0;
    int r = KW;
#pragma unroll
    for (int j = 0; j < KW; ++j) {
      sum += wj[j] * tot[j];
#pragma unroll
      for (int jj = j; jj < KW; ++jj) {
        const double term = wj[j] * wj[jj] * tot[r++];
        sq += (jj == j) ? term : 2.0 * term;
      }
    }
    const double mean = sum * invT;
    double var = sq * invT - mean * mean;
    if (var < 0.0) var = 0.0;
    const double rstd = rsqrt(var + 1e-5);
    const double a = rstd * (double)p.gamma[c];
    const float shift = (float)((double)p.beta[c] - mean * a);
    p.gn_a[(long long)row * p.C + c] = (float)a;
    p.gn_b[(long long)row * p.C + c] = shift;
    if (p.gn_wb) {
      // K = 32 row of the tensor-core form: y = sum_k A[f][k] B[c][k] with A[f] = [x_hi | x_lo | x_hi | 1 1] and
      // B[c] = [w_hi | w_hi | w_lo | shift_hi shift_lo], w = filter * rstd * gamma (the lo*lo term, ~2^-18, is dropped)
      static_assert(3 * KW + 2 == 32, "K layout of conv0_mma_kernel");
      __align__(16) __nv_bfloat16 kb[32];
#pragma unroll
      for (int j = 0; j < KW; ++j) {
        const float wf = (float)(wj[j] * a);
        const __nv_bfloat16 hi = __float2bfloat16_rn(wf);
        kb[j] = hi;
        kb[KW + j] = hi;
        kb[2 * KW + j] = __float2bfloat16_rn(wf - __bfloat162float(hi));
      }
      kb[30] = __float2bfloat16_rn(shift);
      kb[31] = __float2bfloat16_rn(shift - __bfloat162float(kb[30]));
      uint4* dst = reinterpret_cast<uint4*>(p.gn_wb + ((long long)row * p.C + c) * 32);
#pragma unroll
      for (int q = 0; q < 4; ++q) dst[q] = reinterpret_cast<const uint4*>(kb)[q];
    }
  }
}

std::string launch_conv0_stats(const Conv0Params& p, cudaStream_t s, int fill) {
  if (p.kw != 10) return "conv0: only kernel width 10 is implemented for layer 0";
  if (p.n == 0) return "";
  if (fill == FILL_BANDS) W2S_CUDA_OK(launch_pdl(conv0_stats_kernel<10, FILL_BANDS>, dim3(p.n), dim3(256), 0, s, 1, p));
  else if (fill == FILL_BG) W2S_CUDA_OK(launch_pdl(conv0_stats_kernel<10, FILL_BG>, dim3(p.n), dim3(256), 0, s, 1, p));
  else W2S_CUDA_OK(launch_pdl(conv0_stats_kernel<10, FILL_PLAIN>, dim3(p.n), dim3(256), 0, s, 1, p));
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// =================================================================================================
// K1b  conv0 + norm + GELU, channels-last bf16 output [n, T0, C].
// CTA = (frame tile of FT frames, waveform row).  The waveform window is staged in shared memory once;
// each thread owns 8 consecutive channels (one 16-byte store per frame) and keeps their 10-tap filters and
// affine constants in registers; all lanes of a warp work on the same frame, so window reads broadcast.
// HF wav2vec2/modeling_wav2vec2.py:302-323 (group) / :275-299 (layer).
// =================================================================================================
template <int KW, bool LAYER, int FILL>
__global__ void __launch_bounds__(256, 2) conv0_kernel(const Conv0Params p, int FT) {
  extern __shared__ float sm[];
  float* xs = sm;                      // FT*stride + KW window
  float* fmean = xs + FT * p.stride + KW;  // [FT] (layer variant)
  float* frstd = fmean + FT;
  float2* xs2 = reinterpret_cast<float2*>(frstd + FT + ((FT * p.stride + KW) & 1));  // (x, x) pairs, 8-byte aligned
  __shared__ uint32_t zs[64];
  const int row = blockIdx.y;
  const int f0 = blockIdx.x * FT;
  const int nf = min(FT, p.T0 - f0);
  const WaveRow<FILL> x = wave_row<FILL>(p.dyn, row, zs);
  const long long x0 = (long long)f0 * p.stride;
  const int nwin = (nf - 1) * p.stride + KW;
  for (int i = threadIdx.x; i < nwin; i += blockDim.x) {
    const float t = x.at(x0 + i);
    xs[i] = t;
    xs2[i] = make_float2(t, t);
  }
  __syncthreads();

  if constexpr (LAYER) {
    // per-frame statistics over channels from the 10-sample window (quadratic form with the filter Gram matrix)
    for (int f = threadIdx.x; f < nf; f += blockDim.x) {
      float xv[KW];
#pragma unroll
      for (int j = 0; j < KW; ++j) xv[j] = xs[f * p.stride + j];
      float mean = p.ln_bmean, ex2 = p.ln_b2mean;
#pragma unroll
      for (int j = 0; j < KW; ++j) {
        mean = fmaf(p.ln_wbar[j], xv[j], mean);
        ex2 = fmaf(2.0f * p.ln_wb[j], xv[j], ex2);
        float gj = 0.f;
#pragma unroll
        for (int jj = 0; jj < KW; ++jj) gj = fmaf(p.ln_gram[j * KW + jj], xv[jj], gj);
        ex2 = fmaf(gj, xv[j], ex2);
      }
      const float var = fmaxf(ex2 - mean * mean, 0.f);
      fmean[f] = mean;
      frstd[f] = rsqrtf(var + 1e-5f);
    }
    __syncthreads();
  }

  const int tpf = p.C >> 3;            // threads per frame
  const int fpar = blockDim.x / tpf;   // frames in flight per CTA
  const int c0 = (threadIdx.x % tpf) * 8;
  const int fslot = threadIdx.x / tpf;
  // channel pairs on the packed fp32 pipe: (y[2i], y[2i+1]) += (w[2i][j], w[2i+1][j]) * (x[j], x[j])
  float2 w2[4][KW], ca2[4], cb2[4], bias2[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int j = 0; j < KW; ++j)
      w2[i][j] = make_float2(__ldg(p.w + (c0 + 2 * i) * KW + j), __ldg(p.w + (c0 + 2 * i + 1) * KW + j));
    if constexpr (LAYER) {
      ca2[i] = make_float2(__ldg(p.gamma + c0 + 2 * i), __ldg(p.gamma + c0 + 2 * i + 1));
      cb2[i] = make_float2(__ldg(p.beta + c0 + 2 * i), __ldg(p.beta + c0 + 2 * i + 1));
      bias2[i] = p.bias ? make_float2(__ldg(p.bias + c0 + 2 * i), __ldg(p.bias + c0 + 2 * i + 1)) : make_float2(0.f, 0.f);
    } else {
      const float* ga = p.gn_a + (long long)row * p.C + c0 + 2 * i;
      const float* gb = p.gn_b + (long long)row * p.C + c0 + 2 * i;
      // group norm is affine per (row, channel): fold it into the filters, the accumulator starts at the shift
      ca2[i] = make_float2(ga[0], ga[1]);
      bias2[i] = make_float2(gb[0], gb[1]);
#pragma unroll
      for (int j = 0; j < KW; ++j) w2[i][j] = __fmul2_rn(w2[i][j], ca2[i]);
    }
  }

  __nv_bfloat16* out = p.out + ((long long)row * p.T0 + f0) * p.C + c0;
  for (int f = fslot; f < nf; f += fpar) {
    float2 xv[KW];
#pragma unroll
    for (int j = 0; j < KW; ++j) xv[j] = xs2[f * p.stride + j];
    uint32_t packed[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 a = bias2[i];
#pragma unroll
      for (int j = 0; j < KW; ++j) a = __ffma2_rn(w2[i][j], xv[j], a);
      if constexpr (LAYER) {
        const float m = fmean[f], r = frstd[f];
        a = __ffma2_rn(__fmul2_rn(__fadd2_rn(a, make_float2(-m, -m)), make_float2(r, r)), ca2[i], cb2[i]);
      }
      const float2 y = gelu_erf2(a);
      packed[i] = pack_bf16x2(y.x, y.y);
    }
    *reinterpret_cast<uint4*>(out + (long long)f * p.C) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
  }
}

// Group-norm variant on the warp-level tensor cores.  After the bf16 hi/lo split the whole layer, affine included, is
// one K = 32 contraction per (frame, channel) (layout in conv0_stats_kernel); what is left for the FP32 pipes is the
// GELU.  CTA = (FT frames, waveform row): the im2col rows [FT][32] are built once in shared memory (80-byte pitch:
// conflict-free ldmatrix), each warp owns 64 channels whose B fragments stay in registers, and the channel
// permutation inside a warp is chosen so that a thread ends up with 8 consecutive channels per (frame, half):
// one 16-byte store, 64 contiguous bytes per quad.
template <int KW, bool PRE, int FILL>
__global__ void __launch_bounds__(256, 2) conv0_mma_kernel(const Conv0Params p, int FT) {
  extern __shared__ __align__(16) uint8_t im2col[];
  constexpr int LDA = 80;
  static_assert(3 * KW + 2 == 32, "K layout");
  __shared__ uint32_t zs[64];
  const int row = blockIdx.y;
  const int f0 = blockIdx.x * FT;
  const int nf = min(FT, p.T0 - f0);
  const int nfp = (nf + 15) & ~15;
  const WaveRow<FILL> x = wave_row<FILL>(p.dyn, row, zs);
  const long long x0 = (long long)f0 * p.stride;
  for (int i = threadIdx.x; i < nfp * KW; i += blockDim.x) {
    const int f = i / KW, j = i - f * KW;
    const float v = f < nf ? x.at(x0 + f * p.stride + j) : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    __nv_bfloat16* ar = reinterpret_cast<__nv_bfloat16*>(im2col + f * LDA);
    ar[j] = hi;
    ar[KW + j] = lo;
    ar[2 * KW + j] = hi;
    if (j == 0) *reinterpret_cast<uint32_t*>(ar + 3 * KW) = 0x3f803f80u;  // (1, 1): picks up the shift terms
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  uint32_t bfrag[8][2][2];
  {
    const __nv_bfloat16* wb = p.gn_wb + (long long)row * p.C * 32;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int ch = warp * 64 + (nt >> 2) * 32 + (g >> 1) * 8 + (nt & 3) * 2 + (g & 1);
      const uint32_t* wr = reinterpret_cast<const uint32_t*>(wb + (long long)ch * 32);
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        bfrag[nt][ks][0] = wr[8 * ks + t];
        bfrag[nt][ks][1] = wr[8 * ks + t + 4];
      }
    }
  }
  __syncthreads();
  const uint32_t a_base = smem_u32(im2col) + (lane & 15) * LDA + (lane >> 4) * 16;
  __nv_bfloat16* out = p.out + ((long long)row * p.T0 + f0) * p.C + warp * 64 + t * 8;
  for (int mb = 0; mb * 16 < nf; ++mb) {
    uint32_t a[2][4];
    ldmatrix_x4(a[0], a_base + mb * 16 * LDA);
    ldmatrix_x4(a[1], a_base + mb * 16 * LDA + 32);
    float c[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
      mma_bf16_16816(c[nt], a[0], bfrag[nt][0]);
      mma_bf16_16816(c[nt], a[1], bfrag[nt][1]);
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int f = mb * 16 + g + 8 * r;
      if (f < nf) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t pk[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 a = make_float2(c[4 * h + q][2 * r], c[4 * h + q][2 * r + 1]);
            const float2 y = PRE ? a : gelu_erf2(a);
            pk[q] = pack_bf16x2(y.x, y.y);
          }
          *reinterpret_cast<uint4*>(out + (long long)f * p.C + h * 32) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
    }
  }
}

// Layer-norm variant (feat_extract_norm = "layer": wav2vec2-large-lv60, the conformer checkpoints) in the same tensor-core
// form.  Per frame f the LayerNorm over channels is affine in the conv output,
//   y[f,c] = rstd_f gamma_c (sum_j w[c,j] x[f,j]) + rstd_f (gamma_c b_c) + (rstd_f mean_f)(-gamma_c) + beta_c,
// so with the frame's rstd folded into the im2col row the whole layer is ONE K = 48 contraction whose B operand is a
// constant of the model (built once at create by conv0_ln_b_kernel):
//   A[f] = [xs_hi | xs_lo | xs_hi | r_hi r_lo r_hi | q_hi q_lo q_hi | 1 1 | 0...],  xs = rstd_f x,  r = rstd_f,  q = rstd_f mean_f
//   B[c] = [gw_hi | gw_hi | gw_lo | t_hi t_hi t_lo | u_hi u_hi u_lo | beta_hi beta_lo | 0...],  gw = gamma_c w[c,:],  t = gamma_c b_c,  u = -gamma_c
// (bf16 hi + lo terms; the lo x lo products, ~2^-18 relative, are dropped).  The frame statistics come from the 10-sample
// window through the Gram matrix of the filter bank, as in the CUDA-core kernel this replaces.
constexpr int C0L_K = 48, C0L_LDA = 112;   // 112-byte row pitch: 7 x 16 B, conflict-free ldmatrix

template <int KW, bool PRE, int FILL>
__global__ void __launch_bounds__(256, 2) conv0_ln_mma_kernel(const Conv0Params p, int FT) {
  extern __shared__ __align__(16) uint8_t smem_ln[];
  __shared__ uint32_t zs[64];
  uint8_t* im2col = smem_ln;                                             // [FT][112 B]
  float* xs = reinterpret_cast<float*>(smem_ln + (size_t)FT * C0L_LDA);   // FT * stride + KW samples
  const int row = blockIdx.y;
  const int f0 = blockIdx.x * FT;
  const int nf = min(FT, p.T0 - f0);
  const int nfp = (nf + 15) & ~15;
  const WaveRow<FILL> x = wave_row<FILL>(p.dyn, row, zs);
  const long long x0 = (long long)f0 * p.stride;
  const int nwin = (nf - 1) * p.stride + KW;
  for (int i = threadIdx.x; i < nwin; i += blockDim.x) xs[i] = x.at(x0 + i);
  __syncthreads();
  for (int f = threadIdx.x; f < nfp; f += blockDim.x) {
    __nv_bfloat16* ar = reinterpret_cast<__nv_bfloat16*>(im2col + (size_t)f * C0L_LDA);
    if (f >= nf) {
#pragma unroll
      for (int q = 0; q < C0L_K / 8; ++q) reinterpret_cast<uint4*>(ar)[q] = make_uint4(0u, 0u, 0u, 0u);
      continue;
    }
    float xv[KW];
#pragma unroll
    for (int j = 0; j < KW; ++j) xv[j] = xs[f * p.stride + j];
    // channel statistics of the conv output of this frame (quadratic form with the filter Gram matrix)
    float mean = p.ln_bmean, ex2 = p.ln_b2mean;
#pragma unroll
    for (int j = 0; j < KW; ++j) {
      mean = fmaf(p.ln_wbar[j], xv[j], mean);
      ex2 = fmaf(2.0f * p.ln_wb[j], xv[j], ex2);
      float gj = 0.f;
#pragma unroll
      for (int jj = 0; jj < KW; ++jj) gj = fmaf(p.ln_gram[j * KW + jj], xv[jj], gj);
      ex2 = fmaf(gj, xv[j], ex2);
    }
    const float rstd = rsqrtf(fmaxf(ex2 - mean * mean, 0.f) + 1e-5f);
    if (PRE && p.ln_rstd_out) p.ln_rstd_out[(long long)row * p.T0 + f0 + f] = rstd;   // kept for the backward pass
    auto split3 = [&](float v, int at) {   // (hi, lo, hi): pairs with (hi, hi, lo) on the B side
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      ar[at] = hi;
      ar[at + 1] = __float2bfloat16_rn(v - __bfloat162float(hi));
      ar[at + 2] = hi;
    };
#pragma unroll
    for (int j = 0; j < KW; ++j) {
      const float v = rstd * xv[j];
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      ar[j] = hi;
      ar[KW + j] = __float2bfloat16_rn(v - __bfloat162float(hi));
      ar[2 * KW + j] = hi;
    }
    split3(rstd, 3 * KW);
    split3(rstd * mean, 3 * KW + 3);
    ar[3 * KW + 6] = __float2bfloat16_rn(1.f);
    ar[3 * KW + 7] = __float2bfloat16_rn(1.f);
#pragma unroll
    for (int k = 3 * KW + 8; k < C0L_K; ++k) ar[k] = __float2bfloat16_rn(0.f);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  uint32_t bfrag[8][3][2];
  {
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int ch = warp * 64 + (nt >> 2) * 32 + (g >> 1) * 8 + (nt & 3) * 2 + (g & 1);
      const uint32_t* wr = reinterpret_cast<const uint32_t*>(p.ln_wb48 + (long long)ch * C0L_K);
#pragma unroll
      for (int ks = 0; ks < 3; ++ks) {
        bfrag[nt][ks][0] = __ldg(wr + 8 * ks + t);
        bfrag[nt][ks][1] = __ldg(wr + 8 * ks + t + 4);
      }
    }
  }
  __syncthreads();
  const uint32_t a_base = smem_u32(im2col) + (lane & 15) * C0L_LDA + (lane >> 4) * 16;
  __nv_bfloat16* out = p.out + ((long long)row * p.T0 + f0) * p.C + warp * 64 + t * 8;
  for (int mb = 0; mb * 16 < nf; ++mb) {
    uint32_t a[3][4];
#pragma unroll
    for (int ks = 0; ks < 3; ++ks) ldmatrix_x4(a[ks], a_base + mb * 16 * C0L_LDA + ks * 32);
    float c[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 3; ++ks) mma_bf16_16816(c[nt], a[ks], bfrag[nt][ks]);
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int f = mb * 16 + g + 8 * r;
      if (f < nf) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t pk[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 a = make_float2(c[4 * h + q][2 * r], c[4 * h + q][2 * r + 1]);
            const float2 y = PRE ? a : gelu_erf2(a);
            pk[q] = pack_bf16x2(y.x, y.y);
          }
          *reinterpret_cast<uint4*>(out + (long long)f * p.C + h * 32) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
    }
  }
}

// B operand of conv0_ln_mma_kernel: [C][48] bf16, a constant of the model (run once at create)
__global__ void conv0_ln_b_kernel(const float* w, const float* bias, const float* gamma, const float* beta, int C, int kw,
                                  __nv_bfloat16* out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  __nv_bfloat16* o = out + (long long)c * C0L_K;
  auto hi = [](float v) { return __float2bfloat16_rn(v); };
  auto lo = [](float v) { return __float2bfloat16_rn(v - __bfloat162float(__float2bfloat16_rn(v))); };
  const float g = gamma[c];
  for (int j = 0; j < kw; ++j) {
    const float v = g * w[c * kw + j];
    o[j] = hi(v);
    o[kw + j] = hi(v);
    o[2 * kw + j] = lo(v);
  }
  const float t = g * (bias ? bias[c] : 0.f), u = -g;
  o[3 * kw] = hi(t); o[3 * kw + 1] = hi(t); o[3 * kw + 2] = lo(t);
  o[3 * kw + 3] = hi(u); o[3 * kw + 4] = hi(u); o[3 * kw + 5] = lo(u);
  o[3 * kw + 6] = hi(beta[c]); o[3 * kw + 7] = lo(beta[c]);
  for (int k = 3 * kw + 8; k < C0L_K; ++k) o[k] = __float2bfloat16_rn(0.f);
}
std::string launch_conv0_ln_b(const float* w, const float* bias, const float* gamma, const float* beta, int C, int kw,
                              __nv_bfloat16* out, cudaStream_t s) {
  if (3 * kw + 8 > C0L_K) return "conv0 (layer norm): kernel too wide for the K = 48 form";
  conv0_ln_b_kernel<<<(C + 127) / 128, 128, 0, s>>>(w, bias, gamma, beta, C, kw, out);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// The gradient path's pre-activation variants (PRE = true) exist for the plain and background fills only: time-frequency
// cells are an evaluation-path input.
template <int FILL>
std::string launch_conv0_t(const Conv0Params& p, bool layer_norm, cudaStream_t s) {
  constexpr bool kPre = FILL != FILL_BANDS;
  if (!kPre && p.pre_act) return "conv0: the band-cell fill has no pre-activation variant";
  if (!layer_norm && p.gn_wb && p.C % 64 == 0 && p.C <= 512 && p.n > 0) {
    const int FT = 512;
    dim3 grid((p.T0 + FT - 1) / FT, p.n);
    if constexpr (kPre) {
      if (p.pre_act) W2S_CUDA_OK(launch_pdl(conv0_mma_kernel<10, true, FILL>, grid, dim3(p.C / 2), (size_t)FT * 80, s, 1, p, FT));
      else W2S_CUDA_OK(launch_pdl(conv0_mma_kernel<10, false, FILL>, grid, dim3(p.C / 2), (size_t)FT * 80, s, 1, p, FT));
    } else {
      W2S_CUDA_OK(launch_pdl(conv0_mma_kernel<10, false, FILL>, grid, dim3(p.C / 2), (size_t)FT * 80, s, 1, p, FT));
    }
    W2S_CUDA_OK(cudaGetLastError());
    return "";
  }
  if (layer_norm && p.ln_wb48 && p.C % 64 == 0 && p.C <= 512 && p.n > 0) {
    const int FT = 512;
    const size_t smem = (size_t)FT * C0L_LDA + (size_t)(FT * p.stride + p.kw + 4) * sizeof(float);
    static bool attr = false;
    if (!attr) {
      W2S_CUDA_OK(cudaFuncSetAttribute(conv0_ln_mma_kernel<10, false, FILL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      if constexpr (kPre)
        W2S_CUDA_OK(cudaFuncSetAttribute(conv0_ln_mma_kernel<10, true, FILL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      attr = true;
    }
    if (smem > 100 * 1024) return "conv0 (layer norm): stride too large for the staged window";
    dim3 grid((p.T0 + FT - 1) / FT, p.n);
    if constexpr (kPre) {
      if (p.pre_act) W2S_CUDA_OK(launch_pdl(conv0_ln_mma_kernel<10, true, FILL>, grid, dim3(p.C / 2), smem, s, 1, p, FT));
      else W2S_CUDA_OK(launch_pdl(conv0_ln_mma_kernel<10, false, FILL>, grid, dim3(p.C / 2), smem, s, 1, p, FT));
    } else {
      W2S_CUDA_OK(launch_pdl(conv0_ln_mma_kernel<10, false, FILL>, grid, dim3(p.C / 2), smem, s, 1, p, FT));
    }
    W2S_CUDA_OK(cudaGetLastError());
    return "";
  }
  const int tpf = p.C / 8;
  if (p.C % 8 || tpf > 256 || (256 % tpf)) return "conv0: channel count must be 8 * (a divisor of 256)";
  if (p.n == 0) return "";
  const int FT = p.T0 >= 4096 ? 512 : 128;
  dim3 grid((p.T0 + FT - 1) / FT, p.n);
  const size_t smem = (size_t)(3 * (FT * p.stride + p.kw) + 2 * FT + 2) * sizeof(float);
  if (layer_norm) W2S_CUDA_OK(launch_pdl(conv0_kernel<10, true, FILL>, grid, dim3(256), smem, s, 1, p, FT));
  else W2S_CUDA_OK(launch_pdl(conv0_kernel<10, false, FILL>, grid, dim3(256), smem, s, 1, p, FT));
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

std::string launch_conv0(const Conv0Params& p, bool layer_norm, cudaStream_t s, int fill) {
  if (p.kw != 10) return "conv0: only kernel width 10 is implemented for layer 0";
  if (fill == FILL_BANDS) return launch_conv0_t<FILL_BANDS>(p, layer_norm, s);
  return fill == FILL_BG ? launch_conv0_t<FILL_BG>(p, layer_norm, s) : launch_conv0_t<FILL_PLAIN>(p, layer_norm, s);
}

// filter-bank statistics for the layer-norm variant: one CTA, trivially small
__global__ void conv0_ln_prep_kernel(const float* w, const float* bias, int C, int kw, float* wbar, float* gram,
                                     float* wb, float* scalars) {
  const int t = threadIdx.x;
  if (t < kw * kw) {
    const int j = t / kw, jj = t % kw;
    double s = 0.0;
    for (int c = 0; c < C; ++c) s += (double)w[c * kw + j] * (double)w[c * kw + jj];
    gram[t] = (float)(s / C);
  }
  if (t < kw) {
    double s = 0.0, sb = 0.0;
    for (int c = 0; c < C; ++c) {
      s += (double)w[c * kw + t];
      if (bias) sb += (double)w[c * kw + t] * (double)bias[c];
    }
    wbar[t] = (float)(s / C);
    wb[t] = (float)(sb / C);
  }
  if (t == 0) {
    double s = 0.0, s2 = 0.0;
    if (bias)
      for (int c = 0; c < C; ++c) {
        s += (double)bias[c];
        s2 += (double)bias[c] * (double)bias[c];
      }
    scalars[0] = (float)(s / C);
    scalars[1] = (float)(s2 / C);
  }
}
std::string launch_conv0_ln_prep(const float* w, const float* bias, int C, int kw, float* wbar, float* gram,
                                 float* wb, float* scalars, cudaStream_t s) {
  if (kw * kw > 256) return "conv0 prep: kernel too wide";
  conv0_ln_prep_kernel<<<1, 256, 0, s>>>(w, bias, C, kw, wbar, gram, wb, scalars);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// =================================================================================================
// LayerNorm over the last dimension, one warp per row, values held in registers (H <= 1024),
// fp32 statistics (two-pass), optional activation, bf16 (and optional fp32) output.
// =================================================================================================
template <bool IN_F32>
__global__ void __launch_bounds__(256) layernorm_kernel(const void* __restrict__ in, long long rows, int H,
                                                         const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, float eps, int act,
                                                         __nv_bfloat16* __restrict__ out, float* __restrict__ out_f32) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  constexpr int MAXV = 32;
  float v[MAXV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    float t = 0.f;
    if (idx < H) {
      if constexpr (IN_F32) t = reinterpret_cast<const float*>(in)[row * H + idx];
      else t = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(in)[row * H + idx]);
    }
    v[i] = t;
    sum += t;
  }
  const float mean = warp_sum(sum) / (float)H;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    const float d = v[i] - mean;
    if (idx < H) sq = fmaf(d, d, sq);
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)H + eps);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int idx = lane + 32 * i;
    if (idx < H) {
      float y = fmaf((v[i] - mean) * rstd, __ldg(gamma + idx), __ldg(beta + idx));
      y = apply_act(y, act);
      if (out) out[row * H + idx] = __float2bfloat16_rn(y);
      if (out_f32) out_f32[row * H + idx] = y;
    }
  }
}

// vectorised variant: H = 128 * NV, each lane owns NV float4 (columns 4*(lane + 32*i) ..)
template <bool IN_F32, int NV>
__global__ void __launch_bounds__(256) layernorm_vec_kernel(const void* __restrict__ in,
                                                             const __nv_bfloat16* __restrict__ residual, long long rows,
                                                             const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, float eps, int act,
                                                             __nv_bfloat16* __restrict__ out,
                                                             float* __restrict__ out_f32) {
  constexpr int H = 128 * NV;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  float4 v[NV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c4 = lane + 32 * i;
    if constexpr (IN_F32) {
      v[i] = __ldcs(reinterpret_cast<const float4*>(in) + row * (H / 4) + c4);
    } else {
      const uint2 u = __ldcs(reinterpret_cast<const uint2*>(in) + row * (H / 4) + c4);
      v[i] = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
    }
    if (residual) {   // post-LN blocks: LayerNorm(sublayer output + its bf16 input), HF wav2vec2 :597-602
      const uint2 u = __ldg(reinterpret_cast<const uint2*>(residual) + row * (H / 4) + c4);
      v[i].x += bf16_lo(u.x);
      v[i].y += bf16_hi(u.x);
      v[i].z += bf16_lo(u.y);
      v[i].w += bf16_hi(u.y);
    }
    sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(sum) * (1.0f / H);
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    sq += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(sq) * (1.0f / H) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c4 = lane + 32 * i;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c4);
    const float4 bt = __ldg(reinterpret_cast<const float4*>(beta) + c4);
    float4 y;
    y.x = fmaf((v[i].x - mean) * rstd, g.x, bt.x);
    y.y = fmaf((v[i].y - mean) * rstd, g.y, bt.y);
    y.z = fmaf((v[i].z - mean) * rstd, g.z, bt.z);
    y.w = fmaf((v[i].w - mean) * rstd, g.w, bt.w);
    if (act == ACT_GELU) {
      y.x = gelu_erf(y.x); y.y = gelu_erf(y.y); y.z = gelu_erf(y.z); y.w = gelu_erf(y.w);
    } else if (act == ACT_SWISH) {
      y.x = swish(y.x); y.y = swish(y.y); y.z = swish(y.z); y.w = swish(y.w);
    }
    if (out) {
      uint2 u;
      u.x = pack_bf16x2(y.x, y.y);
      u.y = pack_bf16x2(y.z, y.w);
      reinterpret_cast<uint2*>(out)[row * (H / 4) + c4] = u;
    }
    if (out_f32) reinterpret_cast<float4*>(out_f32)[row * (H / 4) + c4] = y;
  }
}

template <bool IN_F32>
static bool launch_ln_vec(const void* in, const __nv_bfloat16* residual, long long rows, int H, const float* gamma,
                          const float* beta, float eps, int act, __nv_bfloat16* out, float* out_f32, cudaStream_t s) {
  const unsigned grid = (unsigned)((rows + 7) / 8);
  switch (H) {
    case 128: launch_pdl(layernorm_vec_kernel<IN_F32, 1>, dim3(grid), dim3(256), 0, s, 1, in, residual, rows, gamma, beta, eps, act, out, out_f32); return true;
    case 256: launch_pdl(layernorm_vec_kernel<IN_F32, 2>, dim3(grid), dim3(256), 0, s, 1, in, residual, rows, gamma, beta, eps, act, out, out_f32); return true;
    case 512: launch_pdl(layernorm_vec_kernel<IN_F32, 4>, dim3(grid), dim3(256), 0, s, 1, in, residual, rows, gamma, beta, eps, act, out, out_f32); return true;
    case 768: launch_pdl(layernorm_vec_kernel<IN_F32, 6>, dim3(grid), dim3(256), 0, s, 1, in, residual, rows, gamma, beta, eps, act, out, out_f32); return true;
    case 1024: launch_pdl(layernorm_vec_kernel<IN_F32, 8>, dim3(grid), dim3(256), 0, s, 1, in, residual, rows, gamma, beta, eps, act, out, out_f32); return true;
    default: return false;
  }
}

std::string launch_layernorm(const void* in, int in_fp32, long long rows, int H, const float* gamma,
                             const float* beta, float eps, int act, __nv_bfloat16* out, float* out_f32,
                             cudaStream_t s, const __nv_bfloat16* residual) {
  if (H > 1024) return "layernorm: H > 1024 not supported";
  if (rows == 0) return "";
  const bool vec = in_fp32 ? launch_ln_vec<true>(in, residual, rows, H, gamma, beta, eps, act, out, out_f32, s)
                           : launch_ln_vec<false>(in, residual, rows, H, gamma, beta, eps, act, out, out_f32, s);
  if (!vec) {
    if (residual) return "layernorm: fused residual needs H in {128, 256, 512, 768, 1024}";
    const unsigned grid = (unsigned)((rows + 7) / 8);
    if (in_fp32) layernorm_kernel<true><<<grid, 256, 0, s>>>(in, rows, H, gamma, beta, eps, act, out, out_f32);
    else layernorm_kernel<false><<<grid, 256, 0, s>>>(in, rows, H, gamma, beta, eps, act, out, out_f32);
  }
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// =================================================================================================
// positional-conv staging: zero-padded, 64-channel-per-group layout so that each tap of each group is one
// 128-byte-wide TMA box (HF wav2vec2/modeling_wav2vec2.py:326-379: padding = k/2 on both sides).
// =================================================================================================
__global__ void __launch_bounds__(256) pos_pad_kernel(const __nv_bfloat16* __restrict__ h, int T, int H, int G,
                                                       int kpos, int left, __nv_bfloat16* __restrict__ out) {
  // one thread = 8 consecutive channels (16 bytes) of one padded row
  const int cpg = H / G;
  const int Tp = T + kpos;
  const int W8 = G * 8;
  const int b = blockIdx.y;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)Tp * W8;
       i += (long long)gridDim.x * blockDim.x) {
    const int tp = (int)(i / W8);
    const int c8 = (int)(i - (long long)tp * W8);
    const int g = c8 >> 3, c = (c8 & 7) * 8;
    const int t = tp - left;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (t >= 0 && t < T && c < cpg) {
      const __nv_bfloat16* src = h + ((long long)b * T + t) * H + g * cpg + c;
      if (c + 8 <= cpg && (cpg % 8) == 0) {
        v = *reinterpret_cast<const uint4*>(src);
      } else {
        __nv_bfloat16 tmp[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) tmp[k] = (c + k < cpg) ? src[k] : __float2bfloat16_rn(0.f);
        v = *reinterpret_cast<uint4*>(tmp);
      }
    }
    reinterpret_cast<uint4*>(out + (long long)b * Tp * G * 64)[i] = v;
  }
}
std::string launch_pos_pad(const __nv_bfloat16* h, int B, int T, int H, int G, int kpos, __nv_bfloat16* out,
                           cudaStream_t s, int left) {
  if (left < 0) left = kpos / 2;
  if (H % G || H / G > 64) return "pos_pad: channels per group must be <= 64";
  if (B == 0) return "";
  const long long per = (long long)(T + kpos) * G * 8;
  dim3 grid((unsigned)((per + 255) / 256 > 1024 ? 1024 : (per + 255) / 256), B);
  W2S_CUDA_OK(launch_pdl(pos_pad_kernel, grid, dim3(256), 0, s, 1, h, T, H, G, kpos, left, out));
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

// =================================================================================================
// one-off weight re-layout
// =================================================================================================
__global__ void axpy_kernel(const float* x, float* y, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] += x[i];
}
std::string launch_axpy(const float* x, float* y, int n, cudaStream_t s) {
  axpy_kernel<<<(n + 255) / 256, 256, 0, s>>>(x, y, n);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

__global__ void cast_bf16_kernel(const float* src, __nv_bfloat16* dst, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dst[i] = __float2bfloat16_rn(src[i]);
}
std::string launch_cast_bf16(const float* src, __nv_bfloat16* dst, long long n, cudaStream_t s) {
  if (n == 0) return "";
  cast_bf16_kernel<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, dst, n);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

__global__ void repack_conv_kernel(const float* src, __nv_bfloat16* dst, int O, int C, int kw) {
  const long long n = (long long)O * C * kw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int j = (int)((i / C) % kw);
    const int o = (int)(i / ((long long)C * kw));
    dst[i] = __float2bfloat16_rn(src[((long long)o * C + c) * kw + j]);
  }
}
std::string launch_repack_conv(const float* src, __nv_bfloat16* dst, int O, int C, int kw, cudaStream_t s) {
  const long long n = (long long)O * C * kw;
  repack_conv_kernel<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, dst, O, C, kw);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

__global__ void repack_posconv_kernel(const float* src, __nv_bfloat16* dst, int H, int G, int kw) {
  const int cpg = H / G;
  const long long n = (long long)H * kw * 64;  // [G][cpg][kw*64]
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i & 63);
    const int j = (int)((i >> 6) % kw);
    const int o = (int)(i / ((long long)kw * 64));  // output channel g*cpg + n
    float v = 0.f;
    if (c < cpg) v = src[((long long)o * cpg + c) * kw + j];
    dst[i] = __float2bfloat16_rn(v);
  }
}
std::string launch_repack_posconv(const float* src, __nv_bfloat16* dst, int H, int G, int kw, cudaStream_t s) {
  const long long n = (long long)H * kw * 64;
  repack_posconv_kernel<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, dst, H, G, kw);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

__global__ void repack_glu_kernel(const float* src, __nv_bfloat16* dst, int half, int K) {
  const long long n = (long long)2 * half * K;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % K);
    const int r = (int)(i / K);
    const int srow = (r & 1) ? (r >> 1) + half : (r >> 1);
    dst[i] = __float2bfloat16_rn(src[(long long)srow * K + k]);
  }
}
std::string launch_repack_glu(const float* src, __nv_bfloat16* dst, int half, int K, cudaStream_t s) {
  const long long n = (long long)2 * half * K;
  repack_glu_kernel<<<(unsigned)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, dst, half, K);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

}  // namespace w2s
