// Self-attention of the encoder (HF wav2vec2/modeling_wav2vec2.py:438-463, :500-549; conformer relative
// positions wav2vec2_conformer/modeling_wav2vec2_conformer.py:509-565).
//
//  * attention_fa.cu       : the tcgen05 kernel of the plain / rotary models (persistent, warp-specialised, key blocks
//                            streamed through independent accumulators; any clip length).
//  * attention_rel_kernel  : conformer relative-position attention on tcgen05 (any clip length).
//  * attention_simt_kernel : CUDA-core cross-check (one warp per query row, with the WavLM bias when given), reachable
//                            through W2S_FLAG_VALIDATE_ATTN only -- never a fallback of the product path.
#include "kernels.cuh"
#include "gemm.cuh"

namespace w2s {

// =================================================================================================
// validation kernel
// =================================================================================================
constexpr int SIMT_MAXC = 32;  // key chunks of 32 -> T <= 1024

__global__ void __launch_bounds__(128) attention_simt_kernel(const AttnParams p) {
  __shared__ float qs[4][2][128];  // per warp: q + u, q + v  (hd <= 128)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long gw = (long long)blockIdx.x * 4 + warp;
  const long long total = (long long)p.B * p.heads * p.T;
  if (gw >= total) return;
  const int i = (int)(gw % p.T);
  const int h = (int)((gw / p.T) % p.heads);
  const int b = (int)(gw / ((long long)p.T * p.heads));
  const int H3 = p.ld;
  const __nv_bfloat16* qrow = p.qkv + ((long long)b * p.T + i) * H3 + h * p.hd;
  for (int d = lane; d < p.hd; d += 32) {
    qs[warp][0][d] = __bfloat162float(qrow[p.q_off + d]);
    qs[warp][1][d] = p.pos_proj ? __bfloat162float(qrow[p.qv_off + d]) : 0.f;
  }
  __syncwarp();
  // WavLM: gate * table entry (log2 units) * ln 2 = the natural-units bias
  const float gb = p.rel_bias ? p.gate[((long long)b * p.heads + h) * p.T + i] * 0.6931471805599453f : 0.f;
  const float* brow = p.rel_bias ? p.rel_bias + (long long)h * rel_bias_ld(p.T) + REL_BIAS_PAD + p.T - 1 - i : nullptr;
  float s[SIMT_MAXC];
  float mx = -INFINITY;
#pragma unroll
  for (int c = 0; c < SIMT_MAXC; ++c) {
    const int j = c * 32 + lane;
    float acc = -INFINITY;
    if (j < p.T) {
      const __nv_bfloat16* krow = p.qkv + ((long long)b * p.T + j) * H3 + p.k_off + h * p.hd;
      acc = 0.f;
      for (int d = 0; d < p.hd; d += 2) {
        const uint32_t kk = *reinterpret_cast<const uint32_t*>(krow + d);
        acc = fmaf(qs[warp][0][d], bf16_lo(kk), acc);
        acc = fmaf(qs[warp][0][d + 1], bf16_hi(kk), acc);
      }
      if (p.pos_proj) {
        // shift trick as index arithmetic: bd[i, j] = (q_i + v) . pos_proj[T - 1 - i + j]
        const __nv_bfloat16* prow = p.pos_proj + (long long)(p.T - 1 - i + j) * p.H + h * p.hd;
        for (int d = 0; d < p.hd; d += 2) {
          const uint32_t pp = *reinterpret_cast<const uint32_t*>(prow + d);
          acc = fmaf(qs[warp][1][d], bf16_lo(pp), acc);
          acc = fmaf(qs[warp][1][d + 1], bf16_hi(pp), acc);
        }
      }
      acc *= p.scale;
      if (brow) acc = fmaf(gb, brow[j], acc);
    }
    s[c] = acc;
    mx = fmaxf(mx, acc);
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int c = 0; c < SIMT_MAXC; ++c) {
    const float e = (c * 32 + lane < p.T) ? __expf(s[c] - mx) : 0.f;
    s[c] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  const float inv = 1.0f / sum;
  float o[4] = {0.f, 0.f, 0.f, 0.f};  // hd <= 128
#pragma unroll
  for (int c = 0; c < SIMT_MAXC; ++c) {
    if (c * 32 >= p.T) break;
    for (int l = 0; l < 32; ++l) {
      const int j = c * 32 + l;
      const float pj = __shfl_sync(0xffffffffu, s[c], l);
      if (j < p.T) {
        const __nv_bfloat16* vrow = p.qkv + ((long long)b * p.T + j) * H3 + p.v_off + h * p.hd;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int d = lane + 32 * r;
          if (d < p.hd) o[r] = fmaf(pj, __bfloat162float(vrow[d]), o[r]);
        }
      }
    }
  }
  __nv_bfloat16* orow = p.ctx + ((long long)b * p.T + i) * p.H + h * p.hd;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int d = lane + 32 * r;
    if (d < p.hd) orow[d] = __float2bfloat16_rn(o[r] * inv);
  }
}

std::string launch_attention_simt(const AttnParams& p, cudaStream_t s) {
  if (p.T > 32 * SIMT_MAXC) return "attention (validation kernel): T' > 1024 not supported";
  if (p.hd > 128 || (p.hd & 1)) return "attention (validation kernel): head_dim must be even and <= 128";
  const long long total = (long long)p.B * p.heads * p.T;
  if (total == 0) return "";
  attention_simt_kernel<<<(unsigned)((total + 3) / 4), 128, 0, s>>>(p);
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

__device__ __forceinline__ uint64_t umma_desc_sw128_mn(uint32_t smem_addr) {
  // MN-major operand (rows = K index, 128 contiguous bytes = 64 MN elements, 128B swizzle):
  // 8-row (K) groups are 1024 B apart (SBO); LBO (next 64-wide MN block) unused for N = 64.
  return umma_desc_sw128(smem_addr);
}
__host__ __device__ constexpr uint32_t umma_idesc_bf16_bmn(int M, int N) {
  return umma_idesc_bf16(M, N) | (1u << 16);  // b_major = MN
}

// =================================================================================================
// conformer relative-position attention on tcgen05 (HF wav2vec2_conformer/modeling_wav2vec2_conformer.py:509-565)
//   scores[i, j] = ((q_i + u) . k_j + (q_i + v) . pp[T-1-i+j]) / sqrt(d)
// One CTA per (128-query tile, head, coalition), keys in halves of 128.  Per half two MMA chains fill TMEM:
//   AC  [128 x 128] = (Q+u) K^T                               columns   0..127
//   BD  [128 x 256] = (Q+v) PP_window^T, window row w <-> r = r_lo + w  columns 128..383
// and the "shift trick" of the reference is an index shift per query row: bd[i, j] = BD[i, 127 - i_local + (j - j0)].
// Each warp reads its 64 raw BD columns per 32-key chunk, stages them in its private shared-memory strip and reads
// them back with the lane-dependent offset.  Each key block keeps its own softmax maximum and its own O accumulator
// (columns 384..447 / 448..511, alternating); a finished block is folded into a per-thread running (max, sum, 32 output
// columns) while the next block's scores are computed, so nothing in TMEM is ever rescaled and the number of key
// blocks -- the clip length -- is unbounded.
// =================================================================================================
struct AttnRelDev {
  __nv_bfloat16* ctx;
  int B, T, H, heads, nh;
  float scale_log2e;
};
struct AttnRelPlan {
  CUtensorMap mapQU, mapQV, mapK, mapV, mapP;
  AttnRelDev dev;
  dim3 grid;
};
constexpr int REL_QU = 0, REL_QV = 16384, REL_K = 32768, REL_V = 49152, REL_PP = 65536, REL_P = 98304,
              REL_STG = 131072, REL_STG_STRIDE = 67;
constexpr size_t REL_SMEM = REL_STG + 8 * 32 * REL_STG_STRIDE * 4 + 1024;

__global__ void __launch_bounds__(256, 1)
attention_rel_kernel(const __grid_constant__ CUtensorMap mapQU, const __grid_constant__ CUtensorMap mapQV,
                     const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapV,
                     const __grid_constant__ CUtensorMap mapP, const AttnRelDev p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ float s_red[2][128];
  __shared__ float s_sum[1][2][128];
  __shared__ uint64_t s_bar[4];
  __shared__ uint32_t s_tmem;
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - raw_addr);
  const uint32_t bar_q = smem_u32(&s_bar[0]), bar_load = smem_u32(&s_bar[1]), bar_mma = smem_u32(&s_bar[2]),
                 bar_pv = smem_u32(&s_bar[3]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qd = warp & 3, hf = warp >> 2;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int row = qd * 32 + lane;
  float* stg = reinterpret_cast<float*>(base_ptr + REL_STG) + warp * 32 * REL_STG_STRIDE + lane * REL_STG_STRIDE;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&mapQU);
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
    tma_prefetch_desc(&mapP);
    for (int i = 0; i < 4; ++i) mbar_init(smem_u32(&s_bar[i]), 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 0) {
    tmem_alloc<512>(smem_u32(&s_tmem));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(&s_tmem);
  const uint32_t trow = tmem + (static_cast<uint32_t>(qd * 32) << 16);

  if (warp == 0 && elect_one()) {
    mbar_expect_tx(bar_q, 32768);
    tma_load_4d(base + REL_QU, &mapQU, bar_q, 0, qt * 128, h, b);
    tma_load_4d(base + REL_QV, &mapQV, bar_q, 0, qt * 128, h, b);
  }

  // running state of this thread's query row: its 32 output columns relative to m_run (maximum over the FOLDED blocks),
  // and its share of the row sum (its 64 keys per block) relative to m_l (maximum over the blocks whose softmax is done:
  // one block ahead of m_run, because a block's output is folded only after its P V has completed)
  float m_run = -3.0e38f, m_l = -3.0e38f, l_run = 0.f;
  float o_run[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) o_run[j] = 0.f;
  float m_prev = 0.f;   // maximum of the block whose P V is in flight (folded one block later)

  // fold block hk (maximum m_blk, accumulator slot hk & 1) into the running state; its P V has completed
  auto fold = [&](int hk, float m_blk) {
    const float m_new = fmaxf(m_run, m_blk);
    const float alpha = ex2_approx((m_run - m_new) * p.scale_log2e);
    const float a = ex2_approx((m_blk - m_new) * p.scale_log2e);
    float v[32];
    tmem_ld_32x32(trow + 384 + 64 * (hk & 1) + hf * 32, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) o_run[j] = fmaf(alpha, o_run[j], a * v[j]);
    m_run = m_new;
  };

  for (int hk = 0; hk < p.nh; ++hk) {
    const int j0 = hk * 128;
    if (warp == 0 && elect_one()) {
      if (hk > 0) mbar_wait(bar_pv, (hk - 1) & 1);  // previous P V has finished reading V and P
      mbar_expect_tx(bar_load, 16384 + 16384 + 32768);
      tma_load_4d(base + REL_K, &mapK, bar_load, 0, j0, h, b);
      tma_load_4d(base + REL_V, &mapV, bar_load, 0, j0, h, b);
      tma_load_4d(base + REL_V + 8192, &mapV, bar_load, 0, j0 + 64, h, b);
      tma_load_3d(base + REL_PP, &mapP, bar_load, 0, p.T - 1 - (qt * 128 + 127) + j0, h);
      if (hk == 0) mbar_wait(bar_q, 0);
      mbar_wait(bar_load, hk & 1);
      tc_fence_after();
      const uint64_t dqu = umma_desc_sw128(base + REL_QU), dqv = umma_desc_sw128(base + REL_QV);
      const uint64_t dk = umma_desc_sw128(base + REL_K), dp = umma_desc_sw128(base + REL_PP);
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_bf16(tmem, dqu + 2u * k, dk + 2u * k, umma_idesc_bf16(128, 128), k != 0);
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_bf16(tmem + 128, dqv + 2u * k, dp + 2u * k, umma_idesc_bf16(128, 256), k != 0);
      umma_commit(bar_mma);
    }
    // while the score MMAs of this block run: fold the previous block (its P V is complete once bar_pv has flipped)
    if (hk > 0) {
      mbar_wait(bar_pv, (hk - 1) & 1);
      tc_fence_after();
      fold(hk - 1, m_prev);
    }
    mbar_wait(bar_mma, hk & 1);
    tc_fence_after();

    // ---- scores of this thread's 64 keys (two chunks of 32) --------------------------------------------------------
    float sc[64];
    float mx = -INFINITY;
    const int base_q = 96 - 32 * qd;
#pragma unroll
    for (int ch = 0; ch < 2; ++ch) {
      const int c_local = hf * 64 + ch * 32;
      float ac[32], r0[32], r1[32];
      tmem_ld_32x32(trow + c_local, ac);
      tmem_ld_32x32(trow + 128 + base_q + c_local, r0);
      tmem_ld_32x32(trow + 128 + base_q + c_local + 32, r1);
#pragma unroll
      for (int k2 = 0; k2 < 32; ++k2) {
        stg[k2] = r0[k2];
        stg[32 + k2] = r1[k2];
      }
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 32; ++t) {
        const float v = ac[t] + stg[31 - lane + t];
        const bool ok = (j0 + c_local + t) < p.T;
        sc[ch * 32 + t] = ok ? v : -3.0e38f;   // finite sentinel: exp2 underflows to 0 without a select
        mx = fmaxf(mx, sc[ch * 32 + t]);
      }
      __syncwarp();
    }
    s_red[hf][row] = mx;
    __syncthreads();
    mx = fmaxf(s_red[0][row], s_red[1][row]);
    const float2 sc2 = make_float2(p.scale_log2e, p.scale_log2e);
    const float2 nm2 = make_float2(-mx * p.scale_log2e, -mx * p.scale_log2e);
    float2 acc2 = make_float2(0.f, 0.f);
    const uint32_t sp_row = base + REL_P + hf * 16384 + row * 128;
#pragma unroll
    for (int c8 = 0; c8 < 8; ++c8) {
      float2 e[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float2 a = __ffma2_rn(make_float2(sc[c8 * 8 + 2 * t], sc[c8 * 8 + 2 * t + 1]), sc2, nm2);
        e[t] = make_float2(ex2_approx(a.x), ex2_approx(a.y));
        acc2 = __fadd2_rn(acc2, e[t]);
      }
      sts128(sp_row + (((uint32_t)c8 ^ ((uint32_t)row & 7u)) << 4), pack_bf16x2(e[0].x, e[0].y),
             pack_bf16x2(e[1].x, e[1].y), pack_bf16x2(e[2].x, e[2].y), pack_bf16x2(e[3].x, e[3].y));
    }
    {
      const float m_new = fmaxf(m_l, mx);
      l_run = fmaf(l_run, ex2_approx((m_l - m_new) * p.scale_log2e),
                   (acc2.x + acc2.y) * ex2_approx((mx - m_new) * p.scale_log2e));
      m_l = m_new;
    }
    m_prev = mx;
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();   // also orders the s_red reads above before the next block overwrites it
    if (warp == 0 && elect_one()) {
      tc_fence_after();
      constexpr uint32_t idesc = umma_idesc_bf16_bmn(128, 64);
      for (int kb = 0; kb < 2; ++kb) {
        const uint64_t dpp = umma_desc_sw128(base + REL_P + kb * 16384);
        const uint64_t dv = umma_desc_sw128_mn(base + REL_V + kb * 8192);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem + 384 + 64 * (hk & 1), dpp + 2u * k, dv + 128u * k, idesc, (kb | k) != 0);
      }
      umma_commit(bar_pv);
    }
  }
  // ---- last block, then out = o_run / (row sum over both key halves of every block) ---------------------------------
  mbar_wait(bar_pv, (p.nh - 1) & 1);
  tc_fence_after();
  fold(p.nh - 1, m_prev);
  s_sum[0][hf][row] = l_run;
  __syncthreads();
  const float inv = 1.0f / (s_sum[0][0][row] + s_sum[0][1][row]);
  const int i = qt * 128 + row;
  __nv_bfloat16* orow = p.ctx + ((long long)b * p.T + i) * p.H + h * 64 + hf * 32;
  if (i < p.T) {
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      uint4 u;
      u.x = pack_bf16x2(o_run[j] * inv, o_run[j + 1] * inv);
      u.y = pack_bf16x2(o_run[j + 2] * inv, o_run[j + 3] * inv);
      u.z = pack_bf16x2(o_run[j + 4] * inv, o_run[j + 5] * inv);
      u.w = pack_bf16x2(o_run[j + 6] * inv, o_run[j + 7] * inv);
      *reinterpret_cast<uint4*>(orow + j) = u;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
}

bool attention_rel_supported(const AttnParams& p) {
  return p.pos_proj != nullptr && p.hd == 64 && (p.H % 8 == 0);
}
std::string attention_rel_init() {
  cudaError_t e = cudaFuncSetAttribute(attention_rel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)REL_SMEM);
  if (e != cudaSuccess) return std::string("cudaFuncSetAttribute(attention_rel_kernel): ") + cudaGetErrorString(e);
  return "";
}
std::string attention_rel_prepare(const AttnParams& p, AttnRelPlan** out) {
  if (!attention_rel_supported(p)) return "attention (tcgen05, relative): unsupported shape";
  AttnRelPlan* pl = new AttnRelPlan();
  pl->dev.ctx = p.ctx;
  pl->dev.B = p.B; pl->dev.T = p.T; pl->dev.H = p.H; pl->dev.heads = p.heads;
  pl->dev.nh = (p.T + 127) / 128;
  pl->dev.scale_log2e = p.scale * 1.4426950408889634f;
  pl->grid = dim3((p.T + 127) / 128, p.heads, p.B);
  const uint64_t ld = (uint64_t)p.ld;
  uint64_t dims[4] = {64, (uint64_t)p.T, (uint64_t)p.heads, (uint64_t)p.B};
  uint64_t str[3] = {ld * 2, 128, (uint64_t)p.T * ld * 2};
  uint32_t box128[4] = {64, 128, 1, 1};
  uint32_t box64[4] = {64, 64, 1, 1};
  std::string err = make_tensor_map_bf16(&pl->mapQU, p.qkv + p.q_off, 4, dims, str, box128);
  if (err.empty()) err = make_tensor_map_bf16(&pl->mapQV, p.qkv + p.qv_off, 4, dims, str, box128);
  if (err.empty()) err = make_tensor_map_bf16(&pl->mapK, p.qkv + p.k_off, 4, dims, str, box128);
  if (err.empty()) err = make_tensor_map_bf16(&pl->mapV, p.qkv + p.v_off, 4, dims, str, box64);
  if (err.empty()) {
    uint64_t pd[3] = {64, (uint64_t)(2 * p.T - 1), (uint64_t)p.heads};
    uint64_t ps[2] = {(uint64_t)p.H * 2, 128};
    uint32_t pb[3] = {64, 256, 1};
    err = make_tensor_map_bf16(&pl->mapP, p.pos_proj, 3, pd, ps, pb);
  }
  if (!err.empty()) {
    delete pl;
    return err;
  }
  *out = pl;
  return "";
}
std::string attention_rel_launch(const AttnRelPlan* pl, cudaStream_t s) {
  W2S_CUDA_OK(launch_pdl(attention_rel_kernel, pl->grid, dim3(256), REL_SMEM, s, 1, pl->mapQU, pl->mapQV, pl->mapK, pl->mapV, pl->mapP, pl->dev));
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}
void attention_rel_free(AttnRelPlan* plan) { delete plan; }

}  // namespace w2s
