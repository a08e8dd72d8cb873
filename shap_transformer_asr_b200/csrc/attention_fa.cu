// Self-attention (no mask, head_dim 64, any number of frames) as a persistent, warp-specialised tcgen05 kernel.
//
// Work item = (128-query tile, head, coalition); keys are walked in blocks of 128, two blocks form a CHUNK.  Blocks are
// INDEPENDENT: every block keeps its own softmax maximum m_j, partial sum l_j and its own O_j accumulator in TMEM,
// and a merge step combines them,  out = sum_j a_j O_j / sum_j a_j l_j,  a_j = exp(m_j - max_j m_j),  so nothing is
// ever rescaled in TMEM and the three engines run decoupled:
//   warp 8  (TMA)     Q tile per item (double-buffered), K_j through a 3-stage and V_j through a 4-stage ring
//   warp 9  (MMA)     S_j = Q K_j^T into one of two S buffers (128 fp32 columns each), O_j = P_j V_j one block behind,
//                     into the O slot of the block's chunk (2 chunk slots x 2 blocks x 64 columns: double-buffered)
//   warps 0-7 (softmax) two groups of four warps, group g takes the blocks with running index g (mod 2): one thread per
//                     query row reads S_j from TMEM, writes P_j = exp(S_j - m_j) as bf16 into the group's swizzled smem
//                     buffer; both groups merge every chunk (32 of the 64 output columns each), one chunk late, so the
//                     P V MMAs finish behind useful work
// Clips of up to 256 frames are one chunk per item (NBT = 1, 2: everything static).  Longer clips (NBT = 0) stream
// chunk after chunk through the two O slots: the merge folds each chunk into a per-thread running (max, sum, 32
// output columns) in registers -- the flash-attention recurrence at chunk granularity -- so T' is unbounded and the
// O accumulators stay double-buffered (the first version held all blocks of an item in TMEM: T' <= 512, single-buffered
// beyond 256).
// HF wav2vec2/modeling_wav2vec2.py:438-463 (softmax(Q K^T / sqrt d) V, no mask, eval mode).
// BIAS (WavLM, HF wavlm/modeling_wavlm.py:147-186): every score gains the gated relative-position bias
// g[b, h, i] * E[bucket(j - i), h].  The softmax thread of query row i adds it to each score read from TMEM, in both
// passes, before the padding mask; the Toeplitz table is read through L1 (lanes are consecutive query rows, so a warp's
// read of one key column covers 32 consecutive floats), shared memory being full.
#include "kernels.cuh"
#include "gemm.cuh"

#include <type_traits>

namespace w2s {

struct AttnFaDev {
  __nv_bfloat16* ctx;
  float* lse;   // optional [B, heads, T]: log2-domain log-sum-exp of the scaled scores (the gradient path's backward kernel)
  int B, T, H, heads, qtiles, num_items, nb;
  float scale_log2e;
};
// the bias variant's parameters extend the plain ones (which stay as they are: a larger parameter block alone changes
// how the plain variants are scheduled)
struct AttnFaBiasDev : AttnFaDev {
  const float* rel_bias;   // [heads, rel_bias_ld(T)], see AttnParams
  const float* gate;       // [B, heads, T]
};
struct AttnFaPlan {
  CUtensorMap mapQ, mapK, mapV;
  AttnFaBiasDev dev;   // rel_bias == null: the plain variant
  int nb, grid;
};

// K and V travel through separate rings.  A K block is dead as soon as its score MMAs have run, a V block lives until
// the softmax of its block is done; with one {K, V} ring a stage was recycled only after P V, and the ~3000-cycle
// TMA round trip of the next load then sat on the critical path (measured with clock64 stamps: the MMA thread waited
// for K/V about a third of every item).
constexpr int FA_KS = 3, FA_VS = 4;
constexpr int FA_SQ = 0, FA_SK = 2 * 16384, FA_SV = FA_SK + FA_KS * 16384, FA_SP = FA_SV + FA_VS * 16384,
              FA_RED = FA_SP + 2 * 32768, FA_BAR = FA_RED + 2 * (4 * 4 * 128 * 4);
constexpr size_t FA_SMEM = FA_BAR + 512 + 1024;

__device__ __forceinline__ uint64_t fa_desc_mn(uint32_t a) { return umma_desc_sw128(a); }

template <int NBT, bool BIAS>
__global__ void __launch_bounds__(384, 1)
attention_fa_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                    const __grid_constant__ CUtensorMap mapV, const std::conditional_t<BIAS, AttnFaBiasDev, AttnFaDev> p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - raw);
  float* s_m = reinterpret_cast<float*>(base_ptr + FA_RED);               // [item mod 4][4][128] block maxima
  float* s_l = s_m + 4 * 4 * 128;                                          // [item mod 4][4][128] block sums
  const uint32_t bars = base + FA_BAR;
  auto k_full = [&](int s) { return bars + 8u * s; };
  auto k_empty = [&](int s) { return bars + 24 + 8u * s; };
  auto v_full = [&](int s) { return bars + 48 + 8u * s; };
  auto v_empty = [&](int s) { return bars + 80 + 8u * s; };
  auto s_full = [&](int i) { return bars + 112 + 8u * i; };
  auto s_empty = [&](int i) { return bars + 128 + 8u * i; };
  auto p_full = [&](int i) { return bars + 144 + 8u * i; };
  auto p_empty = [&](int i) { return bars + 160 + 8u * i; };
  auto q_full = [&](int i) { return bars + 176 + 8u * i; };
  auto q_empty = [&](int i) { return bars + 192 + 8u * i; };
  auto o_full = [&](int i) { return bars + 208 + 8u * i; };
  auto o_empty = [&](int i) { return bars + 224 + 8u * i; };
  auto ml_full = [&](int i) { return bars + 240 + 8u * i; };
  const uint32_t tmem_slot = bars + 272;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + FA_BAR + 272);
  constexpr bool STREAM = NBT == 0;
  const int NB = STREAM ? p.nb : NBT;      // key blocks per item
  const int CPI = (NB + 1) >> 1;           // chunks per item

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&mapQ);
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
  }
  if (warp == 9 && lane == 0) {
    for (int s = 0; s < FA_KS; ++s) {
      mbar_init(k_full(s), 1);
      mbar_init(k_empty(s), 1);
    }
    for (int s = 0; s < FA_VS; ++s) {
      mbar_init(v_full(s), 1);
      mbar_init(v_empty(s), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(q_full(i), 1);
      mbar_init(q_empty(i), 1);
      mbar_init(o_full(i), 1);
      mbar_init(o_empty(i), 8);
      mbar_init(s_full(i), 1);
      mbar_init(s_empty(i), 4);
      mbar_init(p_full(i), 4);
      mbar_init(p_empty(i), 1);
    }
    for (int i = 0; i < 4; ++i) mbar_init(ml_full(i), 8);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 9) {
    __syncwarp();   // reconverge after the lane-0 barrier initialisation: the allocation is warp-collective
    tmem_alloc<512>(tmem_slot);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  // TMEM columns: S buffers at 0 / 128; O of block jj (0 / 1) of a chunk with running index gcx at 256 + 128 (gcx & 1) + 64 jj

  if (warp == 8) {
    if (elect_one()) {
      uint32_t kvc = 0;
      int it = 0;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x, ++it) {
        const int qt = item % p.qtiles, h = (item / p.qtiles) % p.heads, b = item / (p.qtiles * p.heads);
        // Q is double-buffered: the tile of item i+1 (and its first K/V stage) is in flight while item i computes
        mbar_wait(q_empty(it & 1), ((uint32_t)(it >> 1) & 1u) ^ 1u);
        mbar_expect_tx(q_full(it & 1), 16384);
        tma_load_4d(base + FA_SQ + (it & 1) * 16384, &mapQ, q_full(it & 1), 0, qt * 128, h, b);
#pragma unroll 1
        for (int j = 0; j < NB; ++j, ++kvc) {
          const int ks = kvc % FA_KS, vs = kvc % FA_VS;
          mbar_wait(k_empty(ks), ((kvc / FA_KS) & 1u) ^ 1u);
          mbar_expect_tx(k_full(ks), 16384);
          tma_load_4d(base + FA_SK + ks * 16384, &mapK, k_full(ks), 0, j * 128, h, b);
          mbar_wait(v_empty(vs), ((kvc / FA_VS) & 1u) ^ 1u);
          mbar_expect_tx(v_full(vs), 16384);
          tma_load_4d(base + FA_SV + vs * 16384, &mapV, v_full(vs), 0, j * 128, h, b);
        }
      }
    }
  } else if (warp == 9) {
    if (elect_one()) {
      constexpr uint32_t idesc_qk = umma_idesc_bf16(128, 128);
      constexpr uint32_t idesc_pv = umma_idesc_bf16(128, 64) | (1u << 16);   // B operand (V) is MN-major
      uint32_t kvc = 0, sc = 0, pc = 0;
      int it = 0;
      auto issue_pv = [&](int jj, uint32_t blk, uint32_t gcx) {
        const int vs = blk % FA_VS;
        const int pb = pc & 1;
        // a chunk's O slot is overwritten from the chunk's first P V on: only then must the merge of the chunk that
        // used the slot before (two chunks back) have drained it (waiting here instead of before the score MMAs lets
        // the next scores be computed while the softmax warps still finish the previous chunk)
        const uint32_t cp = gcx & 1u;
        if (jj == 0) mbar_wait(o_empty(cp), ((gcx >> 1) & 1u) ^ 1u);
        mbar_wait(v_full(vs), (blk / FA_VS) & 1u);
        mbar_wait(p_full(pb), (pc >> 1) & 1u);
        tc_fence_after();
#pragma unroll
        for (int kb = 0; kb < 2; ++kb) {
          const uint64_t dp = umma_desc_sw128(base + FA_SP + pb * 32768 + kb * 16384);
          const uint64_t dv = fa_desc_mn(base + FA_SV + vs * 16384 + kb * 8192);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem + 256 + 128 * cp + 64 * jj, dp + 2u * k, dv + 128u * k, idesc_pv, (kb | k) != 0 ? 1u : 0u);
        }
        umma_commit(p_empty(pb));
        umma_commit(v_empty(vs));
        ++pc;
      };
      // Blocks form ONE stream across items: S_g is issued, then P V of block g-1 -- also across an item boundary, so the
      // first score block of the next item is already in TMEM when the softmax warps finish the previous item.
      bool pending = false;
      int pend_j = 0;
      uint32_t pend_blk = 0, pend_gcx = 0;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x, ++it) {
        mbar_wait(q_full(it & 1), (uint32_t)(it >> 1) & 1u);
#pragma unroll 1
        for (int j = 0; j < NB; ++j, ++kvc, ++sc) {
          const int ks = kvc % FA_KS, sb = sc & 1;
          mbar_wait(k_full(ks), (kvc / FA_KS) & 1u);
          mbar_wait(s_empty(sb), ((sc >> 1) & 1u) ^ 1u);
          tc_fence_after();
          const uint64_t dq = umma_desc_sw128(base + FA_SQ + (it & 1) * 16384);
          const uint64_t dk = umma_desc_sw128(base + FA_SK + ks * 16384);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(tmem + sb * 128, dq + 2u * k, dk + 2u * k, idesc_qk, k != 0 ? 1u : 0u);
          umma_commit(s_full(sb));
          umma_commit(k_empty(ks));
          if (j == NB - 1) umma_commit(q_empty(it & 1));
          if (pending) {
            issue_pv(pend_j & 1, pend_blk, pend_gcx);
            if ((pend_j & 1) == 1 || pend_j == NB - 1) umma_commit(o_full(pend_gcx & 1u));   // last block of its chunk
          }
          pending = true;
          pend_j = j;
          pend_blk = kvc;
          pend_gcx = (uint32_t)it * (uint32_t)CPI + (uint32_t)(j >> 1);
        }
      }
      if (pending) {
        issue_pv(pend_j & 1, pend_blk, pend_gcx);
        umma_commit(o_full(pend_gcx & 1u));
      }
    }
  } else if (warp < 8) {
    // Two softmax groups of four warps.  Group g owns every key block whose running index is g (mod 2) -- S buffer g,
    // P buffer g -- and one thread owns one query row with all 128 keys of the block, so a block needs no exchange
    // between threads and the two groups drift apart: while one waits for TMEM or the MMA warp, the other keeps the
    // MUFU / FMA pipes of the same scheduler busy.  Scores are read from TMEM twice (maximum, then exponentials)
    // instead of being held in 128 registers.  The merge of item i is deferred until after the group's first block
    // of item i+1, so the P V MMAs of item i finish behind useful work.
    const int grp = warp >> 2, qd = warp & 3;
    const int row = qd * 32 + lane;
    const uint32_t trow = tmem + (static_cast<uint32_t>(qd * 32) << 16);
    const uint32_t s_addr = trow + grp * 128;
    const uint32_t sp_row = base + FA_SP + grp * 32768 + row * 128;
    const uint32_t sw = (uint32_t)row & 7u;
    const float2 sc2 = make_float2(p.scale_log2e, p.scale_log2e);
    // BIAS: this thread's query row i of the current item reads table entry 128 + T - 1 - i + key, scaled by its gate
    // (divided by scale_log2e: the scores stay unscaled until the exponentials)
    const float* brow = nullptr;
    float gsc = 0.f;
    auto add_bias = [&](float (&v)[32], int key0) {
      if constexpr (BIAS) {
#pragma unroll
        for (int t = 0; t < 32; ++t) v[t] = fmaf(gsc, __ldg(brow + key0 + t), v[t]);
      }
    };

    auto mask_tail = [&](float (&v)[32], int col0, int nvalid) {
#pragma unroll
      for (int g8 = 0; g8 < 4; ++g8) {
        if (col0 + 8 * g8 + 8 > nvalid) {   // warp-uniform
#pragma unroll
          for (int t = 0; t < 8; ++t)
            if (col0 + 8 * g8 + t >= nvalid) v[8 * g8 + t] = -3.0e38f;   // finite: exp2 underflows to 0 by itself
        }
      }
    };
    auto max32 = [&](const float (&v)[32]) {
      float m0 = v[0], m1 = v[1], m2 = v[2], m3 = v[3];
#pragma unroll
      for (int t = 4; t < 32; t += 4) {
        m0 = fmaxf(m0, v[t]);
        m1 = fmaxf(m1, v[t + 1]);
        m2 = fmaxf(m2, v[t + 2]);
        m3 = fmaxf(m3, v[t + 3]);
      }
      return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
    };

    // Running state of the item this group is merging (streaming variant; with one chunk per item it is dead code).
    float m_run = 0.f, l_run = 0.f;
    float o_run[32];
#pragma unroll
    for (int t = 0; t < 32; ++t) o_run[t] = 0.f;

    // Fold chunk `gcx` (nbc blocks; `first` / `last` chunk of `item`) into the running state; the last chunk normalises
    // and stores this thread's 32 output columns.
    auto merge = [&](int item, uint32_t gcx, int nbc, bool first, bool last) {
      const float* pm = s_m + (gcx & 3u) * (4 * 128) + row;
      const float* pl = s_l + (gcx & 3u) * (4 * 128) + row;
      const uint32_t cp = gcx & 1u;
      mbar_wait(ml_full(gcx & 3u), (gcx >> 2) & 1u);
      const float m0 = pm[0], m1 = nbc > 1 ? pm[128] : pm[0];
      float m = fmaxf(m0, m1);
      float alpha = 0.f;
      if (STREAM && !first) {
        m = fmaxf(m, m_run);
        alpha = ex2_approx((m_run - m) * p.scale_log2e);
      }
      const float a0 = ex2_approx((m0 - m) * p.scale_log2e);
      const float a1 = nbc > 1 ? ex2_approx((m1 - m) * p.scale_log2e) : 0.f;
      float L = a0 * pl[0];
      if (nbc > 1) L = fmaf(a1, pl[128], L);
      if (STREAM && !first) L = fmaf(alpha, l_run, L);
      mbar_wait(o_full(cp), (gcx >> 1) & 1u);
      tc_fence_after();
      // accumulate straight into the running columns (no second 32-register array next to the TMEM load)
      {
        float v[32];
        tmem_ld_32x32(trow + 256 + 128 * cp + grp * 32, v);
#pragma unroll
        for (int t = 0; t < 32; ++t) o_run[t] = (STREAM && !first) ? fmaf(alpha, o_run[t], a0 * v[t]) : a0 * v[t];
        if (nbc > 1) {
          tmem_ld_32x32(trow + 256 + 128 * cp + 64 + grp * 32, v);
#pragma unroll
          for (int t = 0; t < 32; ++t) o_run[t] = fmaf(a1, v[t], o_run[t]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty(cp));
      if (STREAM && !last) {
        m_run = m;
        l_run = L;
        return;
      }
      const float inv = rcp_approx(L);
      const int qt = item % p.qtiles, h = (item / p.qtiles) % p.heads, b = item / (p.qtiles * p.heads);
      const int i = qt * 128 + row;
      if (!BIAS && p.lse && grp == 0 && i < p.T) p.lse[((long long)b * p.heads + h) * p.T + i] = fmaf(m, p.scale_log2e, __log2f(L));
      if (i < p.T) {
        __nv_bfloat16* orow = p.ctx + ((long long)b * p.T + i) * p.H + h * 64 + grp * 32;
#pragma unroll
        for (int t = 0; t < 32; t += 8) {
          uint4 u;
          u.x = pack_bf16x2(o_run[t] * inv, o_run[t + 1] * inv);
          u.y = pack_bf16x2(o_run[t + 2] * inv, o_run[t + 3] * inv);
          u.z = pack_bf16x2(o_run[t + 4] * inv, o_run[t + 5] * inv);
          u.w = pack_bf16x2(o_run[t + 6] * inv, o_run[t + 7] * inv);
          *reinterpret_cast<uint4*>(orow + t) = u;
        }
      }
    };

    // One key block of this group: S_j (TMEM) -> block maximum, P_j = exp2((S_j - m_j) scale) as bf16 into the group's P
    // buffer, (m_j, l_j) into slot jj of the chunk's ring entry.
    auto block = [&](int j, float* pm_jj, float* pl_jj, uint32_t par) {
      const int nvalid = p.T - j * 128;   // columns >= nvalid of this block are padding (last block only)
      mbar_wait(s_full(grp), par);
      tc_fence_after();
      float s0[32], s1[32];
      // pass 1: block maximum; the second half stays in registers for pass 2
      tmem_ld_32x32_issue(s_addr, s0);
      tmem_ld_32x32_issue(s_addr + 32, s1);
      tmem_ld_wait();
      add_bias(s0, j * 128);
      add_bias(s1, j * 128 + 32);
      if (nvalid < 64) {
        mask_tail(s0, 0, nvalid);
        mask_tail(s1, 32, nvalid);
      }
      float mx = fmaxf(max32(s0), max32(s1));
      tmem_ld_32x32_issue(s_addr + 64, s0);
      tmem_ld_32x32_issue(s_addr + 96, s1);
      tmem_ld_wait();
      add_bias(s0, j * 128 + 64);
      add_bias(s1, j * 128 + 96);
      if (nvalid < 128) {
        mask_tail(s0, 64, nvalid);
        mask_tail(s1, 96, nvalid);
      }
      mx = fmaxf(mx, fmaxf(max32(s0), max32(s1)));
      const float2 nm2 = make_float2(-mx * p.scale_log2e, -mx * p.scale_log2e);
      float2 acc4[4] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
      auto exp_store = [&](const float (&v)[32], int c) {   // 32-column chunk c of the block -> P (bf16, 128B swizzle)
        const uint32_t dst = sp_row + (uint32_t)(c >> 1) * 16384u;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float2 e[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 a = __ffma2_rn(make_float2(v[q * 8 + 2 * t], v[q * 8 + 2 * t + 1]), sc2, nm2);
            e[t] = make_float2(ex2_approx(a.x), ex2_approx(a.y));
            acc4[t] = __fadd2_rn(acc4[t], e[t]);   // four independent chains
          }
          sts128(dst + ((((uint32_t)(c & 1) * 4u + (uint32_t)q) ^ sw) << 4), pack_bf16x2(e[0].x, e[0].y),
                 pack_bf16x2(e[1].x, e[1].y), pack_bf16x2(e[2].x, e[2].y), pack_bf16x2(e[3].x, e[3].y));
        }
      };
      mbar_wait(p_empty(grp), par ^ 1u);   // the P V MMAs of this group's previous block have drained the P buffer
      exp_store(s0, 2);
      exp_store(s1, 3);
      tmem_ld_32x32_issue(s_addr, s0);
      tmem_ld_32x32_issue(s_addr + 32, s1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_empty(grp));   // the MMA warp may overwrite this S buffer
      add_bias(s0, j * 128);
      add_bias(s1, j * 128 + 32);
      if (nvalid < 64) {
        mask_tail(s0, 0, nvalid);
        mask_tail(s1, 32, nvalid);
      }
      exp_store(s0, 0);
      exp_store(s1, 1);
      const float2 acc2 = __fadd2_rn(__fadd2_rn(acc4[0], acc4[1]), __fadd2_rn(acc4[2], acc4[3]));
      *pm_jj = mx;
      *pl_jj = acc2.x + acc2.y;
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full(grp));
    };

    uint32_t cblk = 0, mine = 0;
    int it = 0;
    bool pend = false, pend_first = false, pend_last = false;
    int pend_item = 0, pend_nbc = 0;
    uint32_t pend_gcx = 0;
    for (int item = blockIdx.x; item < p.num_items; item += gridDim.x, ++it) {
      if constexpr (BIAS) {
        const int qt = item % p.qtiles, h = (item / p.qtiles) % p.heads, b = item / (p.qtiles * p.heads);
        const int i = qt * 128 + row;   // padding rows (i >= T') stay inside the table's zero margins, with gate 0
        brow = p.rel_bias + (long long)h * rel_bias_ld(p.T) + REL_BIAS_PAD + (p.T - 1 - i);
        gsc = i < p.T ? p.gate[((long long)b * p.heads + h) * p.T + i] / p.scale_log2e : 0.f;
      }
#pragma unroll 1
      for (int c = 0; c < CPI; ++c) {
        const uint32_t gcx = (uint32_t)it * (uint32_t)CPI + (uint32_t)c;
        const int nbc = (NB - 2 * c) < 2 ? (NB - 2 * c) : 2;
        // (m_j, l_j) ring of four chunks: a group may run ahead of the other group's merge
        float* pm = s_m + (gcx & 3u) * (4 * 128) + row;
        float* pl = s_l + (gcx & 3u) * (4 * 128) + row;
        for (int jj = 0; jj < nbc; ++jj, ++cblk) {
          if ((cblk & 1u) != (uint32_t)grp) continue;
          block(2 * c + jj, pm + jj * 128, pl + jj * 128, mine & 1u);
          ++mine;
        }
        // every block this group owns in the chunk is published (a single-block chunk belongs to one group only: the
        // other still has to arrive) -- before the deferred merge below, so the other group's merge of this chunk never
        // waits for ours of the previous one
        __syncwarp();
        if (lane == 0) mbar_arrive(ml_full(gcx & 3u));
        if (pend) merge(pend_item, pend_gcx, pend_nbc, pend_first, pend_last);
        pend = true;
        pend_item = item;
        pend_gcx = gcx;
        pend_nbc = nbc;
        pend_first = c == 0;
        pend_last = c == CPI - 1;
      }
    }
    if (pend) merge(pend_item, pend_gcx, pend_nbc, pend_first, pend_last);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
}

bool attention_fa_supported(const AttnParams& p) {
  return p.hd == 64 && p.pos_proj == nullptr && (p.H % 8 == 0);
}

template <bool BIAS>
static cudaError_t attention_fa_set_smem() {
  cudaError_t e = cudaFuncSetAttribute(attention_fa_kernel<1, BIAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FA_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_fa_kernel<2, BIAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FA_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_fa_kernel<0, BIAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FA_SMEM);
  return e;
}

std::string attention_fa_init() {
  cudaError_t e = attention_fa_set_smem<false>();
  if (e == cudaSuccess) e = attention_fa_set_smem<true>();
  if (e != cudaSuccess) return std::string("cudaFuncSetAttribute(attention_fa_kernel): ") + cudaGetErrorString(e);
  return "";
}

std::string attention_fa_prepare(const AttnParams& p, int num_sms, AttnFaPlan** out) {
  if (!attention_fa_supported(p)) return "attention (tcgen05): unsupported shape";
  if ((p.rel_bias == nullptr) != (p.gate == nullptr)) return "attention (tcgen05): the bias table and the gate go together";
  if (p.rel_bias && p.lse) return "attention (tcgen05): the log-sum-exp is not written with a relative-position bias";
  AttnFaPlan* pl = new AttnFaPlan();
  pl->dev.ctx = p.ctx;
  pl->dev.lse = p.lse;
  pl->dev.rel_bias = p.rel_bias;
  pl->dev.gate = p.gate;
  pl->dev.B = p.B; pl->dev.T = p.T; pl->dev.H = p.H; pl->dev.heads = p.heads;
  pl->dev.qtiles = (p.T + 127) / 128;
  pl->dev.num_items = pl->dev.qtiles * p.heads * p.B;
  pl->dev.scale_log2e = p.scale * 1.4426950408889634f;
  pl->nb = (p.T + 127) / 128;
  pl->dev.nb = pl->nb;
  pl->grid = pl->dev.num_items < num_sms ? pl->dev.num_items : num_sms;
  const uint64_t ld = (uint64_t)p.ld;
  uint64_t dims[4] = {64, (uint64_t)p.T, (uint64_t)p.heads, (uint64_t)p.B};
  uint64_t str[3] = {ld * 2, 128, (uint64_t)p.T * ld * 2};
  uint32_t box[4] = {64, 128, 1, 1};
  std::string err = make_tensor_map_bf16(&pl->mapQ, p.qkv + p.q_off, 4, dims, str, box);
  if (err.empty()) err = make_tensor_map_bf16(&pl->mapK, p.qkv + p.k_off, 4, dims, str, box);
  if (err.empty()) err = make_tensor_map_bf16(&pl->mapV, p.qkv + p.v_off, 4, dims, str, box);
  if (!err.empty()) {
    delete pl;
    return err;
  }
  *out = pl;
  return "";
}

template <bool BIAS>
static cudaError_t attention_fa_launch_as(const AttnFaPlan* pl, cudaStream_t s) {
  const std::conditional_t<BIAS, AttnFaBiasDev, AttnFaDev>& dev = pl->dev;
  switch (pl->nb) {
    case 1: return launch_pdl(attention_fa_kernel<1, BIAS>, dim3(pl->grid), dim3(384), FA_SMEM, s, 1, pl->mapQ, pl->mapK, pl->mapV, dev);
    case 2: return launch_pdl(attention_fa_kernel<2, BIAS>, dim3(pl->grid), dim3(384), FA_SMEM, s, 1, pl->mapQ, pl->mapK, pl->mapV, dev);
    default: return launch_pdl(attention_fa_kernel<0, BIAS>, dim3(pl->grid), dim3(384), FA_SMEM, s, 1, pl->mapQ, pl->mapK, pl->mapV, dev);
  }
}

std::string attention_fa_launch(const AttnFaPlan* pl, cudaStream_t s) {
  W2S_CUDA_OK(pl->dev.rel_bias ? attention_fa_launch_as<true>(pl, s) : attention_fa_launch_as<false>(pl, s));
  W2S_CUDA_OK(cudaGetLastError());
  return "";
}

void attention_fa_free(AttnFaPlan* pl) { delete pl; }

}  // namespace w2s
