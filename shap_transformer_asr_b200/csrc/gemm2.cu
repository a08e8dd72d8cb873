// CTA-pair contraction kernel: tcgen05.mma cta_group::2, 256 x BN output tile per pair of SMs.
//
// Same roles and pipelines as gemm_tc_kernel, but the two CTAs of a cluster form one MMA unit:
//   * each CTA's TMA producer loads ITS 128 rows of A and ITS half (BN/2 rows) of the W tile -- 32 KB per stage
//     instead of 48 KB, so the tensor core's operand reads plus the TMA fills fit the shared-memory bandwidth
//     (a single CTA needs 96 + 96 B/clk for a 128x256 tile; a pair member needs 64 + 64 B/clk);
//   * both producers report their bytes to the LEADER's full barrier; the leader's MMA thread issues
//     tcgen05.mma.cta_group::2 (M = 256) and commits to the empty / tmem_full barriers of BOTH CTAs;
//   * each CTA's epilogue warps drain their own 128 accumulator rows from their own TMEM and release the
//     accumulator slot on the leader's tmem_empty barrier.
#include "gemm.cuh"
#include "gemm_epi.cuh"

namespace w2s {

template <int BN>
struct Tc2Cfg {
  static constexpr int A_BYTES = 128 * 64 * 2;
  static constexpr int B_BYTES = (BN / 2) * 64 * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int EPI_BYTES = 8 * 4096 + 8 * 512;   // per-warp 32 x 128 B output staging + bias strip
  // the operand ring takes what the epilogue strips leave: 5 x 32 KB (BN = 256) or 7 x 24 KB (BN = 128)
  static constexpr int STAGES = (227 * 1024 - 1024 - 256 - EPI_BYTES) / STAGE_BYTES > 8
                                    ? 8 : (227 * 1024 - 1024 - 256 - EPI_BYTES) / STAGE_BYTES;
  static constexpr int ACC_COLS = BN;
  static constexpr int TMEM_COLS = 2 * ACC_COLS;
  static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + EPI_BYTES + 1024 + 256;
};

// LIST: the 128-row blocks come from a device list instead of the dense (n-tile, m-pair, batch) walk (feature-encoder
// convolutions, frontend_skip.cu): list[0] is the count, list[1 + e] = (batch << 16) | block.  Rank r of a pair takes
// entry 2u + r, so a pair may join blocks of two coalitions (the CTAs share only the W half-tiles); a missing partner of
// an odd count computes a block past the output and stores nothing.  The grid stays as captured, the count is read here.
template <int BN, bool LIST = false>
__global__ void __launch_bounds__(384, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW,
                const __grid_constant__ CUtensorMap mapOut, const GemmDev p, const int tma_out,
                const int* __restrict__ list = nullptr) {
  using C = Tc2Cfg<BN>;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int unit0 = (int)(blockIdx.x >> 1), unit_step = (int)(gridDim.x >> 1);
  const int list_n = LIST ? list[0] : 0;
  const int num_units = LIST ? (list_n + 1) / 2 * p.tiles_n : p.num_units;
  // list entry of this CTA in unit `unit`: (batch, first row); a list dummy gets a row past the output
  auto list_block = [&](int unit, int& b, int& m0) {
    const int e = 2 * (unit / p.tiles_n) + (int)rank;
    const int v = e < list_n ? __ldg(list + 1 + e) : -1;
    b = v < 0 ? 0 : v >> 16;
    m0 = v < 0 ? p.units_m * 256 : (v & 0xffff) * 128;
  };
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t tiles = (raw + 1023u) & ~1023u;
  uint8_t* tiles_ptr = smem_raw + (tiles - raw);
  const uint32_t epi_smem = tiles + C::STAGES * C::STAGE_BYTES;   // 1024-aligned: staging strips, then bias strips
  const uint32_t bars = epi_smem + C::EPI_BYTES;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (C::STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * C::STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * C::STAGES + 2 + a); };
  const uint32_t tmem_slot = bars + 8u * (2 * C::STAGES + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(tiles_ptr + C::STAGES * C::STAGE_BYTES + C::EPI_BYTES + 8 * (2 * C::STAGES + 4));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&mapA);
    tma_prefetch_desc(&mapW);
    if (tma_out) tma_prefetch_desc(&mapOut);
  }
  if (warp == 9 && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(full_bar(s), 1);    // the leader's arrive.expect_tx covers the bytes of BOTH producers (used in the leader only)
      mbar_init(empty_bar(s), 1);   // the leader's MMA commit, multicast to both CTAs
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 16);  // 8 epilogue warps of each CTA (used in the leader only)
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 10) {
    tmem_alloc_2sm<C::TMEM_COLS>(tmem_slot);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 8) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = unit0; unit < num_units; unit += unit_step) {
        int nt = unit % p.tiles_n;
        int r = unit / p.tiles_n;
        const int mu = r % p.units_m;
        r /= p.units_m;
        int b = r % p.Bz, g = r / p.Bz;
        int m0 = (2 * mu + (int)rank) * 128;
        if constexpr (LIST) {
          list_block(unit, b, m0);
          g = 0;
        }
        const int n0 = nt * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t full_leader = mapa_u32(full_bar(stage), 0);
          // The peer's bytes may land before the leader has armed the phase (the tx-count just goes negative);
          // they cannot land in a later phase because the peer's slot is only freed by the leader's MMA commit.
          if (leader) mbar_expect_tx(full_bar(stage), 2 * C::STAGE_BYTES);
          const int krow = kb / p.a_kb_per_row;
          const int kcol = kb - krow * p.a_kb_per_row;
          const uint32_t sa = tiles + stage * C::STAGE_BYTES;
          tma_load_3d_2sm(sa, &mapA, full_leader, g * p.a_g_col + kcol * 64, g * p.a_g_row + m0 + krow, b);
          tma_load_4d_2sm(sa + C::A_BYTES, &mapW, full_leader, kb * 64, n0 + (int)rank * (BN / 2), g, p.w_batched ? b : 0);
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 9) {
    if (leader && elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int unit = unit0; unit < num_units; unit += unit_step) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * C::ACC_COLS;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = tiles + stage * C::STAGE_BYTES;
          const uint64_t da = umma_desc_sw128(sa);
          const uint64_t db = umma_desc_sw128(sa + C::A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16_2sm(d_tmem, da + 2u * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_2sm_mc(empty_bar(stage), (uint16_t)0x3);
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit_2sm_mc(tfull_bar(acc), (uint16_t)0x3);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else if (warp < 8) {
    const int q = warp & 3, hsel = warp >> 2;
    const bool lead = elect_one();   // the lane that owns this warp's TMA-store bulk groups
    const uint32_t stg = epi_smem + warp * 4096;              // this warp's 32 rows x 128 B staging strip
    const uint32_t stg_row = stg + lane * 128;
    float* sbias = reinterpret_cast<float*>(tiles_ptr + C::STAGES * C::STAGE_BYTES + 8 * 4096 + warp * 512);
    const bool f32 = p.epi.out_fp32 != 0;
    // in-place fp32 accumulation (out == residual): let the TMA engine add in L2 instead of loading the residual
    const bool reduce_add = tma_out && f32 && p.epi.res_fp32 && p.epi.residual == p.epi.out;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = unit0; unit < num_units; unit += unit_step) {
      int nt = unit % p.tiles_n;
      int r = unit / p.tiles_n;
      const int mu = r % p.units_m;
      r /= p.units_m;
      int b = r % p.Bz, g = r / p.Bz;
      int m0 = (2 * mu + (int)rank) * 128;
      if constexpr (LIST) {
        list_block(unit, b, m0);
        g = 0;
      }
      const int n0 = nt * BN;
      const bool store = !LIST || m0 < p.M;
      const int m = m0 + q * 32 + lane;
      const bool row_ok = m < p.M;
      const uint32_t t0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * C::ACC_COLS;
      if (tma_out) {
        // Column ownership: blocks of 128 B of output (32 fp32 / 64 bf16 columns); warps 0..3 take the even blocks of
        // their lane quadrant, warps 4..7 the odd ones.  The bias values of the warp's columns are fetched into its
        // shared-memory strip BEFORE the accumulator wait, so the global latency hides behind the MMAs.
        const int bw = f32 ? 32 : 64;
        const int nblk = BN / (2 * bw);
        if (p.epi.bias) {
          for (int i = lane; i < nblk * bw; i += 32) {
            const int col = (2 * (i / bw) + hsel) * bw + (i % bw);
            sbias[i] = __ldg(p.epi.bias + (long long)g * p.N + n0 + col);
          }
        }
        __syncwarp();
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        // 32-column sub-blocks of this warp, software-pipelined: the TMEM load of sub-block s+1 is in flight while the
        // values of s are written to the staging strip, and the wait for the TMA engine to have read the strip (previous
        // store) comes after the math of the sub-block instead of before its load.
        const int nsub = f32 ? nblk : 2 * nblk;
        auto sub_col = [&](int sidx) { return f32 ? (2 * sidx + hsel) * 32 : (2 * (sidx >> 1) + hsel) * 64 + (sidx & 1) * 32; };
        float v[32];
        tmem_ld_32x32_issue(t0 + sub_col(0), v);
#pragma unroll 1
        for (int sidx = 0; sidx < nsub; ++sidx) {
          const int c = sub_col(sidx);
          const int sub = f32 ? 0 : (sidx & 1);
          tmem_ld_wait();
          epi_math32(p.epi, p.epi.bias ? sbias + sidx * 32 : nullptr, p.N, g, b, m, n0 + c, row_ok, v, reduce_add);
          if (f32) {
            if (lead) tma_store_wait_read();   // the previous store of this warp has drained the strip
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; ++j)
              sts128(stg_row + (((uint32_t)j ^ ((uint32_t)lane & 7u)) << 4), __float_as_uint(v[4 * j]),
                     __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
            if (sidx + 1 < nsub) tmem_ld_32x32_issue(t0 + sub_col(sidx + 1), v);
          } else {
            uint32_t pk[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
            if (sidx + 1 < nsub) tmem_ld_32x32_issue(t0 + sub_col(sidx + 1), v);
            if (sub == 0) {
              if (lead) tma_store_wait_read();
              __syncwarp();
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
              sts128(stg_row + (((uint32_t)(sub * 4 + j) ^ ((uint32_t)lane & 7u)) << 4), pk[4 * j], pk[4 * j + 1],
                     pk[4 * j + 2], pk[4 * j + 3]);
          }
          if (f32 || sub == 1) {
            const int cblk = f32 ? c : c - 32;
            fence_proxy_async();
            __syncwarp();
            if (lead && store) {
              if (reduce_add) tma_reduce_add_4d(&mapOut, stg, n0 + cblk, m0 + q * 32, b, g);
              else tma_store_4d(&mapOut, stg, n0 + cblk, m0 + q * 32, b, g);   // rows >= M are clipped by the tensor map
              tma_store_commit();
            }
          }
        }
      } else {
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
#pragma unroll 1
        for (int c = hsel * 32; c < BN; c += 64) {
          float v[32];
          tmem_ld_32x32(t0 + c, v);
          if (row_ok) epi_store<32>(p.epi, p.N, g, b, m, n0 + c, v);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(tempty_bar(acc));
        else mbar_arrive_cluster(mapa_u32(tempty_bar(acc), 0));
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
    if (tma_out && lead) tma_store_wait_all();   // global writes complete before the CTA retires
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc_2sm<C::TMEM_COLS>(tmem_base);
  }
}

std::string gemm2_init() {
  cudaError_t e = cudaFuncSetAttribute(gemm_tc2_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)Tc2Cfg<256>::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(gemm_tc2_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Tc2Cfg<128>::SMEM);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(gemm_tc2_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)Tc2Cfg<256>::SMEM);
  if (e != cudaSuccess) return std::string("cudaFuncSetAttribute(gemm_tc2_kernel): ") + cudaGetErrorString(e);
  return "";
}

size_t gemm2_smem(int bn) { return bn == 256 ? Tc2Cfg<256>::SMEM : Tc2Cfg<128>::SMEM; }

template <int BN>
static cudaError_t launch2(const GemmLaunch& l, cudaStream_t s) {
  return launch_pdl(gemm_tc2_kernel<BN>, dim3(l.grid), dim3(384), Tc2Cfg<BN>::SMEM, s, 2, l.mapA, l.mapW,
                    l.tma_out ? l.mapOut : l.mapA, l.dev, l.tma_out, (const int*)nullptr);
}

std::string gemm2_launch_list(const GemmLaunch& l, const int* list, cudaStream_t s) {
  if (l.mc != 2 || l.bn != 256 || !l.tma_out || l.dev.G != 1) return "gemm (block list): needs the TMA-store pair kernel, BN = 256";
  W2S_CUDA_OK(launch_pdl(gemm_tc2_kernel<256, true>, dim3(l.grid), dim3(384), Tc2Cfg<256>::SMEM, s, 2, l.mapA, l.mapW,
                         l.mapOut, l.dev, l.tma_out, list));
  return "";
}

std::string gemm2_launch(const GemmLaunch& l, cudaStream_t s) {
  if (l.bn == 256) W2S_CUDA_OK(launch2<256>(l, s));
  else if (l.bn == 128) W2S_CUDA_OK(launch2<128>(l, s));
  else return "gemm (CTA pair): BN must be 256 or 128";
  return "";
}

}  // namespace w2s
