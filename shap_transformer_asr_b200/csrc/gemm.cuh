// Contraction engine of the path: one persistent, warp-specialised tcgen05/TMEM/TMA kernel that serves
// every dense contraction of the Wav2Vec2 forward (strided conv layers as implicit GEMM, feature
// projection, grouped positional conv, QKV / out-proj / FFN, conformer pointwise convs), plus the
// CUDA-core validation kernel that computes the same thing from the same bf16 buffers.
#pragma once
#include "common.cuh"

namespace w2s {

// Epilogue: v = act(acc + bias[n]); (glu: v = val * sigmoid(gate)); v = v * alpha + residual; store.
struct EpiParams {
  const float* bias = nullptr;     // [G * N]
  int act = ACT_NONE;
  int glu = 0;                     // columns are (value, gate) pairs; output column = n / 2
  float alpha = 1.0f;
  const void* residual = nullptr;  // same indexing as out
  int res_fp32 = 0;
  void* out = nullptr;
  int out_fp32 = 0;
  long long ldg = 0, ldb = 0, ldm = 0;  // element strides of (group, batch, row); columns contiguous
};

// C[g, b] (M x N) = A[g, b] (M x K) * W[g]^T (N x K).
// A is a bf16 2-D view per batch (a_rows x a_cols, row stride a_row_stride) and K is walked in 64-wide
// blocks: block kb reads columns [g*a_g_col + (kb % a_kb_per_row)*64, +64) of rows m + (kb / a_kb_per_row).
//   plain GEMM      : a_kb_per_row = K/64
//   strided conv    : view = [ceil(T_in/stride), stride*C]  ("stride-rows"), a_kb_per_row = stride*C/64
//   positional conv : view = [T+pad, G*64], a_kb_per_row = 1 (one tap per block), a_g_col = 64
//   per-(batch, head) operands (attention backward): a_g_col = 64 selects a head's columns of a [rows, n_heads*64]
//   buffer, a_g_row = T its row block of a [batch][head][T][K] buffer; W may be batched as well (w_batch_stride != 0)
//   with its own row / group strides, and may hold fewer than N rows (w_rows; the tiles past them are zero-filled)
struct GemmProblem {
  const __nv_bfloat16* a = nullptr;
  long long a_cols = 0, a_rows = 0, a_batches = 1;
  long long a_row_stride = 0, a_batch_stride = 0;  // elements
  int a_kb_per_row = 1, a_g_col = 0, a_g_row = 0;
  const __nv_bfloat16* w = nullptr;  // [G][N][K] unless the strides below say otherwise
  long long w_row_stride = 0, w_g_stride = 0, w_batch_stride = 0;   // elements; 0 = K, N*K, "shared by all batches"
  int w_rows = 0;                                                   // rows present per (group, batch); 0 = N
  int M = 0, N = 0, K = 0, Bz = 1, G = 1;
  EpiParams epi;
};

struct GemmDev {
  int M, N, K, Bz, G;
  int tiles_m, tiles_n, num_tiles, num_kb;
  int units_m, num_units;  // scheduling units: tiles, or M-pairs of tiles for the CTA-pair kernel
  int a_kb_per_row, a_g_col, a_g_row;
  int w_batched;   // W has a batch dimension (4th TMA coordinate = batch index)
  // validation-kernel addressing
  const __nv_bfloat16* a;
  const __nv_bfloat16* w;
  long long a_cols, a_rows, a_row_stride, a_batch_stride;
  EpiParams epi;
};

struct GemmLaunch {
  CUtensorMap mapA, mapW;
  CUtensorMap mapOut;   // pair kernel: output tile written by TMA stores from a swizzled staging strip
  int tma_out = 0;
  GemmDev dev;
  int bn = 0;
  int mc = 0;   // 2: CTA pairs form one tcgen05.mma cta_group::2 unit (256-row tile, W split across the pair); 0: one CTA per tile
  int grid = 0;
  size_t smem = 0;
};

std::string gemm_prepare(const GemmProblem& p, int num_sms, GemmLaunch* out);
std::string gemm_launch_tc(const GemmLaunch& l, cudaStream_t s);
std::string gemm_launch_simt(const GemmLaunch& l, cudaStream_t s);
std::string gemm2_init();
std::string gemm2_launch(const GemmLaunch& l, cudaStream_t s);
// the pair kernel over a device list of 128-row blocks (list[0] = count, then (batch << 16) | block); l.grid as prepared
std::string gemm2_launch_list(const GemmLaunch& l, const int* list, cudaStream_t s);
std::string gemm_init();  // resolves cuTensorMapEncodeTiled, sets kernel attributes

// shared by other translation units that build their own tensor maps (attention)
std::string make_tensor_map_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                                 const uint64_t* strides_bytes, const uint32_t* box);
std::string make_tensor_map(CUtensorMap* map, const void* base, int fp32, int rank, const uint64_t* dims,
                            const uint64_t* strides_bytes, const uint32_t* box);

}  // namespace w2s
