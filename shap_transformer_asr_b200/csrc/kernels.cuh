// Launchers of the non-GEMM kernels of the path (all sm_100a CUDA, no library calls).
#pragma once
#include "common.cuh"

namespace w2s {

// ---- K0: coalition materialisation (segment mask + baseline fill) -----------------------------------
// out[k, i] = bit(z[k], seg_id[i]) ? x[i] : baseline
std::string launch_mask(const float* x, const uint16_t* seg_id, const uint32_t* zbits, int zwords, long long K,
                        long long L, float baseline, float* out, long long ld, cudaStream_t s);
// the same with a background bg[B, bg_ld]: out[k * B + b, i] = bit(z[k], seg_id[i]) ? x[i] : bg[b, i]
std::string launch_mask_bg(const float* x, const uint16_t* seg_id, const uint32_t* zbits, int zwords, long long K,
                           long long L, const float* bg, int B, long long bg_ld, float* out, long long ld, cudaStream_t s);
// the same over time-frequency cells with band components comp[F, comp_ld]: out[k, i] = sum_{b = 0 .. F-1} (bit(z[k],
// seg_id[i] * F + b) ? comp[b, i] : 0), fp32 adds in band order from +0.0
std::string launch_mask_bands(const uint16_t* seg_id, const uint32_t* zbits, int zwords, long long K, long long L,
                              const float* comp, int F, long long comp_ld, float* out, long long ld, cudaStream_t s);

// Where the kernels that read the masked waveform take a dropped sample from (a compile-time variant of each of them):
// FILL_PLAIN the baseline (and the explicit-waveform rows), FILL_BG a background row (DynArgs::bg), FILL_BANDS the band
// components of the kept time-frequency cells (DynArgs::bands)
enum Fill : int { FILL_PLAIN = 0, FILL_BG = 1, FILL_BANDS = 2 };

// ---- per-call arguments, read by the kernels from device memory ---------------------------------------------
// Everything that may change between two evaluations of the same batch-tile plan lives here instead of in kernel
// parameters, so a plan can be captured once into a CUDA graph and replayed: one tiny kernel writes this block
// before each tile (api.cu: set_dyn_kernel), the first and the last kernels of the plan read it.
struct DynArgs {
  // input rows of this tile: explicit waveforms x[n, ld] (w2s_eval_waveforms) ...
  const float* x;
  long long ld;             // row stride of x, or of bg when a background is set
  // ... or the masker folded into the consumer's load (w2s_eval): row r = keep-bit(zbits[r], seg_id[i]) ? clip[i] :
  // baseline, so the [n, L] masked waveforms are never materialised (conformer_test.ipynb:138-141 semantics)
  const float* clip;        // [L]; null selects `x`
  const uint16_t* seg_id;   // [L]
  const uint32_t* zbits;    // [n, zwords]
  int zwords;
  float baseline;
  // output reduction (w2s_set_targets) and destination of this tile
  float* out;               // [n, width]
  int mode, D;
  const int* frames;        // [D] device
  const int* tokens;        // [D] device
  // background fill (w2s_set_background; read only by the BG instantiations of the conv0 kernels): global row g =
  // row0 + r of the call is coalition g / B filled from background row g % B, bg[b, i] = bg[b * ld + i]
  const float* bg;
  int B;
  long long row0;
  // CTC transcripts (w2s_set_transcripts; mode W2S_OUT_CTC, D transcripts): transcript d is ctc_labels[ctc_offsets[d] ..
  // ctc_offsets[d + 1]), with blank id `blank`
  const int* ctc_labels;
  const int* ctc_offsets;   // [D + 1]
  int blank;
  // time-frequency cells (w2s_set_bands; read only by the FILL_BANDS instantiations): F band components bands[b * ld + i],
  // zbits rows hold one bit per cell, bit s * F + b for time segment s and band b
  const float* bands;
  int F;
};

// ---- K1: conv0 (Cin = 1) + GroupNorm-over-time / LayerNorm-over-channels + GELU ------------------------
struct Conv0Params {
  const DynArgs* dyn;    // input rows (device)
  int n, L, T0, C, kw, stride;
  const float* w;        // [C][kw] fp32
  const float* bias;     // [C] or null
  const float* gamma;    // [C]
  const float* beta;     // [C]
  // group-norm variant: per (row, channel) affine produced by the statistics kernel
  float* gn_a;           // [n, C]  rstd * gamma
  float* gn_b;           // [n, C]  beta - mean * rstd * gamma
  __nv_bfloat16* gn_wb;  // [n, C, 32] (optional) filters with the affine folded in, split into bf16 hi/lo terms:
                         //            the B operand of conv0_mma_kernel
  // layer-norm variant: channel statistics of the filter bank (precomputed once)
  const float* ln_wbar;  // [kw]       mean_c w[c][j]
  const float* ln_gram;  // [kw][kw]   mean_c w[c][j] w[c][j']
  const float* ln_wb;    // [kw]       mean_c w[c][j] b[c]
  float ln_bmean, ln_b2mean;
  int pre_act;           // 1: store the normalised pre-activation (no GELU) -- forward of the gradient path
  float* ln_rstd_out;    // [n, T0] (optional, layer-norm variant with pre_act): per-frame rstd, kept for the backward pass
  const __nv_bfloat16* ln_wb48;  // [C][48] (optional) B operand of conv0_ln_mma_kernel: filters, bias and affine terms
                                 // as bf16 hi/lo rows
  __nv_bfloat16* out;    // [n, T0, C] channels-last
};
// fill: which instantiation reads the input rows (Fill); FILL_PLAIN serves the baseline fill and explicit waveforms
std::string launch_conv0_stats(const Conv0Params& p, cudaStream_t s, int fill = FILL_PLAIN);   // group-norm statistics
std::string launch_conv0(const Conv0Params& p, bool layer_norm, cudaStream_t s, int fill = FILL_PLAIN);
// B operand of the tensor-core layer-norm variant (run once at create)
std::string launch_conv0_ln_b(const float* w, const float* bias, const float* gamma, const float* beta, int C, int kw,
                              __nv_bfloat16* out, cudaStream_t s);
// filter-bank statistics for the layer-norm variant (run once at create)
std::string launch_conv0_ln_prep(const float* w, const float* bias, int C, int kw, float* wbar, float* gram,
                                 float* wb, float* scalars /*[2]: mean b, mean b^2*/, cudaStream_t s);

// ---- LayerNorm over the last dimension (fp32 or bf16 in, bf16 out), optional activation ---------------
// `residual` (bf16, optional): normalises in + residual (post-LN transformer blocks)
std::string launch_layernorm(const void* in, int in_fp32, long long rows, int H, const float* gamma,
                             const float* beta, float eps, int act, __nv_bfloat16* out, float* out_f32,
                             cudaStream_t s, const __nv_bfloat16* residual = nullptr);

// ---- positional-conv input staging: [B, T, H] -> zero-padded [B, T + kpos, G*64] ------------------------
// `left` = zero rows in front of frame 0 (default kpos / 2, HF's padding; the backward-data conv uses kpos / 2 - 1)
std::string launch_pos_pad(const __nv_bfloat16* h, int B, int T, int H, int G, int kpos, __nv_bfloat16* out,
                           cudaStream_t s, int left = -1);

// ---- K4: positional conv on tcgen05 with a resident input window (posconv.cu) --------------------------------
struct EpiParams;
struct PosConvPlan;
std::string posconv_init();
bool posconv_supported(int H, int G, int kpos);
std::string posconv_prepare(const __nv_bfloat16* x, const __nv_bfloat16* w, int B, int T, int H, int G, int kpos,
                            const EpiParams& epi, int num_sms, PosConvPlan** out);
std::string posconv_launch(const PosConvPlan* plan, cudaStream_t s);
void posconv_free(PosConvPlan* plan);

// ---- attention -------------------------------------------------------------------------------------
struct AttnParams {
  const __nv_bfloat16* qkv;   // [B*T, ld]: plain models (q | k | v), ld = 3H; conformer relative (q+u | q+v | k | v), ld = 4H
  __nv_bfloat16* ctx;         // [B*T, H]
  int B, T, Tp, H, heads, hd;
  int ld, q_off, qv_off, k_off, v_off;  // column offsets inside a qkv row (qv_off used with pos_proj only)
  float scale;
  // conformer relative positions (null when unused): the biases u / v are already folded into the q+u / q+v columns
  const __nv_bfloat16* pos_proj;  // [2T-1, H] linear_pos(rel_pos_emb), row r <-> relative position T-1-r
  float* lse;                     // optional (attention_fa only): [B, heads, T] log2-domain log-sum-exp, saved for the backward
  // WavLM gated relative-position bias (null when unused; attention_fa and the CUDA-core kernel): score[i, j] +=
  // gate[b, h, i] * E[bucket(j - i), h].  rel_bias[h][REL_BIAS_PAD + T - 1 + j - i] = E[bucket(j - i), h] * log2(e), fp32,
  // with REL_BIAS_PAD zeros on both sides (rows rel_bias_ld(T) apart), so the padding queries and keys of a 128-wide
  // tile index inside the table
  const float* rel_bias;
  const float* gate;              // [B, heads, T] fp32
};
constexpr int REL_BIAS_PAD = 128;
__host__ __device__ constexpr int rel_bias_ld(int T) { return 2 * T - 1 + 2 * REL_BIAS_PAD; }
// rel_bias table of AttnParams, [heads, rel_bias_ld(T)]: from E [num_buckets, heads] and bucket[2T-1] (entry r <->
// relative position r - (T-1)), or, with bucket == null, from a full natural-units table src [heads, 2T-1]
std::string launch_rel_bias_table(const float* src, const int32_t* bucket, int T, int heads, float* out, cudaStream_t s);
// WavLM gate (HF wavlm/modeling_wavlm.py:166-176), head_dim 64: x [B*T, heads*64] bf16 (the attention input), w [8, 64],
// b [8], c [heads] -> gate[B, heads, T] = a (c_h b' - 1) + 2, (a, b') = sigmoid(sums of 4 of the 8 outputs W x_h + b)
std::string launch_wavlm_gate(const __nv_bfloat16* x, int B, int T, int heads, const float* w, const float* b,
                              const float* c, float* gate, cudaStream_t s);
std::string launch_attention_simt(const AttnParams& p, cudaStream_t s);
// persistent, warp-specialised tcgen05 kernel with independent key blocks (attention_fa.cu)
struct AttnFaPlan;
std::string attention_fa_init();
bool attention_fa_supported(const AttnParams& p);
std::string attention_fa_prepare(const AttnParams& p, int num_sms, AttnFaPlan** plan);
std::string attention_fa_launch(const AttnFaPlan* plan, cudaStream_t s);
void attention_fa_free(AttnFaPlan* plan);
// fused attention backward (attention_bwd.cu): delta + one persistent tcgen05 kernel + dQ cast; needs the forward's lse
struct AttnBwdPlan;
std::string attention_bwd_init();
bool attention_bwd_supported(const AttnParams& p);
std::string attention_bwd_prepare(const AttnParams& p, const __nv_bfloat16* dctx, const float* lse, float* delta, float* dq,
                                  __nv_bfloat16* dqkv, int num_sms, AttnBwdPlan** plan);
std::string attention_bwd_launch(const AttnBwdPlan* plan, const __nv_bfloat16* dctx, const __nv_bfloat16* ctx, int q_off,
                                 cudaStream_t s);
void attention_bwd_free(AttnBwdPlan* plan);
// conformer relative-position attention on tcgen05
struct AttnRelPlan;
std::string attention_rel_init();
bool attention_rel_supported(const AttnParams& p);
std::string attention_rel_prepare(const AttnParams& p, AttnRelPlan** plan);
std::string attention_rel_launch(const AttnRelPlan* plan, cudaStream_t s);
void attention_rel_free(AttnRelPlan* plan);

// ---- conformer-only CUDA-core kernels (conformer.cu) ---------------------------------------------------------
std::string launch_bn_fold(const float* g, const float* b, const float* mean, const float* var, int n, float eps,
                           float* scale, float* shift, cudaStream_t s);
// w: depthwise taps stored [k][H] (transposed from the HF [H][1][k] layout)
std::string launch_depthwise(const __nv_bfloat16* in, int B, int T, int H, int k, const float* w, const float* scale,
                             const float* shift, int act, __nv_bfloat16* out, cudaStream_t s);
std::string launch_transpose_f32(const float* src, float* dst, int R, int C, cudaStream_t s);
// inverse = 1 applies the transposed rotation (the backward of the forward one)
std::string launch_rotary(const __nv_bfloat16* x, long long rows, int T, int H, int hd, int base, __nv_bfloat16* out,
                          cudaStream_t s, int inverse = 0);
std::string launch_relpos(int T, int H, __nv_bfloat16* out, cudaStream_t s);

// ---- K9: lm_head + log-softmax + gather -----------------------------------------------------------------
struct HeadParams {
  const __nv_bfloat16* h;     // [n*T, H]
  const __nv_bfloat16* w;     // [V, H]
  const float* bias;          // [V]
  int n, T, H, V;
  int ldl;                    // row stride of the logits buffer (V rounded up to a multiple of 32)
  const DynArgs* dyn;         // mode, targets and output pointer of this call (device)
};
// CUDA-core validation variant (W2S_FLAG_VALIDATE_GEMM): lm_head + reduction in one kernel
std::string launch_head(const HeadParams& p, cudaStream_t s);
// tensor-core variant: the contraction kernel writes logits[n*T, ldl] (fp32, bias added), this reduces them
std::string launch_head_reduce(const float* logits, const HeadParams& p, cudaStream_t s);
// background mean: out[k, c] = sum_b w[b] * rows[k * B + b, c] (fp32, one fmaf per term from 0, b = 0 .. B-1)
std::string launch_bg_mean(const float* rows, const float* w, int B, long long K, long long width, float* out,
                           cudaStream_t s);

// ---- K12: KernelSHAP constrained WLS -----------------------------------------------------------------------
std::string launch_wls(const uint32_t* zbits, int zwords, const double* w, const float* y, long long K, int M,
                       int D, const double* fx, const double* fnull, double* phi, int32_t* status,
                       double* work /* 2 * ((M-1)*(M-1) + (M-1)*D) doubles */, cudaStream_t s);

// ---- backward (input-gradient) kernels of the expected-gradients path (grad.cu) -------------------------------------
std::string launch_gelu_fwd(const __nv_bfloat16* u, __nv_bfloat16* y, long long n, cudaStream_t s);
std::string launch_gelu_bwd(const __nv_bfloat16* u, __nv_bfloat16* d, long long n, cudaStream_t s);
std::string launch_add_gelu(const __nv_bfloat16* h0, const __nv_bfloat16* up, float* out, long long n, cudaStream_t s);
std::string launch_grad_cast(const float* g, const __nv_bfloat16* u, __nv_bfloat16* out, long long n, cudaStream_t s);
// dy: fp32, or bf16 when dy_fp32 == 0 (then dx16 may alias dy: a warp reads its row before writing it)
std::string launch_ln_bwd(const void* dy, const void* x, int x_fp32, long long rows, int H, const float* gamma, float eps,
                          const float* add, float* dx, __nv_bfloat16* dx16, cudaStream_t s, int dy_fp32 = 1);
// conv0 + LayerNorm over channels (layer-norm front ends), backward to the waveform
std::string launch_conv0_ln_bwd(const __nv_bfloat16* du, const __nv_bfloat16* u, const float* rstd, int n, long long L, int T0, int C,
                                int kw, int stride, const float* w, const float* gamma, const float* beta, float* g, float* dx,
                                long long ld, cudaStream_t s);
std::string launch_head_bwd(const float* logits, int ldl, int V, const __nv_bfloat16* w_head, int n, int T, int H,
                            const int* frames, float* dh, float* out_val, cudaStream_t s, int active = -1);
// CTC seed (ctc.cuh) of w2s_grad_transcripts: for row r and transcript which[r], out_val[r] = log p and
// dz[r, t, v] = d log p / d logits[r, t, v] (row stride ldz), then, when dh is given, dh[r, t, :] = dz[r, t, :] W_head.
// alpha: scratch [n, T, s_max] with s_max >= 2 U + 1 of every transcript used, lse: scratch [n, T]
std::string launch_ctc_seed(const float* logits, int ldl, int V, const __nv_bfloat16* w_head, int n, int T, int H,
                            const int* labels, const int* offsets, const int* which, int blank, int s_max, float* alpha,
                            float* lse, float* dz, int ldz, float* dh, float* out_val, cudaStream_t s);
std::string launch_head_vjp(const float* logits, int ldl, int V, const __nv_bfloat16* w_head, int n, int T, int H,
                            const float* gout, float* dh, float* out_all, cudaStream_t s);
std::string launch_attn_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* dctx, int B, int T, int H, int heads, float scale,
                            __nv_bfloat16* dqkv, float* stats, cudaStream_t s);
// bd != null: relative-position scores [BH, T, Rp] added with the rel-shift index arithmetic while the row is read
std::string launch_attn_softmax_t(const float* S, int BH, int T, int Tp, __nv_bfloat16* P, __nv_bfloat16* PT, cudaStream_t s,
                                  const float* bd = nullptr, int Rp = 0);
std::string launch_attn_ds_t(const __nv_bfloat16* P, const float* dP, int BH, int T, int Tp, __nv_bfloat16* dS,
                             __nv_bfloat16* dST, cudaStream_t s);
std::string launch_head_transpose(const __nv_bfloat16* src, int ld, int off, int B, int T, int Tp, int heads, __nv_bfloat16* dst,
                                  cudaStream_t s);
std::string launch_conv_gather(const __nv_bfloat16* dcol, int n, int T_in, int T_out, int C, int kw, int stride,
                               const __nv_bfloat16* u_prev, __nv_bfloat16* out, cudaStream_t s);
// conv0 + GroupNorm over time, backward to the waveform.  m12: scratch of n * C * (3 + 64) floats (per-(row, channel)
// coefficients + 32 time-chunk partial sums); g: scratch [n, T0, kw]
std::string launch_conv0_bwd(const __nv_bfloat16* du, const __nv_bfloat16* u, int n, long long L, int T0, int C, int kw, int stride,
                             const float* w, const float* gn_a, const float* gamma, const float* beta, float* m12, float* g,
                             float* dx, long long ld, cudaStream_t s);
// conformer encoder pieces of the gradient path
std::string launch_act_fwd(const __nv_bfloat16* u, __nv_bfloat16* y, long long n, int act, cudaStream_t s);
// paired: rows are [explained | reference] halves and the explained half uses the DeepLIFT rescale multiplier
std::string launch_act_bwd(const __nv_bfloat16* u, __nv_bfloat16* d, long long n, int act, const float* chan_scale, int H,
                           cudaStream_t s, int paired = 0);
std::string launch_glu_fwd(const __nv_bfloat16* raw, __nv_bfloat16* out, long long n, cudaStream_t s);
std::string launch_glu_bwd(const __nv_bfloat16* raw, const __nv_bfloat16* dout, __nv_bfloat16* draw, long long n, cudaStream_t s,
                           int placeholder_paired = 0);
std::string launch_rel_unshift(const __nv_bfloat16* dS, __nv_bfloat16* dBD, int BH, int T, int Tp, int Rp, cudaStream_t s);
std::string launch_flip_taps(const float* src, float* dst, int k, int H, cudaStream_t s);
std::string launch_fill_f32(float* dst, float v, int n, cudaStream_t s);
std::string launch_transpose_bf16(const __nv_bfloat16* src, __nv_bfloat16* dst, int R, int C, cudaStream_t s);
std::string launch_repack_posconv_bwd(const float* src, __nv_bfloat16* dst, int H, int G, int kw, cudaStream_t s);

// ---- weight re-layout (run once at create) -------------------------------------------------------------------
// y[i] += x[i]
std::string launch_axpy(const float* x, float* y, int n, cudaStream_t s);
std::string launch_cast_bf16(const float* src, __nv_bfloat16* dst, long long n, cudaStream_t s);
// conv weight [O][C][kw] fp32 -> [O][j*C + c] bf16
std::string launch_repack_conv(const float* src, __nv_bfloat16* dst, int O, int C, int kw, cudaStream_t s);
// positional conv weight [H][cpg][kw] fp32 -> [G][cpg][kw*64 + c] bf16 (zero for c >= cpg)
std::string launch_repack_posconv(const float* src, __nv_bfloat16* dst, int H, int G, int kw, cudaStream_t s);
// rows interleaved for the GLU epilogue: dst[2j] = src[j], dst[2j+1] = src[j + half]
std::string launch_repack_glu(const float* src, __nv_bfloat16* dst, int half, int K, cudaStream_t s);

}  // namespace w2s
