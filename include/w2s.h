/*
 * w2s.h -- C ABI of the B200-native masked-coalition evaluation path ("wave-to-scores").
 *
 * Drop-in boundary for ONE path of HagenMarin/SHAP-Transformer-ASR: the model-evaluation
 * callback an explainer invokes on masked audio coalitions.  Every entry point names the
 * reference interface it replaces (paths relative to the reference repo; HF = the
 * third-party `transformers` package the reference imports).
 *
 * Conventions: extern "C", plain pointers and sizes, `int` status (0 = ok, non-zero =
 * error; text via w2s_last_error) -- no C++ exceptions and no torch types cross this
 * boundary.  The caller owns every buffer it passes; the handle owns weights, workspace
 * and plans.  Calls are asynchronous on the given CUDA stream (cudaStream_t passed as
 * void*), with no hidden device synchronisation unless stated.  One handle per
 * (device, stream); a handle is not re-entrant.  There is no CPU fallback: every entry
 * point fails with an error when no sm_100 device is present.
 */
#ifndef W2S_H_
#define W2S_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct w2s_handle w2s_handle;

#define W2S_MAX_CONV_LAYERS 8

/* Output reductions (w2s_set_targets `mode`). */
enum {
  W2S_OUT_MAX     = 0, /* max logit per frame           -> [n, T']  shap_calculation.py:50            */
  W2S_OUT_LOGIT   = 1, /* logits[:, t_d, tok_d]          -> [n, D]   feasability_tests/w2v2conformer.py:40-42 */
  W2S_OUT_LOGPROB = 2, /* log_softmax(logits)[t_d,tok_d] -> [n, D]   north-star per-character CTC output      */
  W2S_OUT_MEAN    = 3, /* mean over vocab and time       -> [n, 1]   lime_shap_wav2vec2_comparison.py:68-70   */
  W2S_OUT_LOGITS  = 4, /* raw logits                     -> [n, T', V]  (target selection, parity tests)      */
  W2S_OUT_CTC     = 5  /* log p_CTC(y_d | all frames)     -> [n, D]   set by w2s_set_transcripts only            */
};

/* w2s_config.flags */
enum {
  W2S_FLAG_VALIDATE_GEMM = 1,  /* run every contraction on the CUDA-core validation kernels (same bf16 data) */
  W2S_FLAG_VALIDATE_ATTN = 2,  /* run attention on the CUDA-core validation kernel                            */
  W2S_FLAG_FP32_PRELN    = 4,  /* post-LN models: fp32 (instead of bf16) pre-LayerNorm tensors -- A/B measurement */
  W2S_FLAG_NO_GRAPH      = 16  /* launch the kernels of a tile one by one instead of replaying a CUDA graph        */
};

/* Mirrors transformers.Wav2Vec2Config / Wav2Vec2ConformerConfig (the objects the reference
 * obtains from from_pretrained at shap_calculation.py:218-219, w2v2conformer.py:58-59) / WavLMConfig. */
typedef struct {
  int32_t kind;                 /* 0 = Wav2Vec2ForCTC, 1 = Wav2Vec2ConformerForCTC, 2 = WavLMForCTC */
  int32_t num_conv_layers;
  int32_t conv_dim[W2S_MAX_CONV_LAYERS];
  int32_t conv_kernel[W2S_MAX_CONV_LAYERS];
  int32_t conv_stride[W2S_MAX_CONV_LAYERS];
  int32_t conv_bias;            /* 0 / 1 */
  int32_t feat_extract_norm;    /* 0 = "group", 1 = "layer" */
  int32_t hidden_size;
  int32_t num_hidden_layers;
  int32_t num_attention_heads;
  int32_t intermediate_size;
  int32_t num_conv_pos_embeddings;
  int32_t num_conv_pos_embedding_groups;
  int32_t vocab_size;
  float   layer_norm_eps;
  int32_t do_stable_layer_norm; /* 0 / 1 */
  int32_t position_embeddings_type; /* conformer: 0 none, 1 "relative", 2 "rotary" */
  int32_t conv_depthwise_kernel_size;
  int32_t hidden_act;           /* 0 = "gelu" (erf form), 1 = "swish" */
  int32_t rotary_embedding_base;
  int32_t max_batch;            /* coalitions evaluated per internal batch tile (0 = choose) */
  int32_t flags;                /* W2S_FLAG_* */
  int32_t num_buckets;          /* WavLM: relative-position buckets (320) */
  int32_t max_bucket_distance;  /* WavLM: distance where the log buckets saturate (800) */
} w2s_config;

/* Replaces model construction + .to(device) (shap_calculation.py:218-219,258).
 * `names[i]` are HF state_dict keys ("wav2vec2.feature_extractor.conv_layers.0.conv.weight", ...,
 * "lm_head.bias"; prefix "wav2vec2_conformer." for kind 1, "wavlm." for kind 2; the weight-normed pos-conv must be
 * passed folded as
 * "<prefix>encoder.pos_conv_embed.conv.weight"), `ptrs[i]` fp32 DEVICE pointers in the HF layout with
 * `numels[i]` elements.  Weights are converted/re-laid-out into handle-owned storage; the caller may
 * free its copies after the call returns (the call synchronises the device once). */
int w2s_create(const w2s_config* cfg, const char* const* names, const float* const* ptrs,
               const int64_t* numels, int n_weights, int device, w2s_handle** out);

void w2s_destroy(w2s_handle* h);

/* NULL handle -> message of the last failed w2s_create on this thread. */
const char* w2s_last_error(const w2s_handle* h);

/* L -> T' (HF wav2vec2/modeling_wav2vec2.py:1005-1024). */
int64_t w2s_num_frames(const w2s_handle* h, int64_t num_samples);

/* Replaces the masker's captured state (feasability_tests/conformer_test.ipynb:138-141): the already
 * normalised clip x[L] (fp32, device; copied), the segment partition seg_bounds[M+1] (host, ascending,
 * seg_bounds[0]=0, seg_bounds[M]=L) and the baseline fill value (0.0 in the reference). */
int w2s_set_clip(w2s_handle* h, const float* x_dev, int64_t L, const int32_t* seg_bounds_host, int M,
                 float baseline, void* stream);

/* Background dataset of shap.KernelExplainer(f, data): B rows bg[B, L] (fp32, device, row stride `ld` elements, in the
 * same normalised input space as the clip; copied into the handle, so the caller may free them when this returns) with
 * weights w[B] (host, fp64: finite, >= 0, positive sum; normalised here in fp64 and stored as fp32).  1 <= B <=
 * W2S_MAX_BACKGROUND; L must equal the current clip's length (checked again by w2s_eval / w2s_mask when w2s_set_clip has
 * changed it since).  B = 0 clears the background and restores the baseline fill exactly.
 * While a background is set, coalition k is evaluated as B rows: row (k, b) takes sample i from the clip where segment
 * seg(i) is kept and from bg[b][i] where it is dropped; the baseline of w2s_set_clip is ignored.  w2s_eval then reports
 * out[k, :] = sum_b w_b * f(row (k, b)), accumulated in fp32 in the order b = 0 .. B-1 with one fmaf per term from 0 --
 * independent of the batch tile and of how the coalitions are spread over GPUs.  The call synchronises `stream`. */
#define W2S_MAX_BACKGROUND 256
int w2s_set_background(w2s_handle* h, const float* bg_dev, int64_t B, int64_t L, int64_t ld, const double* weights_host,
                       void* stream);

/* Time-frequency cells: F band components comp[F, L] of the clip (fp32, device, row stride `ld` elements; copied into the
 * handle, so the caller may free them when this returns), 1 <= F <= W2S_MAX_BANDS.  Component b is the clip filtered by the
 * band-b filter H_b of edges 0 = e_0 < e_1 < ... < e_F = sr / 2 (neighbouring edges >= 100 Hz apart): each interior edge e
 * has the crossover c_e(f) = 1 for f <= e - 50 Hz, 0 for f >= e + 50 Hz and cos^2(pi (f - e + 50) / 200) in between, and
 * H_b = c_{e_(b+1)} - c_{e_b} with c_{e_0} = 0, c_{e_F} = 1, so sum_b H_b = 1 at every frequency.  x_b = irfft(rfft(x) H_b,
 * n = L) in float64 (circular over the clip), cast to fp32 (preprocess.band_components computes them).
 * While bands are set, w2s_eval and w2s_mask take coalitions over M * F cells (M = the segments of w2s_set_clip, M * F <=
 * 2048): bit s * F + b of a row keeps cell (segment s, band b), and sample i of coalition row k is
 *   row_k[i] = sum_{b = 0 .. F-1} (keep(k, seg(i) * F + b) ? x_b[i] : 0),
 * fp32 adds in the order b = 0 .. F-1 from +0.0 (a dropped cell adds +0.0).  The clip itself and the baseline are not read:
 * the full coalition is f(sum_b x_b), within fp32 rounding of the clip, the empty one f(zeros).  Everything downstream of the
 * first convolution is unchanged.  w2s_eval_waveforms and the gradient entry points ignore the bands.  Refused before any
 * launch: F out of range, a null buffer, a background set (bands and a background do not combine), L other than the clip's
 * (checked again by w2s_eval / w2s_mask when w2s_set_clip has changed it since) and M * F > 2048.  F = 0 clears the bands
 * and restores the time-only coalitions exactly.  The call synchronises `stream`. */
#define W2S_MAX_BANDS 16
int w2s_set_bands(w2s_handle* h, const float* comp_dev, int64_t F, int64_t L, int64_t ld, void* stream);

/* Replaces timestep_to_explain / token_id_to_explain (w2v2conformer.py:93-110) and the character-frame
 * list of visualization.py:319-327: D (frame, token) pairs (host arrays, copied before the call returns; ignored
 * for MAX/MEAN/LOGITS).  The upload is ordered on `stream` behind evaluations already queued there. */
int w2s_set_targets(w2s_handle* h, const int32_t* frame_idx_host, const int32_t* token_idx_host, int D,
                    int mode, void* stream);

/* Transcript-level output W2S_OUT_CTC: D >= 1 label sequences y_d = labels[offsets[d] .. offsets[d + 1]) (host arrays,
 * offsets[0] = 0, non-decreasing, 0 <= U_d <= W2S_MAX_TRANSCRIPT; every label in [0, V) and != blank; blank in [0, V), the
 * model's pad_token_id).  Row r then reports out[r, d] = log p_CTC(y_d | logits of row r over all T' frames) in natural
 * log: the log of the sum over all alignments of y_d to the T' frames, i.e. -WavXForCTC(x, labels=y_d).loss with
 * ctc_loss_reduction = "sum".  The empty transcript gives sum_t log_softmax(z_t)[blank].  Transcript d needs U_d + (number
 * of adjacent equal labels) frames: w2s_eval / w2s_eval_waveforms fail before any launch when the clip of the call has
 * fewer, naming the transcript, so no accepted transcript yields -inf or NaN.  Each value is one fixed sequence of fp32
 * operations on that row's logits (log-domain forward recursion, one warp per (row, transcript)): bit-identical for any
 * batch tile, position in the tile, number of GPUs and across calls.  With a background the usual weighted mean applies.
 * Everything but the clip length is validated before the device is touched; the upload is ordered on `stream` as in
 * w2s_set_targets.  The transcripts stay stored when w2s_set_targets later selects another mode (w2s_grad_transcripts
 * uses them). */
#define W2S_MAX_TRANSCRIPT 512
int w2s_set_transcripts(w2s_handle* h, const int32_t* labels_host, const int32_t* offsets_host, int D, int blank,
                        void* stream);

/* Number of fp32 values one evaluated row produces under the current mode for clips of L samples. */
int64_t w2s_out_width(const w2s_handle* h, int64_t num_samples);

/* The fused masker + model callable: coalition bit matrix z_bits[K, ceil(M/32)] (device; bit m of row k
 * set = segment m KEPT, clear = replaced by the baseline) -> out[K, width] fp32 (device).  With a background
 * (w2s_set_background) K * B rows are evaluated and out[K, width] holds their weighted means.  With bands
 * (w2s_set_bands) z_bits is [K, ceil(M * F / 32)], one bit per time-frequency cell. */
int w2s_eval(w2s_handle* h, const uint32_t* z_bits_dev, int64_t K, float* out_dev, void* stream);

/* Replaces ModelWrapper.forward (shap_calculation.py:31-50), predict_function
 * (w2v2conformer.py:116-131) and lime_predict_fn (lime_shap_wav2vec2_comparison.py:60-71) for explicit
 * waveform rows x[n, L] (fp32, device, row stride `ld` elements) -> out[n, width] fp32 (device). */
int w2s_eval_waveforms(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld, float* out_dev,
                       void* stream);

/* Expected-gradients path -- the reference's production explainer differentiates ModelWrapper's output
 * (shap.GradientExplainer(wrapped_model, ...).shap_values, shap_calculation.py:133,162; per output index
 * `outputs = self.model(*X); outputs[:, idx]` then autograd, conformer_test.ipynb:95).  For explicit waveform rows
 * x[n, L] (fp32, device, row stride `ld`) and one output frame per row (host array): out[r] = max_v logits[r,
 * frames[r], v] (shap_calculation.py:50) and grad[r, :] = d out[r] / d x[r, :] (fp32 [n, L], device).  Input
 * gradients only -- no weight gradients.  First slice: Wav2Vec2ForCTC with the group-norm front end and a post-LN
 * encoder (wav2vec2-base / -large); other configurations return an error.  WavLMForCTC is refused: the backward of its
 * gated relative-position bias is not built. */
int w2s_grad_waveforms(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld,
                       const int32_t* frames_host, float* grad_dev, float* out_dev, void* stream);
/* The same backward pass seeded with an upstream gradient over ALL output frames -- the vector-Jacobian product autograd
 * asks of ModelWrapper.forward (B1 in SURVEY.md 8b: "autograd graph required"): gout[n, T'] (fp32, device) ->
 * grad[r, :] = sum_t gout[r, t] d out[r, t] / d x[r, :], out[n, T'] = the max logits (may be NULL).  With it the
 * reference's shap.GradientExplainer(wrapped_model, ...) runs unmodified on callbacks.ModelWrapper. */
int w2s_vjp_waveforms(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld, const float* gout_dev,
                      float* grad_dev, float* out_dev, void* stream);
/* The same backward pass for the transcript-level output: out[r] = log p_CTC(y_{which[r]} | x_r) (see
 * w2s_set_transcripts) and grad[r, :] = d out[r] / d x[r, :].  which[n] (host) indexes the transcripts last set.  The seed
 * d log p / d logits[t, v] = gamma_t(v) - softmax(logits_t)_v, with gamma the CTC state occupation from the log-domain
 * alpha / beta recursions, reaches every frame.  Refused before any launch: no transcripts set, an index out of range,
 * a transcript infeasible for the clip, w2s_grad_rules on (DeepLIFT on transcripts is not built), and every model the
 * gradient path refuses (WavLMForCTC included).  out may be NULL. */
int w2s_grad_transcripts(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld, const int32_t* which_host,
                         float* grad_dev, float* out_dev, void* stream);
/* Test hooks of the gradient path.  `on` bit 0: keep snapshots of the gradient after every encoder layer / conv layer
 * ("layer<l>", "h0", "conv<l>", "convu<l>", forward activations "f.*"); bit 1: run attention backward on the CUDA-core
 * cross-check kernels, bit 2: as batched tensor-core contractions + row kernels, instead of the fused tcgen05 kernel.  w2s_grad_peek copies a snapshot out (returns bytes copied, 0 = unknown name, < 0 = buffer
 * too small by that many bytes). */
int w2s_grad_debug(w2s_handle* h, int on);
/* DeepLIFT handler rules of feasability_tests/custom_shap_handlers.py:35-80 for the backward pass of w2s_grad_waveforms.
 * With rules != 0 every call carries PAIRED rows: rows [0, n/2) are explained inputs, row n/2 + r is the reference
 * (background) row of row r; n even and at most 32.  Reference rows receive no output seed: their gradient rows are zero.
 *   bit 0: SiLU activations use the rescale multiplier (act(x) - act(ref)) / (x - ref) (shap's nonlinear_1d; the ordinary
 *          derivative where |x - ref| < 1e-6); LayerNorm / GroupNorm are linear_1d, i.e. the ordinary gradient, like every
 *          module shap has no handler for (GELUActivation, attention);
 *   bit 1: the reference's GLU handler as written: GLU inputs that differ from the reference by >= 1e-6 receive
 *          grad_output * 5e-6 (a placeholder its author left in; off by default).
 * rules = 0 restores the plain gradient. */
int w2s_grad_rules(w2s_handle* h, int rules);
int64_t w2s_grad_peek(w2s_handle* h, const char* name, void* dst_dev, int64_t max_bytes, void* stream);

/* Standalone masker (conformer_test.ipynb:138-141 semantics with keep-bits): materialise
 * out[K, L] = keep ? x : baseline for the clip set by w2s_set_clip; with a background, out[K * B, L] with row k * B + b =
 * keep ? x : bg[b]; with bands, out[K, L] = the cell sums of w2s_set_bands -- the rows w2s_eval evaluates, in its order. */
int w2s_mask(w2s_handle* h, const uint32_t* z_bits_dev, int64_t K, float* out_dev, void* stream);

/* KernelSHAP constrained weighted least squares (shap KernelExplainer.solve with l1_reg=False; SURVEY.md
 * Appendix A step 6): z_bits[K, ceil(M/32)], kernel weights w[K] (fp64), y[K, D] fp32, fx[D], fnull[D]
 * (fp64) -> phi[M, D] fp64, all device pointers.  `status_dev` (int32, device, required) receives 0 when the
 * normal matrix was factored by Cholesky; 2 when the design is rank deficient (fewer distinct coalitions than
 * features, or a feature that never varies) and the minimum-norm least-squares solution was computed instead
 * -- what shap's `solve` returns through its numpy.linalg.lstsq fallback -- by conjugate gradients on the device;
 * 1 if that iteration did not converge (phi is then not to be used). */
int w2s_wls(w2s_handle* h, const uint32_t* z_bits_dev, const double* w_dev, const float* y_dev, int64_t K,
            int M, int D, const double* fx_dev, const double* fnull_dev, double* phi_dev, int32_t* status_dev,
            void* stream);

/* The random half of shap.KernelExplainer's coalition sampler (third-party, never called by the reference: SURVEY.md
 * Appendix A step 4), on the HOST: for every entry of `ind_set` (the subset sizes drawn by np.random.choice) one
 * legacy np.random.permutation(M) on the MT19937 state `mt_key[624]` / `*mt_pos` taken from np.random.get_state()
 * (updated in place, to be handed back with np.random.set_state), de-duplicated rows appended to the bit-packed
 * matrix z_words[cap_rows, ceil(M/32)] from row `added` on, with their hit counts in weights[] and the paired
 * complement rows where shap adds them.  Returns the new row count, or -1 on a bad argument / overflow.
 * No device is touched. */
int64_t w2s_sample_rows(int M, int n_full, int n_paired, const int64_t* ind_set, int64_t n_ind,
                        int64_t samples_left, int64_t added, uint32_t* mt_key, int32_t* mt_pos,
                        uint32_t* z_words, double* weights, int64_t cap_rows, int64_t* ind_used);

/* WavLM's relative-position buckets (HF wavlm/modeling_wavlm.py:253-271, _relative_positions_bucket) for a clip of T
 * frames: out[r] = bucket(r - (T - 1)), r = 0 .. 2T-2, computed on the HOST in double precision.  Returns 0, or 1 on a bad
 * argument (T < 1, num_buckets < 4, max_distance <= num_buckets / 4).  No device is touched. */
int w2s_relative_buckets(int T, int num_buckets, int max_distance, int32_t* out);

/* Test / profiling hooks for the individual kernels (used by tests/ and bench.py only). */
/* out[M, N] = act(a[M, K] w[N, K]^T + bias) * alpha + residual (residual == out with fp32 data: in-place
 * accumulation, which the CTA-pair kernel performs with TMA reduce-add). */
int w2s_debug_gemm(int use_tcgen05, const void* a_bf16, const void* w_bf16, const float* bias,
                   const void* residual, int res_fp32, float alpha, void* out, int M, int N, int K, int act,
                   int out_fp32, void* stream);
/* Self-attention of one layer on caller-owned device buffers, with the operand layout of the model paths: qkv[B*T, 3H] =
 * q | k | v, or with pos_proj [2T-1, H] (row r <-> relative position T-1-r) the relative-position conformer's
 * qkv[B*T, 4H] = q+u | q+v | k | v; H = 64 * heads.  use_tcgen05 = 1: the tensor-core kernel (attention_fa without
 * pos_proj, which also writes lse[B, heads, T], the log2-domain log-sum-exp of the scaled scores, when lse != NULL;
 * attention_rel with it); 0: the CUDA-core validation kernel (T <= 1024, lse must be NULL).  ctx[B*T, H] bf16.
 * Errors via w2s_last_error(NULL). */
int w2s_debug_attention(int use_tcgen05, const void* qkv, const void* pos_proj, int B, int T, int heads, float scale,
                        void* ctx, float* lse, void* stream);
/* w2s_debug_attention (no pos_proj) with WavLM's gated relative-position bias: score[b, h, i, j] += gate[b, h, i] *
 * rel_bias[h, T - 1 + j - i], rel_bias [heads, 2T-1] and gate [B, heads, T] fp32 in natural units, device.  The bias
 * variant writes no log-sum-exp: lse != NULL is an error.  Errors via w2s_last_error(NULL). */
int w2s_debug_attention_bias(int use_tcgen05, const void* qkv, const float* rel_bias, const float* gate, int B, int T,
                             int heads, float scale, void* ctx, float* lse, void* stream);
/* Its backward (no relative positions): d ctx[B*T, H] -> dqkv[B*T, 3H] bf16.  use_tcgen05 = 1: the gradient path's fused
 * kernel with its delta pre-pass and dQ cast, fed the forward's ctx and lse (from w2s_debug_attention); 0: the CUDA-core
 * cross-check kernels (T <= 1024; ctx / lse unused).  The workspace is allocated and freed inside: the call synchronises
 * the stream. */
int w2s_debug_attention_bwd(int use_tcgen05, const void* qkv, const void* ctx, const void* dctx, const float* lse, int B,
                            int T, int heads, float scale, void* dqkv, void* stream);
/* The CTC code of W2S_OUT_CTC on caller logits [n, T, ldl] (fp32, device; V <= ldl used): out[n, D] (device) =
 * log p_CTC(y_d | logits[r]) through the head reduction kernel.  With dlogits [n, T, V] (device, may be NULL), also the
 * gradient seed of w2s_grad_transcripts: dlogits[r] = d out[r, which[r]] / d logits[r].  labels / offsets [D + 1] / which [n]
 * are host arrays, validated as in w2s_set_transcripts plus feasibility for T.  The call synchronises the stream.  Errors via
 * w2s_last_error(NULL). */
int w2s_debug_ctc(const float* logits, int n, int T, int V, int ldl, const int32_t* labels_host, const int32_t* offsets_host,
                  int D, int blank, const int32_t* which_host, float* out_dev, float* dlogits_dev, void* stream);
/* Per-launch CUDA-event profile on the launching stream (bench.py roofline leg): enable, run evaluations,
 * then read per launch class (newline-separated names) total milliseconds, algorithmic FLOPs / bytes and
 * launch counts.  Returns the number of classes, or -1 if `names_cap` is too small. */
int w2s_profile_enable(w2s_handle* h, int on);
int64_t w2s_profile_read(w2s_handle* h, char* names, int64_t names_cap, double* ms, double* flops, double* bytes,
                         int64_t* counts, int64_t max_entries);
int w2s_kernel_count(const w2s_handle* h, int64_t* launches_per_batch, int64_t* batch_tile);
/* kernel launches issued by w2s_eval / w2s_eval_waveforms on this handle since w2s_create (counted at launch,
 * graph-replayed kernels included) */
int64_t w2s_launch_count(const w2s_handle* h);
/* algorithmic FLOPs (2*MAC) of one coalition forward for clips of L samples */
double w2s_flops_per_forward(const w2s_handle* h, int64_t num_samples);

#ifdef __cplusplus
}
#endif
#endif /* W2S_H_ */
