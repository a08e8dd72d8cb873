// C ABI (include/w2s.h): handle, weight re-layout, workspace, per-batch launch plans and the
// orchestration of one masked-coalition forward.  Everything below the boundary is CUDA for sm_100a;
// there is no CPU path.
#include "../../include/w2s.h"
#include "gemm.cuh"
#include "kernels.cuh"
#include "skip.cuh"
#include "ctc.cuh"
#include "errors.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

using namespace w2s;
typedef __nv_bfloat16 bf16;

namespace {

thread_local std::string g_create_error;

struct LayerW {
  // wav2vec2 encoder layer (post-LN / stable-LN)
  bf16 *wqkv = nullptr, *wo = nullptr, *w1 = nullptr, *w2 = nullptr;
  float *bqkv = nullptr, *bo = nullptr, *b1 = nullptr, *b2 = nullptr;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  // conformer extras
  bf16 *f2w1 = nullptr, *f2w2 = nullptr, *wpos = nullptr, *pw1 = nullptr, *pw2 = nullptr;
  float *f2b1 = nullptr, *f2b2 = nullptr;
  float *lnf1_g = nullptr, *lnf1_b = nullptr, *lnf2_g = nullptr, *lnf2_b = nullptr;
  float *lnc_g = nullptr, *lnc_b = nullptr, *lnfin_g = nullptr, *lnfin_b = nullptr;
  float *dw_w = nullptr, *dw_scale = nullptr, *dw_shift = nullptr;  // depthwise taps [H][k], folded BatchNorm
  bf16* pos_proj = nullptr;  // [2T-1, H], built per clip length
  // WavLM: gru_rel_pos_linear [8, 64] / [8] and gru_rel_pos_const [heads] of this layer
  float *gate_w = nullptr, *gate_b = nullptr, *gate_c = nullptr;
};

struct Step {
  std::string name;
  std::function<std::string(cudaStream_t)> run;
  double flops = 0.0;  // algorithmic FLOPs (2*MAC) of this launch, 0 for non-contraction kernels
  double bytes = 0.0;  // algorithmic HBM bytes of this launch (HBM-bound kernels)
  // launches over a device list (frontend skip): the profile reads the count back and charges flops / bytes per entry
  const int* work = nullptr;
};

struct ProfRec {
  std::string name;
  cudaEvent_t e0, e1;
  double flops, bytes;
};

struct Plan {
  int n = 0;
  std::vector<Step> steps;
  std::vector<GemmLaunch*> gemms;
  std::vector<AttnRelPlan*> attn_rel;
  std::vector<PosConvPlan*> posconv;
  std::vector<AttnFaPlan*> attn_fa;
  // the whole tile forward as one CUDA graph (captured on first use; per-call arguments travel through DynArgs)
  cudaGraphExec_t exec = nullptr;
  bool graph_failed = false;
  ~Plan() {
    if (exec) cudaGraphExecDestroy(exec);
    for (auto* f : attn_fa) attention_fa_free(f);
    for (auto* pc : posconv) posconv_free(pc);
    for (auto* g : gemms) delete g;
    for (auto* a : attn_rel) attention_rel_free(a);
  }
};

__global__ void set_dyn_kernel(DynArgs* dst, const DynArgs v) { *dst = v; }

// expected-gradients path: transposed dense weights of one encoder layer (dX = dY W runs as a contraction with W^T)
struct GradW {
  bf16 *wqkvT = nullptr, *woT = nullptr, *w1T = nullptr, *w2T = nullptr;
  // conformer: second macaron feed-forward, pointwise convs, rotary q|k and v projections, reversed depthwise taps
  bf16 *f2w1T = nullptr, *f2w2T = nullptr, *pw1T = nullptr, *pw2T = nullptr, *wqkT = nullptr, *wvT = nullptr;
  float* dw_flip = nullptr;
  // relative positions, per clip length: linear_pos(pe) [2T'-1, H] and its per-head transpose [heads][64][Rp]
  bf16 *pos_proj = nullptr, *pos_projT = nullptr;
};
struct GradPlan;

}  // namespace

struct w2s_handle {
  w2s_config cfg{};
  int device = 0;
  int num_sms = 148;
  bool auto_batch = false;   // max_batch == 0 at create: pick the batch tile per clip length
  std::string err;
  std::vector<void*> allocs;      // weights: live until destroy
  std::vector<void*> ws_allocs;   // workspace: re-made when the clip length changes

  // weights
  float *conv0_w = nullptr, *conv0_b = nullptr, *norm0_g = nullptr, *norm0_b = nullptr;
  float *ln0_wbar = nullptr, *ln0_gram = nullptr, *ln0_wb = nullptr;
  bf16* ln0_wb48 = nullptr;
  float ln0_bmean = 0.f, ln0_b2mean = 0.f;
  bf16* conv_w[W2S_MAX_CONV_LAYERS] = {};
  float* conv_b[W2S_MAX_CONV_LAYERS] = {};
  float* conv_ln_g[W2S_MAX_CONV_LAYERS] = {};
  float* conv_ln_b[W2S_MAX_CONV_LAYERS] = {};
  float *fp_ln_g = nullptr, *fp_ln_b = nullptr, *fp_b = nullptr;
  bf16* fp_w = nullptr;
  bf16* pos_w = nullptr;
  float* pos_b = nullptr;
  float *enc_ln_g = nullptr, *enc_ln_b = nullptr;
  float* rel_embed = nullptr;   // WavLM: layer 0's rel_attn_embed [num_buckets, heads], shared by every layer
  std::vector<LayerW> layers;
  bf16* head_w = nullptr;
  float* head_b = nullptr;

  // clip state
  long long L = 0;
  int M = 0, zwords = 0;
  float baseline = 0.f;
  float* clip = nullptr;
  uint16_t* seg_id = nullptr;
  long long clip_cap = 0, seg_id_cap = 0;   // elements

  // background (w2s_set_background): bg_B rows of bg_L samples replace the baseline; bg_B == 0: none
  int bg_B = 0;
  long long bg_L = 0;
  float* bg = nullptr;              // [bg_B, bg_L]
  long long bg_cap = 0;             // floats
  float* bg_w = nullptr;            // [W2S_MAX_BACKGROUND] normalised weights, fp32
  std::vector<float> bg_w_host;     // staging of the upload
  float* bg_rows = nullptr;         // [K * bg_B, width] per-row outputs of the last w2s_eval, reduced by bg_mean_kernel
  long long bg_rows_cap = 0;        // floats; only grows

  // time-frequency cells (w2s_set_bands): bands_F components of bands_L samples; bands_F == 0: time-only coalitions
  int bands_F = 0;
  long long bands_L = 0;
  float* bands = nullptr;           // [bands_F, bands_L]
  long long bands_cap = 0;          // floats

  // targets
  int mode = W2S_OUT_MAX, D = 0, max_frame = 0;
  int* targets = nullptr;              // [2 D]: the D target frames, then the D tokens
  long long targets_cap = 0;           // ints
  std::vector<int32_t> targets_host;   // staging of the last w2s_set_targets arrays (source of the async upload)

  // transcripts (w2s_set_transcripts): kept across w2s_set_targets, so the gradient entry can use them in any mode
  int ctc_D = 0, ctc_blank = 0, ctc_smax = 1;   // count, blank id, largest 2U + 1
  int *ctc_labels = nullptr, *ctc_offsets = nullptr;
  long long ctc_labels_cap = 0, ctc_offsets_cap = 0;
  std::vector<int32_t> ctc_host;        // staging of the upload: offsets [D + 1], then the labels
  std::vector<int> ctc_need;            // frames each transcript needs
  float *ctc_alpha = nullptr, *ctc_lse = nullptr, *ctc_dz = nullptr;   // gradient-seed scratch, grown on demand
  long long ctc_alpha_cap = 0, ctc_lse_cap = 0, ctc_dz_cap = 0;

  // references (w2s_set_references): the tables of errors.cuh, apart from the transcripts
  int err_D = 0, err_blank = 0, err_unit = 0, err_delim = 0;
  int* err_tab = nullptr;
  long long err_tab_cap = 0;
  std::vector<int32_t> err_host;        // staging of the upload

  // workspace (sized for max_batch rows of the current clip length)
  long long ws_L = -1;
  int T = 0, Tp = 0;
  std::vector<int> Tl;  // conv output lengths
  float *gn_a = nullptr, *gn_b = nullptr;
  bf16* gn_wb = nullptr;
  bf16 *bufA = nullptr, *bufB = nullptr;
  bf16 *fpn = nullptr, *h0 = nullptr, *hp = nullptr, *hb = nullptr, *h1 = nullptr, *qkv = nullptr, *ctx = nullptr,
       *ffn = nullptr;
  float* pre = nullptr;
  float* logits = nullptr;
  bf16* hrot = nullptr;
  float* rel_bias = nullptr;    // WavLM: bias table of the current clip length (AttnParams::rel_bias)
  float* gate = nullptr;        // WavLM: [max_batch, heads, T'] gate of the current layer
  double* wls_work = nullptr;
  long long wls_cap = 0;
  std::map<std::pair<int, int>, std::unique_ptr<Plan>> plans;   // keyed by (tile rows, fill kind | PLAN_SKIP): a graph keeps its conv0

  // constant-frame skip of the feature encoder (frontend_skip.cu), sized with the workspace: block table of the clip
  // (w2s_frontend_blocks, uploaded by w2s_set_clip) and the per-tile block lists of conv1 .. conv_{nl}
  int4* skip_tab = nullptr;
  int skip_rows = 0;
  bool skip_tab_ok = false;                 // skip_tab holds the table of the current clip (w2s_set_clip bounds, L == ws_L)
  std::vector<int32_t> seg_bounds;          // [M + 1] of the current clip: the table is rebuilt with the workspace
  int* skip_live[SKIP_MAX_LAYERS] = {};
  int* skip_fill[SKIP_MAX_LAYERS] = {};
  int* skip_rep = nullptr;

  // optional per-launch CUDA-event profile (bench.py roofline leg)
  bool profiling = false;
  std::vector<ProfRec> prof;

  // expected-gradients path (grad_plan.cuh): backward weights, plans per tile size, per-call pointers
  bool grad_ready = false;
  std::vector<GradW> gradw;
  bf16* conv_wT[W2S_MAX_CONV_LAYERS] = {};
  bf16* fp_wT = nullptr;
  bf16* pos_w_bwd = nullptr;          // flipped / transposed positional-conv filters (built at create)
  float *grad_ones = nullptr, *grad_zeros = nullptr;   // [H]: identity scale / shift of the depthwise backward
  std::vector<void*> grad_pos_allocs;                  // relative-position tables of the current grad_L
  std::map<int, std::shared_ptr<GradPlan>> grad_plans;
  long long grad_L = -1;
  int grad_tile = 32;
  bool grad_debug = false, grad_debug_built = false;
  bool grad_attn_simt = false;        // cross-check: attention backward on the CUDA-core kernels (w2s_grad_debug bit 1)
  bool grad_attn_unfused = false;     // cross-check: attention backward as batched contractions + row kernels (bit 2)
  int grad_rules = 0, grad_rules_built = 0;   // w2s_grad_rules: DeepLIFT handler rules on paired [explained | reference] rows
  // target frames of a tile travel through a ring of pinned slots (a pageable source would make every call wait for the
  // stream); a slot is reused only after the copy that read it has completed
  static constexpr int kFrameSlots = 8;
  int32_t* grad_frames_pinned = nullptr;          // [kFrameSlots][grad_tile]
  cudaEvent_t grad_frames_done[kFrameSlots] = {};
  unsigned grad_frames_next = 0;
  float *grad_out = nullptr, *grad_out_val = nullptr;
  const float* grad_gout = nullptr;
  bool grad_ctc = false;              // w2s_grad_transcripts: the head_bwd step seeds from the CTC log-likelihood

  // per-call arguments of the plan's kernels (kernels.cuh: DynArgs), rewritten before every tile
  DynArgs* dyn_dev = nullptr;
  int head_ldl = 0;             // logits row stride: vocab rounded up to a multiple of 32
  cudaStream_t cap_stream = nullptr;   // graphs are captured here (the caller's stream may be the legacy stream)
  bool use_graphs = true;
  long long launches = 0;       // kernel launches issued by w2s_eval / w2s_eval_waveforms since create

  ~w2s_handle() {
    for (auto& r : prof) {
      cudaEventDestroy(r.e0);
      cudaEventDestroy(r.e1);
    }
    plans.clear();
    grad_plans.clear();
    for (void* p : grad_pos_allocs) cudaFree(p);
    if (grad_frames_pinned) cudaFreeHost(grad_frames_pinned);
    for (auto& e : grad_frames_done)
      if (e) cudaEventDestroy(e);
    if (cap_stream) cudaStreamDestroy(cap_stream);
    if (dyn_dev) cudaFree(dyn_dev);
    if (clip) cudaFree(clip);
    if (seg_id) cudaFree(seg_id);
    if (bg) cudaFree(bg);
    if (bg_w) cudaFree(bg_w);
    if (bg_rows) cudaFree(bg_rows);
    if (bands) cudaFree(bands);
    if (targets) cudaFree(targets);
    for (void* p : {(void*)ctc_labels, (void*)ctc_offsets, (void*)ctc_alpha, (void*)ctc_lse, (void*)ctc_dz, (void*)err_tab})
      if (p) cudaFree(p);
    if (wls_work) cudaFree(wls_work);
    for (void* p : ws_allocs) cudaFree(p);
    for (void* p : allocs) cudaFree(p);
  }
};

namespace {

template <typename T>
std::string dalloc(std::vector<void*>& pool, T** out, size_t count, bool zero = false) {
  void* p = nullptr;
  const size_t bytes = count * sizeof(T) + 65536;  // slack: strided-conv views may touch a few rows past the end
  W2S_CUDA_OK(cudaMalloc(&p, bytes));
  if (zero) W2S_CUDA_OK(cudaMemset(p, 0, bytes));
  pool.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return "";
}

// Grow-on-demand device buffer: afterwards *p holds at least `need` elements, max(need, min_cap) when it had to grow.
// Work queued on s may still read the old buffer, so s is synchronised before it is freed; a failed allocation leaves
// *p == nullptr and *cap == 0, not a dangling pointer.  Errors: "stream error", "out of device memory".
template <typename T>
std::string grow(T** p, long long* cap, long long need, long long min_cap, cudaStream_t s) {
  if (*cap >= need) return "";
  if (cudaStreamSynchronize(s) != cudaSuccess) return "stream error";
  if (*p) cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  const long long n = std::max(need, min_cap);
  if (cudaMalloc((void**)p, sizeof(T) * n) != cudaSuccess) {
    *p = nullptr;
    return "out of device memory";
  }
  *cap = n;
  return "";
}

struct WeightTable {
  std::map<std::string, std::pair<const float*, int64_t>> t;
  std::string prefix;
  std::string get(const std::string& name, int64_t expect, const float** out) const {
    auto it = t.find(name);
    if (it == t.end()) return "missing weight '" + name + "'";
    if (expect >= 0 && it->second.second != expect)
      return "weight '" + name + "' has " + std::to_string(it->second.second) + " elements, expected " +
             std::to_string(expect);
    *out = it->second.first;
    return "";
  }
};

std::string copy_f32(w2s_handle* h, const WeightTable& wt, const std::string& name, int64_t n, float** dst) {
  const float* src = nullptr;
  W2S_TRY(wt.get(name, n, &src));
  W2S_TRY(dalloc(h->allocs, dst, (size_t)n));
  W2S_CUDA_OK(cudaMemcpy(*dst, src, sizeof(float) * n, cudaMemcpyDeviceToDevice));
  return "";
}
std::string copy_bf16(w2s_handle* h, const WeightTable& wt, const std::string& name, int64_t n, bf16* dst) {
  const float* src = nullptr;
  W2S_TRY(wt.get(name, n, &src));
  return launch_cast_bf16(src, dst, n, 0);
}

std::string load_weights(w2s_handle* h, const WeightTable& wt) {
  const w2s_config& c = h->cfg;
  const std::string P = wt.prefix;
  const int H = c.hidden_size, I = c.intermediate_size, V = c.vocab_size;
  const bool layer = c.feat_extract_norm == 1;
  // ---- feature encoder ----
  for (int l = 0; l < c.num_conv_layers; ++l) {
    const std::string cp = P + "feature_extractor.conv_layers." + std::to_string(l) + ".";
    const int Cin = l == 0 ? 1 : c.conv_dim[l - 1], Cout = c.conv_dim[l], kw = c.conv_kernel[l];
    if (l == 0) {
      W2S_TRY(copy_f32(h, wt, cp + "conv.weight", (int64_t)Cout * kw, &h->conv0_w));
      if (c.conv_bias) W2S_TRY(copy_f32(h, wt, cp + "conv.bias", Cout, &h->conv0_b));
      W2S_TRY(copy_f32(h, wt, cp + "layer_norm.weight", Cout, &h->norm0_g));
      W2S_TRY(copy_f32(h, wt, cp + "layer_norm.bias", Cout, &h->norm0_b));
      if (layer) {
        W2S_TRY(dalloc(h->allocs, &h->ln0_wbar, 16));
        W2S_TRY(dalloc(h->allocs, &h->ln0_gram, 256));
        W2S_TRY(dalloc(h->allocs, &h->ln0_wb, 16));
        float* sc = nullptr;
        W2S_TRY(dalloc(h->allocs, &sc, 2));
        W2S_TRY(launch_conv0_ln_prep(h->conv0_w, h->conv0_b, Cout, kw, h->ln0_wbar, h->ln0_gram, h->ln0_wb, sc, 0));
        float hs[2];
        W2S_CUDA_OK(cudaMemcpy(hs, sc, sizeof(hs), cudaMemcpyDeviceToHost));
        h->ln0_bmean = hs[0];
        h->ln0_b2mean = hs[1];
        if (kw == 10 && Cout % 64 == 0 && Cout <= 512) {
          W2S_TRY(dalloc(h->allocs, &h->ln0_wb48, (size_t)Cout * 48));
          W2S_TRY(launch_conv0_ln_b(h->conv0_w, h->conv0_b, h->norm0_g, h->norm0_b, Cout, kw, h->ln0_wb48, 0));
        }
      }
    } else {
      const float* src = nullptr;
      W2S_TRY(wt.get(cp + "conv.weight", (int64_t)Cout * Cin * kw, &src));
      W2S_TRY(dalloc(h->allocs, &h->conv_w[l], (size_t)Cout * Cin * kw));
      W2S_TRY(launch_repack_conv(src, h->conv_w[l], Cout, Cin, kw, 0));
      if (c.conv_bias) W2S_TRY(copy_f32(h, wt, cp + "conv.bias", Cout, &h->conv_b[l]));
      if (layer) {
        W2S_TRY(copy_f32(h, wt, cp + "layer_norm.weight", Cout, &h->conv_ln_g[l]));
        W2S_TRY(copy_f32(h, wt, cp + "layer_norm.bias", Cout, &h->conv_ln_b[l]));
      }
    }
  }
  // ---- feature projection ----
  const int Cl = c.conv_dim[c.num_conv_layers - 1];
  W2S_TRY(copy_f32(h, wt, P + "feature_projection.layer_norm.weight", Cl, &h->fp_ln_g));
  W2S_TRY(copy_f32(h, wt, P + "feature_projection.layer_norm.bias", Cl, &h->fp_ln_b));
  W2S_TRY(dalloc(h->allocs, &h->fp_w, (size_t)H * Cl));
  W2S_TRY(copy_bf16(h, wt, P + "feature_projection.projection.weight", (int64_t)H * Cl, h->fp_w));
  W2S_TRY(copy_f32(h, wt, P + "feature_projection.projection.bias", H, &h->fp_b));
  // ---- encoder ----
  W2S_TRY(copy_f32(h, wt, P + "encoder.layer_norm.weight", H, &h->enc_ln_g));
  W2S_TRY(copy_f32(h, wt, P + "encoder.layer_norm.bias", H, &h->enc_ln_b));
  h->layers.resize(c.num_hidden_layers);
  if (c.kind != 1) {   // wav2vec2 and WavLM
    const int G = c.num_conv_pos_embedding_groups, kp = c.num_conv_pos_embeddings, cpg = H / G;
    const float* src = nullptr;
    W2S_TRY(wt.get(P + "encoder.pos_conv_embed.conv.weight", (int64_t)H * cpg * kp, &src));
    W2S_TRY(dalloc(h->allocs, &h->pos_w, (size_t)H * kp * 64));
    W2S_TRY(launch_repack_posconv(src, h->pos_w, H, G, kp, 0));
    W2S_TRY(dalloc(h->allocs, &h->pos_w_bwd, (size_t)H * kp * 64));
    W2S_TRY(launch_repack_posconv_bwd(src, h->pos_w_bwd, H, G, kp, 0));
    W2S_TRY(copy_f32(h, wt, P + "encoder.pos_conv_embed.conv.bias", H, &h->pos_b));
    for (int l = 0; l < c.num_hidden_layers; ++l) {
      LayerW& w = h->layers[l];
      const std::string lp = P + "encoder.layers." + std::to_string(l) + ".";
      W2S_TRY(dalloc(h->allocs, &w.wqkv, (size_t)3 * H * H));
      W2S_TRY(copy_bf16(h, wt, lp + "attention.q_proj.weight", (int64_t)H * H, w.wqkv));
      W2S_TRY(copy_bf16(h, wt, lp + "attention.k_proj.weight", (int64_t)H * H, w.wqkv + (size_t)H * H));
      W2S_TRY(copy_bf16(h, wt, lp + "attention.v_proj.weight", (int64_t)H * H, w.wqkv + (size_t)2 * H * H));
      W2S_TRY(dalloc(h->allocs, &w.bqkv, (size_t)3 * H));
      const float* b = nullptr;
      const char* nm[3] = {"attention.q_proj.bias", "attention.k_proj.bias", "attention.v_proj.bias"};
      for (int j = 0; j < 3; ++j) {
        W2S_TRY(wt.get(lp + nm[j], H, &b));
        W2S_CUDA_OK(cudaMemcpy(w.bqkv + (size_t)j * H, b, sizeof(float) * H, cudaMemcpyDeviceToDevice));
      }
      W2S_TRY(dalloc(h->allocs, &w.wo, (size_t)H * H));
      W2S_TRY(copy_bf16(h, wt, lp + "attention.out_proj.weight", (int64_t)H * H, w.wo));
      W2S_TRY(copy_f32(h, wt, lp + "attention.out_proj.bias", H, &w.bo));
      W2S_TRY(copy_f32(h, wt, lp + "layer_norm.weight", H, &w.ln1_g));
      W2S_TRY(copy_f32(h, wt, lp + "layer_norm.bias", H, &w.ln1_b));
      W2S_TRY(dalloc(h->allocs, &w.w1, (size_t)I * H));
      W2S_TRY(copy_bf16(h, wt, lp + "feed_forward.intermediate_dense.weight", (int64_t)I * H, w.w1));
      W2S_TRY(copy_f32(h, wt, lp + "feed_forward.intermediate_dense.bias", I, &w.b1));
      W2S_TRY(dalloc(h->allocs, &w.w2, (size_t)H * I));
      W2S_TRY(copy_bf16(h, wt, lp + "feed_forward.output_dense.weight", (int64_t)H * I, w.w2));
      W2S_TRY(copy_f32(h, wt, lp + "feed_forward.output_dense.bias", H, &w.b2));
      W2S_TRY(copy_f32(h, wt, lp + "final_layer_norm.weight", H, &w.ln2_g));
      W2S_TRY(copy_f32(h, wt, lp + "final_layer_norm.bias", H, &w.ln2_b));
      if (c.kind == 2) {   // HF wavlm/modeling_wavlm.py:141-146
        W2S_TRY(copy_f32(h, wt, lp + "attention.gru_rel_pos_linear.weight", 8 * 64, &w.gate_w));
        W2S_TRY(copy_f32(h, wt, lp + "attention.gru_rel_pos_linear.bias", 8, &w.gate_b));
        W2S_TRY(copy_f32(h, wt, lp + "attention.gru_rel_pos_const", c.num_attention_heads, &w.gate_c));
      }
    }
    if (c.kind == 2)   // only layer 0 has the embedding; HF passes its ungated bias down the stack (:410-430)
      W2S_TRY(copy_f32(h, wt, P + "encoder.layers.0.attention.rel_attn_embed.weight",
                       (int64_t)c.num_buckets * c.num_attention_heads, &h->rel_embed));
  } else {
    const int kd = c.conv_depthwise_kernel_size;
    for (int l = 0; l < c.num_hidden_layers; ++l) {
      LayerW& w = h->layers[l];
      const std::string lp = P + "encoder.layers." + std::to_string(l) + ".";
      auto lin = [&](const std::string& nm, int64_t out, int64_t in, bf16** wdst, float** bdst) -> std::string {
        W2S_TRY(dalloc(h->allocs, wdst, (size_t)out * in));
        W2S_TRY(copy_bf16(h, wt, lp + nm + ".weight", out * in, *wdst));
        if (bdst) W2S_TRY(copy_f32(h, wt, lp + nm + ".bias", out, bdst));
        return "";
      };
      W2S_TRY(copy_f32(h, wt, lp + "ffn1_layer_norm.weight", H, &w.lnf1_g));
      W2S_TRY(copy_f32(h, wt, lp + "ffn1_layer_norm.bias", H, &w.lnf1_b));
      W2S_TRY(lin("ffn1.intermediate_dense", I, H, &w.w1, &w.b1));
      W2S_TRY(lin("ffn1.output_dense", H, I, &w.w2, &w.b2));
      W2S_TRY(copy_f32(h, wt, lp + "self_attn_layer_norm.weight", H, &w.ln1_g));
      W2S_TRY(copy_f32(h, wt, lp + "self_attn_layer_norm.bias", H, &w.ln1_b));
      // relative positions: the query projection is emitted twice, (q + u | q + v | k | v), with pos_bias_u / pos_bias_v
      // folded into the fp32 bias of the respective copy (HF :524-527 adds them to q before the two score matmuls)
      const bool relp = c.position_embeddings_type == 1;
      const int nq = relp ? 2 : 1;
      W2S_TRY(dalloc(h->allocs, &w.wqkv, (size_t)(nq + 2) * H * H));
      W2S_TRY(dalloc(h->allocs, &w.bqkv, (size_t)(nq + 2) * H));
      for (int j = 0; j < nq; ++j)
        W2S_TRY(copy_bf16(h, wt, lp + "self_attn.linear_q.weight", (int64_t)H * H, w.wqkv + (size_t)j * H * H));
      W2S_TRY(copy_bf16(h, wt, lp + "self_attn.linear_k.weight", (int64_t)H * H, w.wqkv + (size_t)nq * H * H));
      W2S_TRY(copy_bf16(h, wt, lp + "self_attn.linear_v.weight", (int64_t)H * H, w.wqkv + (size_t)(nq + 1) * H * H));
      {
        const float *bq = nullptr, *bk = nullptr, *bv = nullptr;
        W2S_TRY(wt.get(lp + "self_attn.linear_q.bias", H, &bq));
        W2S_TRY(wt.get(lp + "self_attn.linear_k.bias", H, &bk));
        W2S_TRY(wt.get(lp + "self_attn.linear_v.bias", H, &bv));
        for (int j = 0; j < nq; ++j)
          W2S_CUDA_OK(cudaMemcpy(w.bqkv + (size_t)j * H, bq, sizeof(float) * H, cudaMemcpyDeviceToDevice));
        W2S_CUDA_OK(cudaMemcpy(w.bqkv + (size_t)nq * H, bk, sizeof(float) * H, cudaMemcpyDeviceToDevice));
        W2S_CUDA_OK(cudaMemcpy(w.bqkv + (size_t)(nq + 1) * H, bv, sizeof(float) * H, cudaMemcpyDeviceToDevice));
      }
      W2S_TRY(lin("self_attn.linear_out", H, H, &w.wo, &w.bo));
      if (relp) {
        W2S_TRY(lin("self_attn.linear_pos", H, H, &w.wpos, nullptr));
        const float *u = nullptr, *v = nullptr;
        W2S_TRY(wt.get(lp + "self_attn.pos_bias_u", H, &u));
        W2S_TRY(wt.get(lp + "self_attn.pos_bias_v", H, &v));
        W2S_TRY(launch_axpy(u, w.bqkv, H, 0));
        W2S_TRY(launch_axpy(v, w.bqkv + H, H, 0));
      }
      W2S_TRY(copy_f32(h, wt, lp + "conv_module.layer_norm.weight", H, &w.lnc_g));
      W2S_TRY(copy_f32(h, wt, lp + "conv_module.layer_norm.bias", H, &w.lnc_b));
      {
        const float* src = nullptr;
        W2S_TRY(wt.get(lp + "conv_module.pointwise_conv1.weight", (int64_t)2 * H * H, &src));
        W2S_TRY(dalloc(h->allocs, &w.pw1, (size_t)2 * H * H));
        W2S_TRY(launch_repack_glu(src, w.pw1, H, H, 0));
      }
      {
        const float* src = nullptr;
        W2S_TRY(wt.get(lp + "conv_module.depthwise_conv.weight", (int64_t)H * kd, &src));
        W2S_TRY(dalloc(h->allocs, &w.dw_w, (size_t)H * kd));
        W2S_TRY(launch_transpose_f32(src, w.dw_w, H, kd, 0));   // [H][k] -> [k][H]: lanes read consecutive channels
      }
      {
        const float *g = nullptr, *b = nullptr, *mu = nullptr, *var = nullptr;
        W2S_TRY(wt.get(lp + "conv_module.batch_norm.weight", H, &g));
        W2S_TRY(wt.get(lp + "conv_module.batch_norm.bias", H, &b));
        W2S_TRY(wt.get(lp + "conv_module.batch_norm.running_mean", H, &mu));
        W2S_TRY(wt.get(lp + "conv_module.batch_norm.running_var", H, &var));
        W2S_TRY(dalloc(h->allocs, &w.dw_scale, (size_t)H));
        W2S_TRY(dalloc(h->allocs, &w.dw_shift, (size_t)H));
        W2S_TRY(launch_bn_fold(g, b, mu, var, H, 1e-5f, w.dw_scale, w.dw_shift, 0));
      }
      W2S_TRY(lin("conv_module.pointwise_conv2", H, H, &w.pw2, nullptr));
      W2S_TRY(copy_f32(h, wt, lp + "ffn2_layer_norm.weight", H, &w.lnf2_g));
      W2S_TRY(copy_f32(h, wt, lp + "ffn2_layer_norm.bias", H, &w.lnf2_b));
      W2S_TRY(lin("ffn2.intermediate_dense", I, H, &w.f2w1, &w.f2b1));
      W2S_TRY(lin("ffn2.output_dense", H, I, &w.f2w2, &w.f2b2));
      W2S_TRY(copy_f32(h, wt, lp + "final_layer_norm.weight", H, &w.lnfin_g));
      W2S_TRY(copy_f32(h, wt, lp + "final_layer_norm.bias", H, &w.lnfin_b));
    }
  }
  // lm_head rows are padded with zeros to a multiple of 32 so that any vocabulary size runs on the contraction kernel
  // (the reduction kernel only reads the first V entries of a logits row)
  {
    const int Vp = (V + 31) / 32 * 32;
    h->head_ldl = Vp;
    W2S_TRY(dalloc(h->allocs, &h->head_w, (size_t)Vp * H, true));
    W2S_TRY(copy_bf16(h, wt, "lm_head.weight", (int64_t)V * H, h->head_w));
    const float* b = nullptr;
    W2S_TRY(wt.get("lm_head.bias", V, &b));
    W2S_TRY(dalloc(h->allocs, &h->head_b, (size_t)Vp, true));
    W2S_CUDA_OK(cudaMemcpy(h->head_b, b, sizeof(float) * V, cudaMemcpyDeviceToDevice));
  }
  W2S_CUDA_OK(cudaDeviceSynchronize());
  return "";
}

GemmProblem plain_problem(const bf16* a, long long rows, int K, const bf16* w, int N) {
  GemmProblem p;
  p.a = a; p.a_cols = K; p.a_rows = rows; p.a_batches = 1; p.a_row_stride = K; p.a_batch_stride = rows * (long long)K;
  p.a_kb_per_row = K / 64; p.a_g_col = 0;
  p.w = w; p.M = (int)rows; p.N = N; p.K = K; p.Bz = 1; p.G = 1;
  p.epi.ldg = 0; p.epi.ldb = 0; p.epi.ldm = N;
  return p;
}

int64_t num_frames(const w2s_config& c, int64_t L, std::vector<int>* lens) {
  int64_t n = L;
  for (int l = 0; l < c.num_conv_layers; ++l) {
    if (n < c.conv_kernel[l]) return 0;
    n = (n - c.conv_kernel[l]) / c.conv_stride[l] + 1;
    if (lens) lens->push_back((int)n);
  }
  return n;
}

void free_workspace(w2s_handle* h) {
  h->plans.clear();
  for (void* p : h->ws_allocs) cudaFree(p);
  h->ws_allocs.clear();
  h->ws_L = -1;
}

// Block table of the current clip into the workspace (w2s_frontend_blocks); the skip is used only after this succeeded.
std::string upload_skip_table(w2s_handle* h, cudaStream_t s) {
  h->skip_tab_ok = false;
  if (!h->skip_rows || h->ws_L != h->L || h->seg_bounds.size() != (size_t)h->M + 1) return "";
  const w2s_config& c = h->cfg;
  std::vector<int32_t> tab((size_t)4 * h->skip_rows);
  if (w2s_frontend_blocks(c.num_conv_layers, c.conv_kernel, c.conv_stride, h->L, h->seg_bounds.data(), h->M, tab.data(),
                          h->skip_rows) != h->skip_rows)
    return "frontend block table: inconsistent clip geometry";
  W2S_CUDA_OK(cudaMemcpyAsync(h->skip_tab, tab.data(), sizeof(int32_t) * tab.size(), cudaMemcpyHostToDevice, s));
  W2S_CUDA_OK(cudaStreamSynchronize(s));
  h->skip_tab_ok = true;
  return "";
}

std::string ensure_workspace(w2s_handle* h, long long L) {
  if (h->ws_L == L) return "";
  cudaDeviceSynchronize();
  free_workspace(h);
  const w2s_config& c = h->cfg;
  h->Tl.clear();
  const int64_t T = num_frames(c, L, &h->Tl);
  if (T <= 0) return "clip of " + std::to_string(L) + " samples is shorter than the conv receptive field";
  h->T = (int)T;
  h->Tp = (int)((T + 63) / 64 * 64);
  if (h->auto_batch) {
    // rows = tile * T' should fill whole waves of 128-row tiles on all SMs (tile = floor(SMs * 128 * k / T')), with at
    // least 128 coalitions per tile to amortise per-launch prologues, and the conv0 output (the largest buffer) <= 8 GB
    long long k = 1;
    while ((long long)h->num_sms * 128 * k / T < 128) ++k;
    long long tile = (long long)h->num_sms * 128 * k / T;
    const long long conv0_bytes = (long long)h->Tl[0] * c.conv_dim[0] * 2;
    while (tile > 8 && tile * conv0_bytes > (8LL << 30)) tile /= 2;
    h->cfg.max_batch = (int)tile;
  }
  const size_t nb = (size_t)c.max_batch;
  const int H = c.hidden_size, I = c.intermediate_size;
  const int Cl = c.conv_dim[c.num_conv_layers - 1];
  auto& pool = h->ws_allocs;
  W2S_TRY(dalloc(pool, &h->gn_a, nb * c.conv_dim[0]));
  W2S_TRY(dalloc(pool, &h->gn_b, nb * c.conv_dim[0]));
  W2S_TRY(dalloc(pool, &h->gn_wb, nb * c.conv_dim[0] * 32));
  size_t szA = 0, szB = 0;
  for (int l = 0; l < c.num_conv_layers; ++l) {
    const size_t s = nb * (size_t)h->Tl[l] * c.conv_dim[l];
    if (l % 2 == 0) szA = s > szA ? s : szA;
    else szB = s > szB ? s : szB;
  }
  {
    std::vector<int32_t> kw(c.conv_kernel, c.conv_kernel + c.num_conv_layers), st(c.conv_stride, c.conv_stride + c.num_conv_layers);
    const int32_t whole[2] = {0, (int32_t)L};
    const int64_t nrows = c.num_conv_layers >= 2 && c.num_conv_layers - 1 <= SKIP_MAX_LAYERS
                              ? w2s_frontend_blocks(c.num_conv_layers, kw.data(), st.data(), L, whole, 1, nullptr, 0) : 0;
    // list entries pack (coalition << 16) | block: beyond that range the plans stay dense
    bool fits = nb < 32768;
    for (int l = 1; l < c.num_conv_layers; ++l) fits = fits && (h->Tl[l] + 127) / 128 < 65536;
    h->skip_rows = nrows > 0 && fits ? (int)nrows : 0;
    h->skip_tab_ok = false;
    if (h->skip_rows) {
      W2S_TRY(dalloc(pool, &h->skip_tab, (size_t)h->skip_rows));
      W2S_TRY(dalloc(pool, &h->skip_rep, nb * (c.num_conv_layers - 1)));
      for (int l = 1; l < c.num_conv_layers; ++l) {
        const size_t cap = 1 + nb * (size_t)((h->Tl[l] + 127) / 128);
        W2S_TRY(dalloc(pool, &h->skip_live[l - 1], cap));
        W2S_TRY(dalloc(pool, &h->skip_fill[l - 1], cap));
      }
    }
  }
  W2S_TRY(dalloc(pool, &h->bufA, szA));
  W2S_TRY(dalloc(pool, &h->bufB, szB ? szB : 1));
  const size_t rows = nb * (size_t)T;
  W2S_TRY(dalloc(pool, &h->fpn, rows * Cl));
  W2S_TRY(dalloc(pool, &h->h0, rows * H));
  W2S_TRY(dalloc(pool, &h->hb, rows * H));
  W2S_TRY(dalloc(pool, &h->h1, rows * H));
  W2S_TRY(dalloc(pool, &h->pre, rows * H));
  W2S_TRY(dalloc(pool, &h->qkv, rows * 4 * H));
  W2S_TRY(dalloc(pool, &h->ctx, rows * H));
  W2S_TRY(dalloc(pool, &h->ffn, rows * I));
  W2S_TRY(dalloc(pool, &h->logits, rows * (size_t)h->head_ldl));
  if (c.kind != 1) {
    W2S_TRY(dalloc(pool, &h->hp,
                   nb * (size_t)(T + c.num_conv_pos_embeddings) * c.num_conv_pos_embedding_groups * 64));
    if (c.kind == 2) {
      // WavLM: the relative-position bias table, input independent, built once per clip length from host-computed
      // buckets (HF modeling_wavlm.py:234-243, :253-271)
      const int heads = c.num_attention_heads;
      std::vector<int32_t> bk((size_t)(2 * T - 1));
      if (w2s_relative_buckets((int)T, c.num_buckets, c.max_bucket_distance, bk.data()) != 0)
        return "WavLM: num_buckets / max_bucket_distance out of range";
      int32_t* bk_dev = nullptr;
      W2S_TRY(dalloc(pool, &bk_dev, bk.size()));
      W2S_CUDA_OK(cudaMemcpy(bk_dev, bk.data(), sizeof(int32_t) * bk.size(), cudaMemcpyHostToDevice));
      W2S_TRY(dalloc(pool, &h->rel_bias, (size_t)heads * rel_bias_ld((int)T)));
      W2S_TRY(launch_rel_bias_table(h->rel_embed, bk_dev, (int)T, heads, h->rel_bias, 0));
      W2S_TRY(dalloc(pool, &h->gate, rows * heads));
      W2S_CUDA_OK(cudaDeviceSynchronize());
    }
  } else {
    if (c.position_embeddings_type == 2) W2S_TRY(dalloc(pool, &h->hrot, rows * H));
    if (c.position_embeddings_type == 1) {
      // relative position table and its per-layer projection linear_pos(pe): input independent, built once per
      // clip length (HF modeling_wav2vec2_conformer.py:159-205, :509-518)
      const long long R = 2 * T - 1;
      bf16* pe = nullptr;
      W2S_TRY(dalloc(pool, &pe, (size_t)R * H));
      W2S_TRY(launch_relpos((int)T, H, pe, 0));
      for (int l = 0; l < c.num_hidden_layers; ++l) {
        LayerW& w = h->layers[l];
        W2S_TRY(dalloc(pool, &w.pos_proj, (size_t)R * H));
        GemmProblem p = plain_problem(pe, R, H, w.wpos, H);
        p.epi.out = w.pos_proj;
        GemmLaunch gl;
        W2S_TRY(gemm_prepare(p, h->num_sms, &gl));
        W2S_TRY((h->cfg.flags & W2S_FLAG_VALIDATE_GEMM) ? gemm_launch_simt(gl, 0) : gemm_launch_tc(gl, 0));
      }
      W2S_CUDA_OK(cudaDeviceSynchronize());
    }
  }
  h->ws_L = L;
  // a workspace rebuilt for the clip's length (e.g. after w2s_eval_waveforms at another length) gets the clip's table back
  if (L == h->L) W2S_TRY(upload_skip_table(h, 0));
  return "";
}

// ------------------------------------------------------------------------------------------------
// plan construction: every launch of one batch-tile forward, with tensor maps encoded once
// ------------------------------------------------------------------------------------------------
struct PlanBuilder {
  w2s_handle* h;
  Plan* plan;
  int n;
  bool simt_gemm, simt_attn;
  int fill;   // which conv0 instantiation reads the input rows (kernels.cuh: Fill)
  bool skip;  // conv1 .. conv6 contract only the blocks that see kept audio (frontend_skip.cu)

  std::string add_gemm(const std::string& name, const GemmProblem& p) {
    GemmLaunch* gl = new GemmLaunch();
    plan->gemms.push_back(gl);
    W2S_TRY(gemm_prepare(p, h->num_sms, gl));
    const bool simt = simt_gemm;
    Step st{name, [gl, simt](cudaStream_t s) { return simt ? gemm_launch_simt(*gl, s) : gemm_launch_tc(*gl, s); }};
    st.flops = 2.0 * p.M * (double)p.N * p.K * p.Bz * p.G;
    plan->steps.push_back(std::move(st));
    return "";
  }
  void add(const std::string& name, std::function<std::string(cudaStream_t)> f, double flops = 0.0, double bytes = 0.0) {
    Step st{name, std::move(f)};
    st.flops = flops;
    st.bytes = bytes;
    plan->steps.push_back(std::move(st));
  }
  std::string add_ln(const std::string& name, const void* in, int in_fp32, long long rows, int H, const float* g,
                     const float* b, float eps, int act, bf16* out, float* out_f32, const bf16* residual = nullptr) {
    // algorithmic HBM bytes: the row read once (+ the bf16 residual) and every output written once
    const double bytes = (double)rows * H * ((in_fp32 ? 4 : 2) + (residual ? 2 : 0) + (out ? 2 : 0) + (out_f32 ? 4 : 0));
    add(name, [=](cudaStream_t s) { return launch_layernorm(in, in_fp32, rows, H, g, b, eps, act, out, out_f32, s, residual); },
        0.0, bytes);
    return "";
  }
  static GemmProblem plain(const bf16* a, long long rows, int K, const bf16* w, int N) {
    return plain_problem(a, rows, K, w, N);
  }

  std::string build_conformer();

  // K9: lm_head on the contraction kernel (N = vocab padded to a multiple of 32) into an fp32 logits buffer, then the
  // warp-level reduction, which reads mode / targets / destination from the per-call argument block.  The fused
  // CUDA-core head kernel exists for W2S_FLAG_VALIDATE_GEMM only.
  std::string add_head() {
    const w2s_config& c = h->cfg;
    const int T = h->T, H = c.hidden_size, V = c.vocab_size;
    HeadParams hp{};
    hp.h = h->hb; hp.w = h->head_w; hp.bias = h->head_b;
    hp.n = n; hp.T = T; hp.H = H; hp.V = V; hp.ldl = h->head_ldl; hp.dyn = h->dyn_dev;
    if (simt_gemm) {
      add("head", [=](cudaStream_t s) { return launch_head(hp, s); });
      return "";
    }
    GemmProblem p = plain(h->hb, (long long)n * T, H, h->head_w, h->head_ldl);
    p.epi.bias = h->head_b;
    p.epi.out = h->logits;
    p.epi.out_fp32 = 1;
    W2S_TRY(add_gemm("lm_head", p));
    const float* logits = h->logits;
    add("head_reduce", [=](cudaStream_t s) { return launch_head_reduce(logits, hp, s); }, 0.0,
        (double)n * T * V * 4.0);
    return "";
  }

  std::string build() {
    const w2s_config& c = h->cfg;
    const int T = h->T, H = c.hidden_size, I = c.intermediate_size;
    const bool layer = c.feat_extract_norm == 1;
    const long long rows = (long long)n * T;
    w2s_handle* hh = h;
    const int nn = n;

    // ---- K1: conv0 + norm + GELU -------------------------------------------------------------------
    {
      Conv0Params cp{};
      cp.dyn = h->dyn_dev;
      cp.n = n; cp.L = (int)h->ws_L; cp.T0 = h->Tl[0]; cp.C = c.conv_dim[0]; cp.kw = c.conv_kernel[0];
      cp.stride = c.conv_stride[0];
      cp.w = h->conv0_w; cp.bias = h->conv0_b; cp.gamma = h->norm0_g; cp.beta = h->norm0_b;
      cp.gn_a = h->gn_a; cp.gn_b = h->gn_b; cp.gn_wb = h->gn_wb;
      cp.ln_wbar = h->ln0_wbar; cp.ln_gram = h->ln0_gram; cp.ln_wb = h->ln0_wb;
      cp.ln_bmean = h->ln0_bmean; cp.ln_b2mean = h->ln0_b2mean; cp.ln_wb48 = h->ln0_wb48;
      cp.out = h->bufA;
      const int fill = this->fill;
      // with a background every row reads its background row besides the clip, with cells the F band components (all
      // L2-resident across the tile)
      const double wave_bytes = (fill == FILL_BANDS ? 4.0 * h->bands_F : fill == FILL_BG ? 8.0 : 4.0) * (double)h->ws_L;
      if (!layer)
        add("conv0_stats", [=](cudaStream_t s) { return launch_conv0_stats(cp, s, fill); }, 0.0,
            (wave_bytes + (double)cp.C * (8.0 + 64.0)) * n);
      add("conv0", [=](cudaStream_t s) { return launch_conv0(cp, layer, s, fill); },
          2.0 * cp.T0 * (double)cp.C * cp.kw * n, ((double)cp.T0 * cp.C * 2.0 + wave_bytes) * n);
    }
    // ---- K2: conv1..6 as implicit GEMM over the stride-row view of the previous layer ---------------------
    // With the skip, the block lists of every layer are built first (one launch), each contraction walks its list and a
    // fill launch copies the representative row into the blocks of constant frames that the next layer reads.
    SkipParams sp{};
    const size_t list_step = plan->steps.size();
    if (skip) {
      sp.dyn = h->dyn_dev; sp.tab = h->skip_tab; sp.nl = c.num_conv_layers - 1; sp.n = n; sp.total = h->skip_rows;
      sp.rep = h->skip_rep;
      for (int l = 0, o = 0; l < sp.nl; ++l) {
        sp.nb[l] = (h->Tl[l + 1] + 127) / 128;
        sp.off[l] = o;
        o += sp.nb[l];
        sp.live[l] = h->skip_live[l];
        sp.fill[l] = h->skip_fill[l];
      }
      add("frontend_lists", nullptr, 0.0, (double)n * (h->skip_rows * (16.0 + 8.0) + h->zwords * 4.0));
    }
    bf16* cur = h->bufA;
    for (int l = 1; l < c.num_conv_layers; ++l) {
      bf16* nxt = (l % 2 == 1) ? h->bufB : h->bufA;
      const int Cin = c.conv_dim[l - 1], Cout = c.conv_dim[l], kw = c.conv_kernel[l], st = c.conv_stride[l];
      const int Tin = h->Tl[l - 1], Tout = h->Tl[l];
      if ((st * Cin) % 64) return "conv layer " + std::to_string(l) + ": stride * in_channels must be a multiple of 64";
      GemmProblem p;
      p.a = cur; p.a_cols = (long long)st * Cin; p.a_rows = (Tin + st - 1) / st; p.a_batches = n;
      p.a_row_stride = (long long)st * Cin; p.a_batch_stride = (long long)Tin * Cin;
      p.a_kb_per_row = st * Cin / 64; p.a_g_col = 0;
      p.w = h->conv_w[l]; p.M = Tout; p.N = Cout; p.K = kw * Cin; p.Bz = n; p.G = 1;
      p.epi.bias = h->conv_b[l];
      p.epi.act = layer ? ACT_NONE : ACT_GELU;
      p.epi.out = nxt; p.epi.ldb = (long long)Tout * Cout; p.epi.ldm = Cout;
      W2S_TRY(add_gemm("conv" + std::to_string(l), p));
      const GemmLaunch* gl = plan->gemms.back();
      sp.dense[l - 1] = !(gl->mc == 2 && gl->bn == 256 && gl->tma_out && !simt_gemm);
      if (skip && !sp.dense[l - 1]) {
        Step& st = plan->steps.back();
        const int* live = sp.live[l - 1];
        st.run = [gl, live](cudaStream_t s) { return gemm2_launch_list(*gl, live, s); };
        st.flops = 2.0 * 128 * (double)p.N * p.K;   // per listed block
        st.work = live;
        const int* fl = sp.fill[l - 1];
        const int* rp = sp.rep + (size_t)(l - 1) * n;
        const int nsm = h->num_sms;
        Step f{"conv" + std::to_string(l) + "_fill",
               [fl, rp, nxt, Tout, Cout, nsm](cudaStream_t s) { return launch_skip_fill(fl, rp, nxt, Tout, Cout, nsm, s); }};
        f.bytes = 128.0 * Cout * 2.0;   // per filled block (the representative rows are L2-resident)
        f.work = fl;
        plan->steps.push_back(std::move(f));
      }
      if (layer)
        add_ln("conv" + std::to_string(l) + "_ln_gelu", nxt, 0, (long long)n * Tout, Cout, h->conv_ln_g[l],
               h->conv_ln_b[l], 1e-5f, ACT_GELU, nxt, nullptr);
      cur = nxt;
    }
    if (skip) plan->steps[list_step].run = [sp](cudaStream_t s) { return launch_skip_lists(sp, s); };
    // ---- K3: feature projection ---------------------------------------------------------------------------
    const int Cl = c.conv_dim[c.num_conv_layers - 1];
    add_ln("featproj_ln", cur, 0, rows, Cl, h->fp_ln_g, h->fp_ln_b, c.layer_norm_eps, ACT_NONE, h->fpn, nullptr);
    {
      GemmProblem p = plain(h->fpn, rows, Cl, h->fp_w, H);
      p.epi.bias = h->fp_b;
      if (c.kind != 1) {
        p.epi.out = h->h0;
      } else {  // conformer: the un-normalised residual stream lives in fp32
        p.epi.out = h->pre;
        p.epi.out_fp32 = 1;
      }
      W2S_TRY(add_gemm("featproj", p));
    }
    if (c.kind == 1) return build_conformer();
    const bool wavlm = c.kind == 2;
    const bool stable = c.do_stable_layer_norm != 0;
    // ---- K4: positional conv (grouped, k=128) + GELU + residual (+ LayerNorm) ----------------------------
    {
      const int G = c.num_conv_pos_embedding_groups, kp = c.num_conv_pos_embeddings, cpg = H / G;
      add("pos_pad", [=](cudaStream_t s) { return launch_pos_pad(hh->h0, nn, T, H, G, kp, hh->hp, s); }, 0.0,
          ((double)T * H + (double)(T + kp) * G * 64) * 2.0 * n);
      GemmProblem p;
      p.a = h->hp; p.a_cols = (long long)G * 64; p.a_rows = T + kp; p.a_batches = n;
      p.a_row_stride = (long long)G * 64; p.a_batch_stride = (long long)(T + kp) * G * 64;
      p.a_kb_per_row = 1; p.a_g_col = 64;
      p.w = h->pos_w; p.M = T; p.N = cpg; p.K = kp * 64; p.Bz = n; p.G = G;
      p.epi.bias = h->pos_b; p.epi.act = ACT_GELU;
      p.epi.residual = h->h0; p.epi.res_fp32 = 0;
      p.epi.out = h->pre; p.epi.out_fp32 = 1;
      p.epi.ldg = cpg; p.epi.ldb = (long long)T * H; p.epi.ldm = H;
      if (!simt_gemm && posconv_supported(H, G, kp)) {
        PosConvPlan* pc = nullptr;
        W2S_TRY(posconv_prepare(h->hp, h->pos_w, n, T, H, G, kp, p.epi, h->num_sms, &pc));
        plan->posconv.push_back(pc);
        add("pos_conv", [=](cudaStream_t s) { return posconv_launch(pc, s); }, 2.0 * n * T * (double)H * cpg * kp);
      } else {
        W2S_TRY(add_gemm("pos_conv", p));
      }
      if (!stable)
        add_ln("encoder_ln", h->pre, 1, rows, H, h->enc_ln_g, h->enc_ln_b, c.layer_norm_eps, ACT_NONE, h->hb, nullptr);
    }
    // ---- K5-K8: transformer layers ------------------------------------------------------------------------
    AttnParams ap{};
    ap.qkv = h->qkv; ap.ctx = h->ctx; ap.B = n; ap.T = T; ap.Tp = h->Tp; ap.H = H;
    ap.heads = c.num_attention_heads; ap.hd = H / c.num_attention_heads;
    ap.ld = 3 * H; ap.q_off = 0; ap.qv_off = 0; ap.k_off = H; ap.v_off = 2 * H;
    ap.scale = 1.0f / sqrtf((float)ap.hd);
    if (wavlm) {
      ap.rel_bias = h->rel_bias;
      ap.gate = h->gate;
    }
    // attention: the persistent tcgen05 kernel, or -- W2S_FLAG_VALIDATE_ATTN only -- the CUDA-core cross-check.
    // A shape the tensor-core kernel cannot take is an error, never a silent change of code path.
    AttnFaPlan* afl = nullptr;
    if (!simt_attn) {
      if (!attention_fa_supported(ap))
        return "attention: head_dim " + std::to_string(ap.hd) + " is not supported (the tcgen05 kernel needs head_dim 64)";
      W2S_TRY(attention_fa_prepare(ap, h->num_sms, &afl));
      plan->attn_fa.push_back(afl);
    }
    const double attn_flops = 4.0 * T * (double)T * H * n;
    const int act = c.hidden_act == 1 ? ACT_SWISH : ACT_GELU;
    const bool ln_res = !stable && (H == 128 || H == 256 || H == 512 || H == 768 || H == 1024);
    // Post-LN models write the pre-LayerNorm tensor of out_proj / ffn2 as bf16: it halves the traffic of the one
    // HBM-bound contraction and of both LayerNorms (163.5 vs 170.4 ms per C2 step) at the price of one more bf16
    // rounding per sub-layer, inside the parity tolerances (tests/test_gpu_parity.py).  W2S_FLAG_FP32_PRELN restores fp32.
    const bool bf16_preln = (c.flags & W2S_FLAG_FP32_PRELN) == 0;
    const int pre32 = (bf16_preln && ln_res) ? 0 : 1;
    for (int l = 0; l < c.num_hidden_layers; ++l) {
      const LayerW& w = h->layers[l];
      const std::string ls = "L" + std::to_string(l) + ".";
      if (stable) add_ln(ls + "ln1", h->pre, 1, rows, H, w.ln1_g, w.ln1_b, c.layer_norm_eps, ACT_NONE, h->hb, nullptr);
      {
        GemmProblem p = plain(h->hb, rows, H, w.wqkv, 3 * H);
        p.epi.bias = w.bqkv;
        p.epi.out = h->qkv;
        W2S_TRY(add_gemm(ls + "qkv", p));
      }
      if (wavlm) {   // the gate reads the attention input hb (HF modeling_wavlm.py:160-176)
        const float *gw = w.gate_w, *gb = w.gate_b, *gc = w.gate_c;
        const int heads = ap.heads;
        add(ls + "wavlm_gate", [=](cudaStream_t s) { return launch_wavlm_gate(hh->hb, nn, T, heads, gw, gb, gc, hh->gate, s); },
            2.0 * rows * 8 * H, (double)rows * H * 2.0 + (double)rows * heads * 4.0);
      }
      if (afl) add(ls + "attention", [=](cudaStream_t s) { return attention_fa_launch(afl, s); }, attn_flops);
      else add(ls + "attention", [=](cudaStream_t s) { return launch_attention_simt(ap, s); }, attn_flops);
      {
        GemmProblem p = plain(h->ctx, rows, H, w.wo, H);
        p.epi.bias = w.bo;
        // post-LN: the bf16 residual is added by the LayerNorm kernel (coalesced), not by the GEMM epilogue
        if (stable || !ln_res) {
          p.epi.residual = stable ? (const void*)h->pre : (const void*)h->hb;
          p.epi.res_fp32 = stable ? 1 : 0;
        }
        p.epi.out = h->pre; p.epi.out_fp32 = pre32;
        W2S_TRY(add_gemm(ls + "out_proj", p));
      }
      if (stable) add_ln(ls + "ln2", h->pre, 1, rows, H, w.ln2_g, w.ln2_b, c.layer_norm_eps, ACT_NONE, h->h1, nullptr);
      else add_ln(ls + "ln1", h->pre, pre32, rows, H, w.ln1_g, w.ln1_b, c.layer_norm_eps, ACT_NONE, h->h1, nullptr,
                  ln_res ? h->hb : nullptr);
      {
        GemmProblem p = plain(h->h1, rows, H, w.w1, I);
        p.epi.bias = w.b1; p.epi.act = act;
        p.epi.out = h->ffn;
        W2S_TRY(add_gemm(ls + "ffn1", p));
      }
      {
        GemmProblem p = plain(h->ffn, rows, I, w.w2, H);
        p.epi.bias = w.b2;
        if (stable || !ln_res) {
          p.epi.residual = stable ? (const void*)h->pre : (const void*)h->h1;
          p.epi.res_fp32 = stable ? 1 : 0;
        }
        p.epi.out = h->pre; p.epi.out_fp32 = pre32;
        W2S_TRY(add_gemm(ls + "ffn2", p));
      }
      if (!stable) add_ln(ls + "ln2", h->pre, pre32, rows, H, w.ln2_g, w.ln2_b, c.layer_norm_eps, ACT_NONE, h->hb, nullptr,
                          ln_res ? h->h1 : nullptr);
    }
    if (stable)
      add_ln("encoder_ln", h->pre, 1, rows, H, h->enc_ln_g, h->enc_ln_b, c.layer_norm_eps, ACT_NONE, h->hb, nullptr);
    // ---- K9: lm_head + reduction ---------------------------------------------------------------------------
    W2S_TRY(add_head());
    return "";
  }
};

std::string PlanBuilder::build_conformer() {
  // HF wav2vec2_conformer/modeling_wav2vec2_conformer.py:633-717 (encoder), :568-630 (layer).  The residual
  // stream `pre` is fp32; every sub-block reads a LayerNorm'd bf16 copy and adds its result back in the
  // GEMM epilogue (alpha = 0.5 for the two macaron feed-forward blocks).
  const w2s_config& c = h->cfg;
  const int T = h->T, H = c.hidden_size, I = c.intermediate_size;
  const long long rows = (long long)n * T;
  const int act = c.hidden_act == 1 ? ACT_SWISH : ACT_GELU;
  w2s_handle* hh = h;
  const int nn = n;
  AttnParams ap{};
  const bool rel = c.position_embeddings_type == 1, rotary = c.position_embeddings_type == 2;
  ap.qkv = h->qkv; ap.ctx = h->ctx; ap.B = n; ap.T = T; ap.Tp = h->Tp; ap.H = H;
  ap.heads = c.num_attention_heads; ap.hd = H / c.num_attention_heads;
  ap.scale = 1.0f / sqrtf((float)ap.hd);
  const int nq = rel ? 2 : 1;
  ap.ld = (nq + 2) * H; ap.q_off = 0; ap.qv_off = rel ? H : 0; ap.k_off = nq * H; ap.v_off = (nq + 1) * H;
  AttnFaPlan* afl = nullptr;
  if (!simt_attn && !rel) {
    if (!attention_fa_supported(ap))
      return "attention: head_dim " + std::to_string(ap.hd) + " is not supported (the tcgen05 kernel needs head_dim 64)";
    W2S_TRY(attention_fa_prepare(ap, h->num_sms, &afl));
    plan->attn_fa.push_back(afl);
  }
  double attn_flops = 4.0 * T * (double)T * H * n;
  if (rel) attn_flops += 2.0 * T * (2.0 * T - 1) * H * n;   // (q + v) . linear_pos(pe) over the 2T'-1 relative positions
  auto ffn = [&](const std::string& ls, const float* lg, const float* lb, const bf16* w1, const float* b1,
                 const bf16* w2, const float* b2) -> std::string {
    add_ln(ls + "ln", h->pre, 1, rows, H, lg, lb, 1e-5f, ACT_NONE, h->hb, nullptr);
    GemmProblem p = plain(h->hb, rows, H, w1, I);
    p.epi.bias = b1; p.epi.act = act; p.epi.out = h->ffn;
    W2S_TRY(add_gemm(ls + "ffn1", p));
    GemmProblem q = plain(h->ffn, rows, I, w2, H);
    q.epi.bias = b2; q.epi.alpha = 0.5f;
    q.epi.residual = h->pre; q.epi.res_fp32 = 1; q.epi.out = h->pre; q.epi.out_fp32 = 1;
    W2S_TRY(add_gemm(ls + "ffn2", q));
    return "";
  };
  for (int l = 0; l < c.num_hidden_layers; ++l) {
    const LayerW& w = h->layers[l];
    const std::string ls = "L" + std::to_string(l) + ".";
    W2S_TRY(ffn(ls + "mac1_", w.lnf1_g, w.lnf1_b, w.w1, w.b1, w.w2, w.b2));
    // ---- self-attention ----
    add_ln(ls + "attn_ln", h->pre, 1, rows, H, w.ln1_g, w.ln1_b, 1e-5f, ACT_NONE, h->hb, nullptr);
    if (rotary) {
      const int base = c.rotary_embedding_base, hd = ap.hd;
      add(ls + "rotary", [=](cudaStream_t s) { return launch_rotary(hh->hb, rows, T, H, hd, base, hh->hrot, s); }, 0.0,
          (double)rows * H * 4.0);
      GemmProblem p = plain(h->hrot, rows, H, w.wqkv, 2 * H);
      p.epi.bias = w.bqkv; p.epi.out = h->qkv; p.epi.ldm = 3 * H;
      W2S_TRY(add_gemm(ls + "qk", p));
      GemmProblem v = plain(h->hb, rows, H, w.wqkv + (size_t)2 * H * H, H);
      v.epi.bias = w.bqkv + 2 * H; v.epi.out = h->qkv + 2 * H; v.epi.ldm = 3 * H;
      W2S_TRY(add_gemm(ls + "v", v));
    } else {
      GemmProblem p = plain(h->hb, rows, H, w.wqkv, (nq + 2) * H);
      p.epi.bias = w.bqkv; p.epi.out = h->qkv;
      W2S_TRY(add_gemm(ls + "qkv", p));
    }
    if (afl) {
      add(ls + "attention", [=](cudaStream_t s) { return attention_fa_launch(afl, s); }, attn_flops);
    } else {
      AttnParams lp = ap;
      if (rel) lp.pos_proj = w.pos_proj;
      if (rel && !simt_attn) {
        if (!attention_rel_supported(lp))
          return "attention (relative positions): head_dim " + std::to_string(lp.hd) + " is not supported (needs 64)";
        AttnRelPlan* rp = nullptr;
        W2S_TRY(attention_rel_prepare(lp, &rp));
        plan->attn_rel.push_back(rp);
        add(ls + "attention", [=](cudaStream_t s) { return attention_rel_launch(rp, s); }, attn_flops);
      } else {
        add(ls + "attention", [=](cudaStream_t s) { return launch_attention_simt(lp, s); }, attn_flops);
      }
    }
    {
      GemmProblem p = plain(h->ctx, rows, H, w.wo, H);
      p.epi.bias = w.bo; p.epi.residual = h->pre; p.epi.res_fp32 = 1; p.epi.out = h->pre; p.epi.out_fp32 = 1;
      W2S_TRY(add_gemm(ls + "out_proj", p));
    }
    // ---- convolution module: LN -> pointwise (GLU epilogue) -> depthwise + BatchNorm + act -> pointwise ----
    add_ln(ls + "conv_ln", h->pre, 1, rows, H, w.lnc_g, w.lnc_b, 1e-5f, ACT_NONE, h->hb, nullptr);
    {
      GemmProblem p = plain(h->hb, rows, H, w.pw1, 2 * H);
      p.epi.glu = 1; p.epi.out = h->h1; p.epi.ldm = H;
      W2S_TRY(add_gemm(ls + "pw1_glu", p));
    }
    {
      const int kd = c.conv_depthwise_kernel_size;
      const float *dw = w.dw_w, *sc = w.dw_scale, *sh = w.dw_shift;
      add(ls + "depthwise", [=](cudaStream_t s) { return launch_depthwise(hh->h1, nn, T, H, kd, dw, sc, sh, act, hh->ctx, s); },
          2.0 * rows * (double)H * kd, (double)rows * H * 4.0);
    }
    {
      GemmProblem p = plain(h->ctx, rows, H, w.pw2, H);
      p.epi.residual = h->pre; p.epi.res_fp32 = 1; p.epi.out = h->pre; p.epi.out_fp32 = 1;
      W2S_TRY(add_gemm(ls + "pw2", p));
    }
    W2S_TRY(ffn(ls + "mac2_", w.lnf2_g, w.lnf2_b, w.f2w1, w.f2b1, w.f2w2, w.f2b2));
    add_ln(ls + "final_ln", h->pre, 1, rows, H, w.lnfin_g, w.lnfin_b, 1e-5f, ACT_NONE, nullptr, h->pre);
  }
  add_ln("encoder_ln", h->pre, 1, rows, H, h->enc_ln_g, h->enc_ln_b, c.layer_norm_eps, ACT_NONE, h->hb, nullptr);
  W2S_TRY(add_head());
  return "";
}

// plan kind: the Fill of conv0, plus PLAN_SKIP for coalition evaluations that take the constant-frame skip
constexpr int PLAN_SKIP = 8;

std::string get_plan(w2s_handle* h, int n, int fill, Plan** out) {
  auto it = h->plans.find({n, fill});
  if (it != h->plans.end()) {
    *out = it->second.get();
    return "";
  }
  std::unique_ptr<Plan> pl(new Plan());
  pl->n = n;
  PlanBuilder b{h, pl.get(), n, (h->cfg.flags & W2S_FLAG_VALIDATE_GEMM) != 0, (h->cfg.flags & W2S_FLAG_VALIDATE_ATTN) != 0,
                fill & ~PLAN_SKIP, (fill & PLAN_SKIP) != 0};
  W2S_TRY(b.build());
  *out = pl.get();
  h->plans[{n, fill}] = std::move(pl);
  return "";
}

// D of the current mode: transcripts (CTC), references (ERRORS) or (frame, token) targets (LOGIT / LOGPROB; 0 otherwise)
int out_count(const w2s_handle* h) {
  return h->mode == W2S_OUT_CTC ? h->ctc_D : h->mode == W2S_OUT_ERRORS ? h->err_D : h->D;
}

// blank id of the current mode: that of the references (ERRORS), else that of the transcripts
int out_blank(const w2s_handle* h) { return h->mode == W2S_OUT_ERRORS ? h->err_blank : h->ctc_blank; }

int64_t out_width(const w2s_handle* h, int64_t L) {
  const int64_t T = num_frames(h->cfg, L, nullptr);
  switch (h->mode) {
    case W2S_OUT_MAX: return T;
    case W2S_OUT_MEAN: return 1;
    case W2S_OUT_LOGITS: return T * h->cfg.vocab_size;
    default: return out_count(h);
  }
}

// Capture every launch of a tile plan into one CUDA graph (on the handle's own stream: the caller's may be the legacy
// default stream, which cannot be captured).  A capture that fails for any reason leaves the plan on the eager path.
void capture_plan(w2s_handle* h, Plan* pl) {
  pl->graph_failed = true;
  if (cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
    cudaGetLastError();
    return;
  }
  bool ok = true;
  for (const Step& st : pl->steps)
    if (!st.run(h->cap_stream).empty()) {
      ok = false;
      break;
    }
  cudaGraph_t g = nullptr;
  if (cudaStreamEndCapture(h->cap_stream, &g) != cudaSuccess || !g) ok = false;
  if (ok && cudaGraphInstantiate(&pl->exec, g, 0) != cudaSuccess) {
    pl->exec = nullptr;
    ok = false;
  }
  if (g) cudaGraphDestroy(g);
  cudaGetLastError();
  pl->graph_failed = !ok;
}

// Profiled launch of one step (w2s_profile_enable): CUDA events around it, accumulated per launch class.
std::string run_step(w2s_handle* h, const Step& st, cudaStream_t s) {
  ProfRec rec;
  if (h->profiling) {
    rec.name = st.name;
    rec.flops = st.flops;
    rec.bytes = st.bytes;
    cudaEventCreate(&rec.e0);
    cudaEventCreate(&rec.e1);
    cudaEventRecord(rec.e0, s);
  }
  std::string e = st.run(s);
  if (h->profiling) {
    cudaEventRecord(rec.e1, s);
    if (st.work) {   // the work this launch executed: entries of its device list
      int cnt = 0;
      cudaMemcpyAsync(&cnt, st.work, sizeof(int), cudaMemcpyDeviceToHost, s);
      cudaStreamSynchronize(s);
      rec.flops *= cnt;
      rec.bytes *= cnt;
    }
    h->prof.push_back(rec);
  }
  return e.empty() ? "" : st.name + ": " + e;
}

// One evaluation call: rows in tiles of max_batch (the last tile ragged), each tile = one DynArgs update + the plan.
// With a background (zbits set and bg_B > 0) the call evaluates K * B rows, row g = (coalition g / B, background row
// g % B), into the handle's per-row scratch, and bg_mean_kernel reduces each coalition's B rows into out[K, width].
// With time-frequency cells (zbits set and bands_F > 0) each coalition is one row whose bit row has one bit per cell.
std::string run_batches(w2s_handle* h, const uint32_t* zbits, const float* x, long long ld, int64_t K, float* out,
                        cudaStream_t s) {
  const int64_t width = out_width(h, h->ws_L);
  if (width <= 0) return "no outputs selected (w2s_set_targets)";
  const bool graphs = h->use_graphs && !h->profiling;
  const bool bg = zbits && h->bg_B > 0;
  const bool cells = zbits && h->bands_F > 0;
  const int fill = bg ? FILL_BG : cells ? FILL_BANDS : FILL_PLAIN;
  const int zwords = cells ? (h->M * h->bands_F + 31) / 32 : h->zwords;
  const int64_t rows = bg ? K * h->bg_B : K;
  // the constant-frame skip: coalitions over the baseline fill, group-norm front end, tensor-core contractions
  const bool skip = zbits && fill == FILL_PLAIN && h->skip_tab_ok && h->cfg.feat_extract_norm == 0 &&
                    (h->cfg.flags & (W2S_FLAG_DENSE_FRONTEND | W2S_FLAG_VALIDATE_GEMM)) == 0;
  float* dst = out;
  if (bg) {
    W2S_TRY(grow(&h->bg_rows, &h->bg_rows_cap, rows * width, 0, s));
    dst = h->bg_rows;
  }
  for (int64_t k0 = 0; k0 < rows; k0 += h->cfg.max_batch) {
    const int n = (int)((rows - k0) < h->cfg.max_batch ? (rows - k0) : h->cfg.max_batch);
    Plan* pl = nullptr;
    W2S_TRY(get_plan(h, n, fill | (skip ? PLAN_SKIP : 0), &pl));
    DynArgs d{};
    if (cells) {
      d.seg_id = h->seg_id; d.zbits = zbits + k0 * zwords; d.zwords = zwords;
      d.bands = h->bands; d.F = h->bands_F; d.ld = h->bands_L;
    } else if (bg) {
      d.clip = h->clip; d.seg_id = h->seg_id; d.zbits = zbits; d.zwords = h->zwords;
      d.bg = h->bg; d.B = h->bg_B; d.ld = h->bg_L; d.row0 = k0;
    } else if (zbits) {
      d.clip = h->clip; d.seg_id = h->seg_id; d.zbits = zbits + k0 * h->zwords; d.zwords = h->zwords;
      d.baseline = h->baseline;
    } else {
      d.x = x + k0 * ld; d.ld = ld;
    }
    d.out = dst + k0 * width;
    d.mode = h->mode; d.D = out_count(h);
    d.frames = h->targets; d.tokens = h->targets ? h->targets + h->D : nullptr;
    d.ctc_labels = h->ctc_labels; d.ctc_offsets = h->ctc_offsets;
    d.blank = out_blank(h);
    d.err_tab = h->err_tab; d.err_unit = h->err_unit; d.delim = h->err_delim;
    set_dyn_kernel<<<1, 1, 0, s>>>(h->dyn_dev, d);
    W2S_CUDA_OK(cudaGetLastError());
    h->launches += 1 + (long long)pl->steps.size();
    if (graphs && !pl->exec && !pl->graph_failed) capture_plan(h, pl);
    if (graphs && pl->exec) {
      W2S_CUDA_OK(cudaGraphLaunch(pl->exec, s));
      continue;
    }
    for (const Step& st : pl->steps) W2S_TRY(run_step(h, st, s));
  }
  if (bg) {
    const float *rows_in = h->bg_rows, *w = h->bg_w;
    const int B = h->bg_B;
    Step st{"bg_mean", [=](cudaStream_t st_s) { return launch_bg_mean(rows_in, w, B, K, width, out, st_s); }};
    st.bytes = 4.0 * (double)K * width * (B + 1);
    h->launches += 1;
    W2S_TRY(run_step(h, st, s));
  }
  return "";
}

// the first transcript that needs more frames than T, as an error
std::string check_transcripts(const w2s_handle* h, int64_t T) {
  if (h->ctc_D <= 0) return "no transcripts set (w2s_set_transcripts)";
  for (int d = 0; d < h->ctc_D; ++d)
    if (h->ctc_need[d] > T)
      return "transcript " + std::to_string(d) + " needs " + std::to_string(h->ctc_need[d]) + " frames, the clip has " +
             std::to_string(T);
  return "";
}

// the band components against the clip of the call (w2s_set_clip may have changed it since w2s_set_bands)
std::string check_bands(const w2s_handle* h) {
  if (h->bands_F <= 0) return "";
  if (h->bands_L != h->L)
    return "the band components have " + std::to_string(h->bands_L) + " samples, the clip has " + std::to_string(h->L) +
           " (w2s_set_bands again, or clear them with F = 0)";
  if ((long long)h->M * h->bands_F > 2048)
    return std::to_string(h->M) + " segments x " + std::to_string(h->bands_F) + " bands = " +
           std::to_string((long long)h->M * h->bands_F) + " cells; at most 2048 are supported";
  return "";
}

std::string check_targets(const w2s_handle* h) {
  if (h->mode == W2S_OUT_CTC) return check_transcripts(h, h->T);
  if (h->mode == W2S_OUT_LOGIT || h->mode == W2S_OUT_LOGPROB) {
    if (out_count(h) <= 0 || !h->targets) return "targets not set (w2s_set_targets)";
    if (h->max_frame >= h->T)
      return "target frame " + std::to_string(h->max_frame) + " beyond the clip's " + std::to_string(h->T) + " frames";
  }
  return "";
}

// w2s_set_transcripts / w2s_debug_ctc argument checks (host only); fills need[d] with the frames transcript d needs
std::string validate_transcripts(const int32_t* labels, const int32_t* offsets, int D, int blank, int V,
                                 std::vector<int>* need) {
  if (D < 1 || !offsets) return "need D >= 1 transcripts and their offsets";
  if (blank < 0 || blank >= V) return "blank " + std::to_string(blank) + " outside the vocabulary [0, " + std::to_string(V) + ")";
  if (offsets[0] != 0) return "offsets[0] must be 0";
  need->assign((size_t)D, 0);
  for (int d = 0; d < D; ++d) {
    const int U = offsets[d + 1] - offsets[d];
    if (U < 0) return "offsets must be non-decreasing (transcript " + std::to_string(d) + ")";
    if (U > W2S_MAX_TRANSCRIPT)
      return "transcript " + std::to_string(d) + " has " + std::to_string(U) + " labels, at most " +
             std::to_string(W2S_MAX_TRANSCRIPT) + " are supported";
    if (U > 0 && !labels) return "labels missing";
    for (int u = offsets[d]; u < offsets[d + 1]; ++u) {
      if (labels[u] < 0 || labels[u] >= V)
        return "transcript " + std::to_string(d) + ": label " + std::to_string(labels[u]) + " outside the vocabulary [0, " +
               std::to_string(V) + ")";
      if (labels[u] == blank) return "transcript " + std::to_string(d) + ": label equal to the blank " + std::to_string(blank);
    }
    (*need)[(size_t)d] = ctc_frames_needed(labels + offsets[d], U);
  }
  return "";
}

// w2s_set_references / w2s_debug_errors / w2s_error_tables: the argument checks (host only) and the tables of errors.cuh
std::string error_tables(const int32_t* labels, const int32_t* offsets, int D, int V, int blank, int unit, int delim,
                         std::vector<int32_t>* tab) {
  std::vector<int> need;
  std::string e = validate_transcripts(labels, offsets, D, blank, V, &need);
  if (!e.empty()) return e;
  if (unit != W2S_ERR_LABELS && unit != W2S_ERR_WORDS)
    return "unit " + std::to_string(unit) + " is neither W2S_ERR_LABELS (0) nor W2S_ERR_WORDS (1)";
  if (unit == W2S_ERR_WORDS && (delim < 0 || delim >= V || delim == blank))
    return "delimiter " + std::to_string(delim) + " outside the vocabulary [0, " + std::to_string(V) + ") or equal to the blank";
  const int total = offsets[D];
  tab->assign((size_t)ERR_HDR * D, 0);
  const int lab0 = (int)tab->size();
  tab->insert(tab->end(), labels, labels + total);
  for (int d = 0; d < D; ++d) {
    int* hdr = nullptr;
    std::vector<int> sym;               // symbol of every unit: its label, or the index of its distinct word
    std::vector<int32_t> rec;           // (start, length) of every distinct word
    int maxw = 0;
    if (unit == W2S_ERR_LABELS) {
      sym.assign(labels + offsets[d], labels + offsets[d + 1]);
    } else {
      std::map<std::vector<int32_t>, int> ids;
      for (int u = offsets[d]; u < offsets[d + 1];) {
        if (labels[u] == delim) {
          ++u;
          continue;
        }
        int v = u;
        while (v < offsets[d + 1] && labels[v] != delim) ++v;
        auto it = ids.emplace(std::vector<int32_t>(labels + u, labels + v), (int)ids.size()).first;
        if (it->second == (int)rec.size() / 2) {
          rec.push_back(lab0 + u);
          rec.push_back(v - u);
        }
        sym.push_back(it->second);
        maxw = std::max(maxw, v - u);
        u = v;
      }
    }
    const int rows = unit == W2S_ERR_LABELS ? V : (int)rec.size() / 2;
    const int dw = (int)tab->size();
    tab->insert(tab->end(), rec.begin(), rec.end());
    const int peq = (int)tab->size();
    tab->resize(tab->size() + (size_t)rows * ERR_LANES, 0);
    for (size_t i = 0; i < sym.size(); ++i)
      (*tab)[peq + (size_t)sym[i] * ERR_LANES + i / 32] |= (int32_t)(1u << (i % 32));
    hdr = tab->data() + (size_t)ERR_HDR * d;
    hdr[0] = (int)sym.size(); hdr[1] = peq; hdr[2] = dw; hdr[3] = (int)rec.size() / 2; hdr[4] = maxw;
  }
  return "";
}

#include "grad_plan.cuh"

int fail(w2s_handle* h, const std::string& e) {
  h->err = e;
  return 1;
}

// SM count of the current device (the debug entry points have no handle)
int debug_num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  return sms;
}

// The operand layout of the model paths (PlanBuilder): q | k | v at 0 / H / 2H of a 3H row, or the relative-position
// conformer's q+u | q+v | k | v at 0 / H / 2H / 3H of a 4H row.
AttnParams debug_attn_params(const void* qkv, const void* pos_proj, int B, int T, int heads, float scale) {
  AttnParams ap{};
  const int H = heads * 64, nq = pos_proj ? 2 : 1;
  ap.qkv = (const bf16*)qkv; ap.B = B; ap.T = T; ap.Tp = (T + 63) / 64 * 64; ap.H = H; ap.heads = heads; ap.hd = 64;
  ap.ld = (nq + 2) * H; ap.q_off = 0; ap.qv_off = pos_proj ? H : 0; ap.k_off = nq * H; ap.v_off = (nq + 1) * H;
  ap.scale = scale;
  ap.pos_proj = (const bf16*)pos_proj;
  return ap;
}

// Device buffers of one w2s_debug_* call.  release() waits for the work queued on s, frees them all and returns the
// stream's error, or "".
struct CallScratch {
  cudaStream_t s;
  std::vector<void*> ptrs;
  template <typename T>
  bool alloc(T** p, size_t count) {
    if (cudaMalloc((void**)p, sizeof(T) * count) != cudaSuccess) {
      *p = nullptr;
      return false;
    }
    ptrs.push_back(*p);
    return true;
  }
  std::string release() {
    const cudaError_t se = cudaStreamSynchronize(s);
    for (void* p : ptrs) cudaFree(p);
    ptrs.clear();
    return se == cudaSuccess ? "" : cudaGetErrorString(se);
  }
};

// head_reduce_kernel on caller logits [n, T, ldl] for the w2s_debug_* entries: d, whose tables are already on the
// device, travels in an argument block of the call's scratch
std::string debug_head_reduce(const float* logits, int n, int T, int V, int ldl, const DynArgs& d, CallScratch& sc) {
  DynArgs* dyn = nullptr;
  if (!sc.alloc(&dyn, 1)) return "out of device memory";
  if (cudaMemcpyAsync(dyn, &d, sizeof(DynArgs), cudaMemcpyHostToDevice, sc.s) != cudaSuccess) return "copy failed";
  HeadParams hp{};
  hp.n = n; hp.T = T; hp.V = V; hp.ldl = ldl; hp.dyn = dyn;
  return launch_head_reduce(logits, hp, sc.s);
}

// result of a w2s_debug_* entry: its error goes where w2s_last_error(NULL) reads it
int debug_result(const std::string& e) {
  g_create_error = e;
  return e.empty() ? 0 : 1;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int w2s_create(const w2s_config* cfg, const char* const* names, const float* const* ptrs, const int64_t* numels,
               int n_weights, int device, w2s_handle** out) {
  g_create_error.clear();
  if (!cfg || !out) {
    g_create_error = "null argument";
    return 1;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    g_create_error = "no CUDA device: this library has no CPU path";
    return 1;
  }
  if (cudaSetDevice(device) != cudaSuccess) {
    g_create_error = "cudaSetDevice failed";
    return 1;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) {
    g_create_error = std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                     std::to_string(prop.minor) + "; this library is built for sm_100a only";
    return 1;
  }
  std::unique_ptr<w2s_handle> h(new w2s_handle());
  h->cfg = *cfg;
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->auto_batch = h->cfg.max_batch <= 0;
  if (h->auto_batch) h->cfg.max_batch = 64;
  // the validation modes launch eagerly
  h->use_graphs = (cfg->flags & (W2S_FLAG_NO_GRAPH | W2S_FLAG_VALIDATE_GEMM | W2S_FLAG_VALIDATE_ATTN)) == 0;
  if (cudaMalloc((void**)&h->dyn_dev, sizeof(DynArgs)) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_create_error = "out of device memory";
    return 1;
  }
  if (cfg->num_conv_layers < 1 || cfg->num_conv_layers > W2S_MAX_CONV_LAYERS) {
    g_create_error = "num_conv_layers out of range";
    return 1;
  }
  if (cfg->kind < 0 || cfg->kind > 2) {
    g_create_error = "unknown model kind " + std::to_string(cfg->kind) +
                     " (0 = Wav2Vec2ForCTC, 1 = Wav2Vec2ConformerForCTC, 2 = WavLMForCTC)";
    return 1;
  }
  if (cfg->kind == 2 && cfg->hidden_size != 64 * cfg->num_attention_heads) {
    g_create_error = "WavLMForCTC: head_dim must be 64";
    return 1;
  }
  if (cfg->hidden_size % cfg->num_attention_heads) {
    g_create_error = "hidden_size must be divisible by num_attention_heads";
    return 1;
  }
  std::string e = gemm_init();
  if (e.empty()) e = attention_rel_init();
  if (e.empty()) e = posconv_init();
  if (e.empty()) e = attention_fa_init();
  if (e.empty()) e = attention_bwd_init();
  if (e.empty()) {
    WeightTable wt;
    wt.prefix = cfg->kind == 1 ? "wav2vec2_conformer." : cfg->kind == 2 ? "wavlm." : "wav2vec2.";
    for (int i = 0; i < n_weights; ++i) wt.t[names[i]] = {ptrs[i], numels[i]};
    e = load_weights(h.get(), wt);
  }
  if (!e.empty()) {
    g_create_error = e;
    return 1;
  }
  *out = h.release();
  return 0;
}

void w2s_destroy(w2s_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  delete h;
}

const char* w2s_last_error(const w2s_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t w2s_num_frames(const w2s_handle* h, int64_t num_samples) { return num_frames(h->cfg, num_samples, nullptr); }

int w2s_set_clip(w2s_handle* h, const float* x_dev, int64_t L, const int32_t* seg_bounds_host, int M, float baseline,
                 void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (L <= 0 || M <= 0 || M > 2048) return fail(h, "set_clip: need L > 0 and 1 <= M <= 2048");
  if (seg_bounds_host[0] != 0 || seg_bounds_host[M] != L) return fail(h, "set_clip: seg_bounds must span [0, L]");
  std::vector<uint16_t> seg((size_t)L);
  for (int m = 0; m < M; ++m) {
    if (seg_bounds_host[m + 1] < seg_bounds_host[m]) return fail(h, "set_clip: seg_bounds must be ascending");
    for (int64_t i = seg_bounds_host[m]; i < seg_bounds_host[m + 1]; ++i) seg[(size_t)i] = (uint16_t)m;
  }
  std::string e = ensure_workspace(h, L);
  if (!e.empty()) return fail(h, e);
  e = grow(&h->clip, &h->clip_cap, L + 16, 0, s);
  if (e.empty()) e = grow(&h->seg_id, &h->seg_id_cap, L + 16, 0, s);
  if (!e.empty()) return fail(h, "set_clip: " + e);
  if (cudaMemcpyAsync(h->clip, x_dev, sizeof(float) * L, cudaMemcpyDeviceToDevice, s) != cudaSuccess ||
      cudaMemcpyAsync(h->seg_id, seg.data(), sizeof(uint16_t) * L, cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return fail(h, std::string("set_clip: copy failed: ") + cudaGetErrorString(cudaGetLastError()));
  h->L = L;
  h->M = M;
  h->zwords = (M + 31) / 32;
  h->baseline = baseline;
  h->seg_bounds.assign(seg_bounds_host, seg_bounds_host + M + 1);
  e = upload_skip_table(h, s);
  if (!e.empty()) return fail(h, "set_clip: " + e);
  return 0;
}

int w2s_set_background(w2s_handle* h, const float* bg_dev, int64_t B, int64_t L, int64_t ld, const double* weights_host,
                       void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (B == 0) {
    h->bg_B = 0;
    h->bg_L = 0;
    return 0;
  }
  if (B < 0 || B > W2S_MAX_BACKGROUND)
    return fail(h, "set_background: B = " + std::to_string(B) + " rows; need 1 <= B <= " +
                       std::to_string(W2S_MAX_BACKGROUND) + " (B = 0 clears the background)");
  if (h->bands_F > 0)
    return fail(h, "set_background: frequency bands are set (w2s_set_bands); a background cannot be combined with them "
                   "(clear the bands with F = 0 first)");
  if (h->L <= 0) return fail(h, "set_background: no clip set (w2s_set_clip)");
  if (L != h->L)
    return fail(h, "set_background: background rows have " + std::to_string(L) + " samples, the clip has " +
                       std::to_string(h->L));
  if (ld < L) return fail(h, "set_background: row stride smaller than the row length");
  if (!bg_dev || !weights_host) return fail(h, "set_background: null buffer");
  double sum = 0.0;
  for (int64_t b = 0; b < B; ++b) {
    const double w = weights_host[b];
    if (!std::isfinite(w) || w < 0.0)
      return fail(h, "set_background: weight " + std::to_string(b) + " is " + std::to_string(w) +
                         "; weights must be finite and >= 0");
    sum += w;
  }
  if (!(sum > 0.0) || !std::isfinite(sum)) return fail(h, "set_background: the weights sum to zero");
  // evaluations in flight on the stream still read the old rows and weights
  if (cudaStreamSynchronize(s) != cudaSuccess) return fail(h, "set_background: stream error");
  h->bg_B = 0;   // a failed allocation or copy below leaves no background set, not a dangling one
  const std::string e = grow(&h->bg, &h->bg_cap, B * L, 0, s);
  if (!e.empty()) return fail(h, "set_background: " + e);
  if (!h->bg_w && cudaMalloc((void**)&h->bg_w, sizeof(float) * W2S_MAX_BACKGROUND) != cudaSuccess)
    return fail(h, "set_background: out of device memory");
  h->bg_w_host.resize((size_t)B);
  for (int64_t b = 0; b < B; ++b) h->bg_w_host[(size_t)b] = (float)(weights_host[b] / sum);
  if (cudaMemcpy2DAsync(h->bg, sizeof(float) * L, bg_dev, sizeof(float) * ld, sizeof(float) * L, (size_t)B,
                        cudaMemcpyDeviceToDevice, s) != cudaSuccess ||
      cudaMemcpyAsync(h->bg_w, h->bg_w_host.data(), sizeof(float) * B, cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return fail(h, std::string("set_background: copy failed: ") + cudaGetErrorString(cudaGetLastError()));
  h->bg_B = (int)B;
  h->bg_L = L;
  return 0;
}

int w2s_set_bands(w2s_handle* h, const float* comp_dev, int64_t F, int64_t L, int64_t ld, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (F == 0) {
    h->bands_F = 0;
    h->bands_L = 0;
    return 0;
  }
  if (F < 0 || F > W2S_MAX_BANDS)
    return fail(h, "set_bands: F = " + std::to_string(F) + " bands; need 1 <= F <= " + std::to_string(W2S_MAX_BANDS) +
                       " (F = 0 clears the bands)");
  if (!comp_dev) return fail(h, "set_bands: null buffer");
  if (h->bg_B > 0)
    return fail(h, "set_bands: a background is set (w2s_set_background); bands cannot be combined with it "
                   "(clear the background with B = 0 first)");
  if (h->L <= 0) return fail(h, "set_bands: no clip set (w2s_set_clip)");
  if (L != h->L)
    return fail(h, "set_bands: band components have " + std::to_string(L) + " samples, the clip has " + std::to_string(h->L));
  if (ld < L) return fail(h, "set_bands: row stride smaller than the row length");
  if ((long long)h->M * F > 2048)
    return fail(h, "set_bands: " + std::to_string(h->M) + " segments x " + std::to_string(F) + " bands = " +
                       std::to_string((long long)h->M * F) + " cells; at most 2048 are supported");
  // evaluations in flight on the stream still read the old components
  if (cudaStreamSynchronize(s) != cudaSuccess) return fail(h, "set_bands: stream error");
  h->bands_F = 0;   // a failed allocation or copy below leaves no bands set, not dangling ones
  const std::string e = grow(&h->bands, &h->bands_cap, F * L, 0, s);
  if (!e.empty()) return fail(h, "set_bands: " + e);
  if (cudaMemcpy2DAsync(h->bands, sizeof(float) * L, comp_dev, sizeof(float) * ld, sizeof(float) * L, (size_t)F,
                        cudaMemcpyDeviceToDevice, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return fail(h, std::string("set_bands: copy failed: ") + cudaGetErrorString(cudaGetLastError()));
  h->bands_F = (int)F;
  h->bands_L = L;
  return 0;
}

int w2s_set_targets(w2s_handle* h, const int32_t* frame_idx_host, const int32_t* token_idx_host, int D, int mode,
                    void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (mode < W2S_OUT_MAX || mode > W2S_OUT_LOGITS) return fail(h, "set_targets: unknown mode");
  if (mode == W2S_OUT_LOGIT || mode == W2S_OUT_LOGPROB) {
    if (D <= 0 || !frame_idx_host || !token_idx_host) return fail(h, "set_targets: need D > 0 (frame, token) pairs");
    for (int d = 0; d < D; ++d)
      if (token_idx_host[d] < 0 || token_idx_host[d] >= h->cfg.vocab_size || frame_idx_host[d] < 0)
        return fail(h, "set_targets: target out of range");
    const std::string e = grow(&h->targets, &h->targets_cap, 2LL * D, 2 * 1024, s);
    if (!e.empty()) return fail(h, "set_targets: " + e);
    // ordered on the caller's stream behind any evaluation still running with the previous targets; the host arrays
    // are staged in the handle so the caller's buffers may be released when this returns
    h->targets_host.assign(frame_idx_host, frame_idx_host + D);
    h->targets_host.insert(h->targets_host.end(), token_idx_host, token_idx_host + D);
    if (cudaMemcpyAsync(h->targets, h->targets_host.data(), sizeof(int) * 2 * D, cudaMemcpyHostToDevice, s) != cudaSuccess)
      return fail(h, "set_targets: copy failed");
    h->D = D;
    h->max_frame = 0;
    for (int d = 0; d < D; ++d) h->max_frame = frame_idx_host[d] > h->max_frame ? frame_idx_host[d] : h->max_frame;
  } else {
    h->D = 0;
  }
  h->mode = mode;
  return 0;
}

int w2s_set_transcripts(w2s_handle* h, const int32_t* labels_host, const int32_t* offsets_host, int D, int blank,
                        void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<int> need;
  const std::string e = validate_transcripts(labels_host, offsets_host, D, blank, h->cfg.vocab_size, &need);
  if (!e.empty()) return fail(h, "set_transcripts: " + e);
  const int total = offsets_host[D];
  const int label_slots = total > 0 ? total : 1;   // all transcripts empty: the kernels still take a valid pointer
  h->ctc_D = 0;   // a failed allocation or copy below leaves no transcripts set, not dangling ones
  std::string ge = grow(&h->ctc_offsets, &h->ctc_offsets_cap, D + 1, 64, s);
  if (ge.empty()) ge = grow(&h->ctc_labels, &h->ctc_labels_cap, label_slots, 1024, s);
  if (!ge.empty()) return fail(h, "set_transcripts: " + ge);
  // ordered on the caller's stream, staged in the handle (as w2s_set_targets)
  h->ctc_host.assign(offsets_host, offsets_host + D + 1);
  h->ctc_host.insert(h->ctc_host.end(), labels_host, labels_host + total);
  if (cudaMemcpyAsync(h->ctc_offsets, h->ctc_host.data(), sizeof(int) * (D + 1), cudaMemcpyHostToDevice, s) != cudaSuccess ||
      (total > 0 && cudaMemcpyAsync(h->ctc_labels, h->ctc_host.data() + D + 1, sizeof(int) * total, cudaMemcpyHostToDevice,
                                    s) != cudaSuccess))
    return fail(h, "set_transcripts: copy failed");
  h->ctc_D = D;
  h->ctc_blank = blank;
  h->ctc_need = need;
  h->ctc_smax = 1;
  for (int d = 0; d < D; ++d) {
    const int S = 2 * (offsets_host[d + 1] - offsets_host[d]) + 1;
    h->ctc_smax = S > h->ctc_smax ? S : h->ctc_smax;
  }
  h->mode = W2S_OUT_CTC;
  return 0;
}

int w2s_set_references(w2s_handle* h, const int32_t* labels_host, const int32_t* offsets_host, int D, int blank, int unit,
                       int delimiter, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<int32_t> tab;
  const std::string e = error_tables(labels_host, offsets_host, D, h->cfg.vocab_size, blank, unit, delimiter, &tab);
  if (!e.empty()) return fail(h, "set_references: " + e);
  h->err_D = 0;   // a failed allocation or copy below leaves no references set, not dangling ones
  const std::string ge = grow(&h->err_tab, &h->err_tab_cap, (long long)tab.size(), 4096, s);
  if (!ge.empty()) return fail(h, "set_references: " + ge);
  // ordered on the caller's stream, staged in the handle (as w2s_set_targets)
  h->err_host = std::move(tab);
  if (cudaMemcpyAsync(h->err_tab, h->err_host.data(), sizeof(int) * h->err_host.size(), cudaMemcpyHostToDevice, s) !=
      cudaSuccess)
    return fail(h, "set_references: copy failed");
  h->err_D = D;
  h->err_blank = blank;
  h->err_unit = unit;
  h->err_delim = delimiter;
  h->mode = W2S_OUT_ERRORS;
  return 0;
}

int64_t w2s_error_tables(const int32_t* labels_host, const int32_t* offsets_host, int D, int V, int blank, int unit,
                         int delimiter, int32_t* out, int64_t cap) {
  std::vector<int32_t> tab;
  if (V < 1 || !error_tables(labels_host, offsets_host, D, V, blank, unit, delimiter, &tab).empty()) return -1;
  if (out && (int64_t)tab.size() <= cap) std::copy(tab.begin(), tab.end(), out);
  return (int64_t)tab.size();
}

int64_t w2s_out_width(const w2s_handle* h, int64_t num_samples) { return out_width(h, num_samples); }

int w2s_eval(w2s_handle* h, const uint32_t* z_bits_dev, int64_t K, float* out_dev, void* stream) {
  if (h->L <= 0) return fail(h, "eval: no clip set (w2s_set_clip)");
  if (K == 0) return 0;   // empty coalition matrix: nothing to evaluate
  if (K < 0 || !z_bits_dev || !out_dev) return fail(h, "eval: null buffer");
  if (h->bg_B > 0 && h->bg_L != h->L)
    return fail(h, "eval: the background rows have " + std::to_string(h->bg_L) + " samples, the clip has " +
                       std::to_string(h->L) + " (w2s_set_background again, or clear it with B = 0)");
  std::string e = check_bands(h);
  if (!e.empty()) return fail(h, "eval: " + e);
  // the workspace (and with it T') follows the clip of THIS call: w2s_eval_waveforms may have left it at another length
  e = ensure_workspace(h, h->L);
  if (e.empty()) e = check_targets(h);
  if (e.empty()) e = run_batches(h, z_bits_dev, nullptr, 0, K, out_dev, (cudaStream_t)stream);
  return e.empty() ? 0 : fail(h, "eval: " + e);
}

int w2s_eval_waveforms(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld, float* out_dev,
                       void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !x_dev || !out_dev) return fail(h, "eval_waveforms: null buffer");
  if (ld < L) return fail(h, "eval_waveforms: row stride smaller than the row length");
  std::string e = ensure_workspace(h, L);
  if (e.empty()) e = check_targets(h);
  if (e.empty()) e = run_batches(h, nullptr, x_dev, ld, n, out_dev, (cudaStream_t)stream);
  return e.empty() ? 0 : fail(h, "eval_waveforms: " + e);
}

int w2s_grad_waveforms(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld, const int32_t* frames_host,
                       float* grad_dev, float* out_dev, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !x_dev || !frames_host || !grad_dev) return fail(h, "grad_waveforms: null buffer");
  if (ld < L) return fail(h, "grad_waveforms: row stride smaller than the row length");
  std::string e = run_grad(h, x_dev, ld, L, n, frames_host, nullptr, grad_dev, out_dev, (cudaStream_t)stream);
  return e.empty() ? 0 : fail(h, "grad_waveforms: " + e);
}

int w2s_grad_transcripts(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld, const int32_t* which_host,
                         float* grad_dev, float* out_dev, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !x_dev || !which_host || !grad_dev) return fail(h, "grad_transcripts: null buffer");
  if (ld < L) return fail(h, "grad_transcripts: row stride smaller than the row length");
  std::string e = grad_supported(h);
  if (e.empty() && h->grad_rules) e = "DeepLIFT rules (w2s_grad_rules) are not built for transcripts: switch them off";
  const int64_t T = num_frames(h->cfg, L, nullptr);
  if (e.empty() && T <= 0) e = "clip shorter than the conv receptive field";
  if (e.empty()) e = h->ctc_D > 0 ? "" : "no transcripts set (w2s_set_transcripts)";
  for (int64_t i = 0; e.empty() && i < n; ++i)
    if (which_host[i] < 0 || which_host[i] >= h->ctc_D)
      e = "transcript index " + std::to_string(which_host[i]) + " outside the " + std::to_string(h->ctc_D) + " set";
  if (e.empty()) e = check_transcripts(h, T);
  if (e.empty()) {
    h->grad_ctc = true;
    e = run_grad(h, x_dev, ld, L, n, which_host, nullptr, grad_dev, out_dev, (cudaStream_t)stream);
    h->grad_ctc = false;
  }
  return e.empty() ? 0 : fail(h, "grad_transcripts: " + e);
}

int w2s_vjp_waveforms(w2s_handle* h, const float* x_dev, int64_t n, int64_t L, int64_t ld, const float* gout_dev,
                      float* grad_dev, float* out_dev, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !x_dev || !gout_dev || !grad_dev) return fail(h, "vjp_waveforms: null buffer");
  if (ld < L) return fail(h, "vjp_waveforms: row stride smaller than the row length");
  std::string e = run_grad(h, x_dev, ld, L, n, nullptr, gout_dev, grad_dev, out_dev, (cudaStream_t)stream);
  return e.empty() ? 0 : fail(h, "vjp_waveforms: " + e);
}

int w2s_grad_debug(w2s_handle* h, int on) {
  const bool snaps = (on & 1) != 0, simt = (on & 2) != 0, unfused = (on & 4) != 0;
  if (simt != h->grad_attn_simt || unfused != h->grad_attn_unfused) h->grad_L = -1;   // rebuild the plans
  h->grad_debug = snaps;
  h->grad_attn_simt = simt;
  h->grad_attn_unfused = unfused;
  return 0;
}

int w2s_grad_rules(w2s_handle* h, int rules) {
  if (!h) return 1;
  if (rules & ~3) return fail(h, "grad_rules: unknown rule bits");
  h->grad_rules = rules;
  return 0;
}

int64_t w2s_grad_peek(w2s_handle* h, const char* name, void* dst_dev, int64_t max_bytes, void* stream) {
  for (auto& kv : h->grad_plans) {
    auto it = kv.second->peek.find(name);
    if (it == kv.second->peek.end()) continue;
    const int64_t bytes = (int64_t)it->second.second;
    if (bytes > max_bytes) return -bytes;
    if (cudaMemcpyAsync(dst_dev, it->second.first, (size_t)bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream) != cudaSuccess)
      return 0;
    return bytes;
  }
  return 0;
}

int w2s_mask(w2s_handle* h, const uint32_t* z_bits_dev, int64_t K, float* out_dev, void* stream) {
  if (h->L <= 0) return fail(h, "mask: no clip set (w2s_set_clip)");
  if (h->bg_B > 0 && h->bg_L != h->L)
    return fail(h, "mask: the background rows have " + std::to_string(h->bg_L) + " samples, the clip has " +
                       std::to_string(h->L) + " (w2s_set_background again, or clear it with B = 0)");
  std::string e = check_bands(h);
  if (!e.empty()) return fail(h, "mask: " + e);
  if (h->bands_F > 0)
    e = launch_mask_bands(h->seg_id, z_bits_dev, (h->M * h->bands_F + 31) / 32, K, h->L, h->bands, h->bands_F, h->bands_L,
                          out_dev, h->L, (cudaStream_t)stream);
  else
    e = h->bg_B > 0 ? launch_mask_bg(h->clip, h->seg_id, z_bits_dev, h->zwords, K, h->L, h->bg, h->bg_B, h->bg_L, out_dev,
                                     h->L, (cudaStream_t)stream)
                    : launch_mask(h->clip, h->seg_id, z_bits_dev, h->zwords, K, h->L, h->baseline, out_dev, h->L,
                                  (cudaStream_t)stream);
  return e.empty() ? 0 : fail(h, e);
}

int w2s_wls(w2s_handle* h, const uint32_t* z_bits_dev, const double* w_dev, const float* y_dev, int64_t K, int M,
            int D, const double* fx_dev, const double* fnull_dev, double* phi_dev, int32_t* status_dev, void* stream) {
  const long long need = 2 * ((long long)(M - 1) * (M - 1) + (long long)(M - 1) * D);
  std::string e = grow(&h->wls_work, &h->wls_cap, need, 0, (cudaStream_t)stream);
  if (!e.empty()) return fail(h, "wls: " + e);
  e = launch_wls(z_bits_dev, (M + 31) / 32, w_dev, y_dev, K, M, D, fx_dev, fnull_dev, phi_dev, status_dev, h->wls_work,
                 (cudaStream_t)stream);
  return e.empty() ? 0 : fail(h, e);
}

int w2s_debug_gemm(int use_tcgen05, const void* a_bf16, const void* w_bf16, const float* bias, const void* residual,
                   int res_fp32, float alpha, void* out, int M, int N, int K, int act, int out_fp32, void* stream) {
  std::string e = gemm_init();
  if (e.empty()) {
    GemmProblem p = PlanBuilder::plain((const bf16*)a_bf16, M, K, (const bf16*)w_bf16, N);
    p.epi.bias = bias; p.epi.act = act; p.epi.out = out; p.epi.out_fp32 = out_fp32;
    p.epi.residual = residual; p.epi.res_fp32 = res_fp32; p.epi.alpha = alpha;
    GemmLaunch gl;
    e = gemm_prepare(p, debug_num_sms(), &gl);
    if (e.empty()) e = use_tcgen05 ? gemm_launch_tc(gl, (cudaStream_t)stream) : gemm_launch_simt(gl, (cudaStream_t)stream);
  }
  return debug_result(e);
}

int w2s_debug_attention(int use_tcgen05, const void* qkv, const void* pos_proj, int B, int T, int heads, float scale,
                        void* ctx, float* lse, void* stream) {
  const cudaStream_t s = (cudaStream_t)stream;
  AttnParams ap = debug_attn_params(qkv, pos_proj, B, T, heads, scale);
  ap.ctx = (bf16*)ctx;
  ap.lse = lse;
  std::string e;
  if (B <= 0 || T <= 0 || heads <= 0 || !qkv || !ctx) {
    e = "debug_attention: need B, T', heads >= 1 and qkv / ctx buffers";
  } else if (lse && (pos_proj || !use_tcgen05)) {
    e = "debug_attention: only the tcgen05 kernel without relative positions writes the log-sum-exp";
  } else if (!(e = gemm_init()).empty()) {
    // the tensor-map encoder the tcgen05 plans need is not available
  } else if (!use_tcgen05) {
    e = launch_attention_simt(ap, s);
  } else if (pos_proj) {
    AttnRelPlan* rp = nullptr;
    e = attention_rel_init();
    if (e.empty()) e = attention_rel_prepare(ap, &rp);
    if (e.empty()) e = attention_rel_launch(rp, s);
    if (rp) attention_rel_free(rp);   // the tensor maps travel in the kernel parameters: the plan may go after the launch
  } else {
    AttnFaPlan* fp = nullptr;
    e = attention_fa_init();
    if (e.empty()) e = attention_fa_prepare(ap, debug_num_sms(), &fp);
    if (e.empty()) e = attention_fa_launch(fp, s);
    if (fp) attention_fa_free(fp);
  }
  return debug_result(e);
}

int w2s_debug_attention_bias(int use_tcgen05, const void* qkv, const float* rel_bias, const float* gate, int B, int T,
                             int heads, float scale, void* ctx, float* lse, void* stream) {
  const cudaStream_t s = (cudaStream_t)stream;
  AttnParams ap = debug_attn_params(qkv, nullptr, B, T, heads, scale);
  ap.ctx = (bf16*)ctx;
  ap.gate = gate;
  std::string e;
  CallScratch sc{s};
  float* table = nullptr;
  if (B <= 0 || T <= 0 || heads <= 0 || !qkv || !ctx || !rel_bias || !gate) {
    e = "debug_attention_bias: need B, T', heads >= 1 and qkv / rel_bias / gate / ctx buffers";
  } else if (lse) {
    e = "debug_attention_bias: the relative-position bias variant writes no log-sum-exp (lse must be NULL)";
  } else if (!sc.alloc(&table, (size_t)heads * rel_bias_ld(T))) {
    e = "debug_attention_bias: out of device memory";
  } else if (!(e = launch_rel_bias_table(rel_bias, nullptr, T, heads, table, s)).empty()) {
  } else if (!(e = gemm_init()).empty()) {
  } else {
    ap.rel_bias = table;
    if (!use_tcgen05) {
      e = launch_attention_simt(ap, s);
    } else {
      AttnFaPlan* fp = nullptr;
      e = attention_fa_init();
      if (e.empty()) e = attention_fa_prepare(ap, debug_num_sms(), &fp);
      if (e.empty()) e = attention_fa_launch(fp, s);
      if (fp) attention_fa_free(fp);
    }
  }
  const std::string se = sc.release();
  if (e.empty() && !se.empty()) e = "debug_attention_bias: " + se;
  return debug_result(e);
}

int w2s_debug_attention_bwd(int use_tcgen05, const void* qkv, const void* ctx, const void* dctx, const float* lse, int B,
                            int T, int heads, float scale, void* dqkv, void* stream) {
  const cudaStream_t s = (cudaStream_t)stream;
  const AttnParams ap = debug_attn_params(qkv, nullptr, B, T, heads, scale);
  const long long rows = (long long)B * T;
  std::string e;
  CallScratch sc{s};
  float *delta = nullptr, *dq = nullptr, *stats = nullptr;
  auto dalloc = [&](float** p, size_t n) {
    if (e.empty() && !sc.alloc(p, n)) e = "debug_attention_bwd: out of device memory";
  };
  if (B <= 0 || T <= 0 || heads <= 0 || !qkv || !dctx || !dqkv) {
    e = "debug_attention_bwd: need B, T', heads >= 1 and qkv / dctx / dqkv buffers";
  } else if (use_tcgen05) {
    if (!ctx || !lse) e = "debug_attention_bwd: the fused kernel needs the forward's ctx and log-sum-exp";
    if (e.empty()) e = gemm_init();   // the tensor-map encoder of the plan
    dalloc(&delta, (size_t)rows * heads);
    dalloc(&dq, (size_t)rows * ap.H);
    AttnBwdPlan* bp = nullptr;
    if (e.empty()) e = attention_bwd_init();
    if (e.empty()) e = attention_bwd_prepare(ap, (const bf16*)dctx, lse, delta, dq, (bf16*)dqkv, debug_num_sms(), &bp);
    if (e.empty()) e = attention_bwd_launch(bp, (const bf16*)dctx, (const bf16*)ctx, ap.q_off, s);
    if (bp) attention_bwd_free(bp);
  } else {
    dalloc(&stats, (size_t)rows * heads * 3);
    if (e.empty()) e = launch_attn_bwd(ap.qkv, (const bf16*)dctx, B, T, ap.H, heads, scale, (bf16*)dqkv, stats, s);
  }
  const std::string se = sc.release();
  if (e.empty() && !se.empty()) e = "debug_attention_bwd: " + se;
  return debug_result(e);
}

int w2s_debug_ctc(const float* logits, int n, int T, int V, int ldl, const int32_t* labels_host, const int32_t* offsets_host,
                  int D, int blank, const int32_t* which_host, float* out_dev, float* dlogits_dev, void* stream) {
  const cudaStream_t s = (cudaStream_t)stream;
  std::vector<int> need;
  std::string e;
  if (n <= 0 || T <= 0 || V <= 0 || V > 128 || ldl < V || !logits || !out_dev)
    e = "debug_ctc: need n, T >= 1, 1 <= V <= 128, ldl >= V and logits / out buffers";
  if (e.empty()) e = validate_transcripts(labels_host, offsets_host, D, blank, V, &need);
  if (!e.empty() && e.compare(0, 10, "debug_ctc:") != 0) e = "debug_ctc: " + e;
  for (int d = 0; e.empty() && d < D; ++d)
    if (need[d] > T) e = "debug_ctc: transcript " + std::to_string(d) + " needs " + std::to_string(need[d]) + " frames, T = " + std::to_string(T);
  for (int r = 0; e.empty() && dlogits_dev && r < n; ++r)
    if (!which_host || which_host[r] < 0 || which_host[r] >= D) e = "debug_ctc: which[r] must index a transcript";
  if (e.empty() && n * (long long)D > 0) {
    const int total = offsets_host[D];
    int smax = 1;
    for (int d = 0; d < D; ++d) smax = std::max(smax, 2 * (offsets_host[d + 1] - offsets_host[d]) + 1);
    CallScratch sc{s};
    int *lab = nullptr, *off = nullptr, *wh = nullptr;
    float *alpha = nullptr, *lse = nullptr, *val = nullptr;
    if (!sc.alloc(&lab, total + 1) || !sc.alloc(&off, D + 1) || !sc.alloc(&wh, n))
      e = "out of device memory";
    else if (cudaMemcpyAsync(off, offsets_host, sizeof(int) * (D + 1), cudaMemcpyHostToDevice, s) != cudaSuccess ||
             (total && cudaMemcpyAsync(lab, labels_host, sizeof(int) * total, cudaMemcpyHostToDevice, s) != cudaSuccess))
      e = "copy failed";
    if (e.empty()) {
      DynArgs d{};
      d.out = out_dev; d.mode = W2S_OUT_CTC; d.D = D; d.ctc_labels = lab; d.ctc_offsets = off; d.blank = blank;
      e = debug_head_reduce(logits, n, T, V, ldl, d, sc);
    }
    if (e.empty() && dlogits_dev) {
      if (!sc.alloc(&alpha, (size_t)n * T * smax) || !sc.alloc(&lse, (size_t)n * T) || !sc.alloc(&val, n))
        e = "out of device memory";
      else if (cudaMemcpyAsync(wh, which_host, sizeof(int) * n, cudaMemcpyHostToDevice, s) != cudaSuccess)
        e = "copy failed";
      if (e.empty())
        e = launch_ctc_seed(logits, ldl, V, nullptr, n, T, 0, lab, off, wh, blank, smax, alpha, lse, dlogits_dev, V, nullptr,
                            val, s);
    }
    const std::string se = sc.release();
    if (e.empty()) e = se;
    if (!e.empty()) e = "debug_ctc: " + e;
  }
  return debug_result(e);
}

int w2s_debug_errors(const float* logits, int n, int T, int V, int ldl, const int32_t* labels_host,
                     const int32_t* offsets_host, int D, int blank, int unit, int delimiter, float* out_dev, void* stream) {
  const cudaStream_t s = (cudaStream_t)stream;
  std::vector<int32_t> tab;
  std::string e;
  if (n <= 0 || T <= 0 || V <= 0 || V > 128 || ldl < V || !logits || !out_dev)
    e = "need n, T >= 1, 1 <= V <= 128, ldl >= V and logits / out buffers";
  if (e.empty()) e = error_tables(labels_host, offsets_host, D, V, blank, unit, delimiter, &tab);
  if (e.empty()) {
    CallScratch sc{s};
    int* dtab = nullptr;
    if (!sc.alloc(&dtab, tab.size()))
      e = "out of device memory";
    else if (cudaMemcpyAsync(dtab, tab.data(), sizeof(int) * tab.size(), cudaMemcpyHostToDevice, s) != cudaSuccess)
      e = "copy failed";
    if (e.empty()) {
      DynArgs d{};
      d.out = out_dev; d.mode = W2S_OUT_ERRORS; d.D = D; d.blank = blank; d.err_tab = dtab; d.err_unit = unit; d.delim = delimiter;
      e = debug_head_reduce(logits, n, T, V, ldl, d, sc);
    }
    const std::string se = sc.release();
    if (e.empty()) e = se;
  }
  return debug_result(e.empty() ? e : "debug_errors: " + e);
}

int w2s_profile_enable(w2s_handle* h, int on) {
  cudaDeviceSynchronize();
  for (auto& r : h->prof) {
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  h->prof.clear();
  h->profiling = on != 0;
  return 0;
}

int64_t w2s_profile_read(w2s_handle* h, char* names, int64_t names_cap, double* ms, double* flops, double* bytes,
                         int64_t* counts, int64_t max_entries) {
  cudaDeviceSynchronize();
  // aggregate by launch class: strip the "L<i>." layer prefix
  std::vector<std::string> keys;
  std::vector<double> tms, tfl, tby;
  std::vector<int64_t> cnt;
  for (auto& r : h->prof) {
    std::string k = r.name;
    std::string pre;
    if (k.compare(0, 5, "grad.") == 0) {   // gradient path: "grad.L3.qkv" / "grad.B3.qkv_bwd" -> "grad.qkv" / "grad.qkv_bwd"
      pre = "grad.";
      k = k.substr(5);
    }
    if (k.size() > 1 && (k[0] == 'L' || k[0] == 'B') && isdigit((unsigned char)k[1])) k = k.substr(k.find('.') + 1);
    k = pre + k;
    size_t i = 0;
    for (; i < keys.size(); ++i)
      if (keys[i] == k) break;
    if (i == keys.size()) {
      keys.push_back(k);
      tms.push_back(0.0); tfl.push_back(0.0); tby.push_back(0.0); cnt.push_back(0);
    }
    float t = 0.f;
    cudaEventElapsedTime(&t, r.e0, r.e1);
    tms[i] += t; tfl[i] += r.flops; tby[i] += r.bytes; cnt[i] += 1;
  }
  std::string joined;
  int64_t n = 0;
  for (size_t i = 0; i < keys.size() && n < max_entries; ++i, ++n) {
    joined += keys[i] + "\n";
    ms[n] = tms[i]; flops[n] = tfl[i]; bytes[n] = tby[i]; counts[n] = cnt[i];
  }
  if ((int64_t)joined.size() + 1 > names_cap) return -1;
  memcpy(names, joined.c_str(), joined.size() + 1);
  return n;
}

int w2s_kernel_count(const w2s_handle* h, int64_t* launches_per_batch, int64_t* batch_tile) {
  if (batch_tile) *batch_tile = h->cfg.max_batch;
  int64_t n = 0;
  for (auto& kv : h->plans)
    if ((int64_t)kv.second->steps.size() > n) n = (int64_t)kv.second->steps.size();
  if (launches_per_batch) *launches_per_batch = n + 1;  // + the per-call argument kernel
  return 0;
}

int64_t w2s_launch_count(const w2s_handle* h) { return h->launches; }

double w2s_flops_per_forward(const w2s_handle* h, int64_t L) {
  const w2s_config& c = h->cfg;
  std::vector<int> Tl;
  const double T = (double)num_frames(c, L, &Tl);
  if (T <= 0) return 0.0;
  double f = 0.0;
  for (int l = 0; l < c.num_conv_layers; ++l)
    f += 2.0 * Tl[l] * c.conv_dim[l] * (l == 0 ? 1 : c.conv_dim[l - 1]) * c.conv_kernel[l];
  const double H = c.hidden_size, I = c.intermediate_size;
  f += 2.0 * T * c.conv_dim[c.num_conv_layers - 1] * H;
  if (c.kind != 1) f += 2.0 * T * H * (H / c.num_conv_pos_embedding_groups) * c.num_conv_pos_embeddings;
  double per_layer = 2.0 * T * H * 3 * H + 4.0 * T * T * H + 2.0 * T * H * H + 4.0 * T * H * I;
  if (c.kind == 2) per_layer += 2.0 * T * 8 * H;                    // WavLM gate
  if (c.kind == 1) {
    per_layer += 4.0 * T * H * I;                                   // second macaron FFN
    per_layer += 2.0 * T * H * 2 * H + 2.0 * T * H * c.conv_depthwise_kernel_size + 2.0 * T * H * H;  // conv module
    if (c.position_embeddings_type == 1) per_layer += 2.0 * (2 * T - 1) * H * H + 2.0 * T * (2 * T - 1) * H;
  }
  f += per_layer * c.num_hidden_layers;
  f += 2.0 * T * H * c.vocab_size;
  return f;
}

}  // extern "C"
