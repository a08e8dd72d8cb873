// Expected-gradients path (the reference's production explainer: shap.GradientExplainer over ModelWrapper,
// shap_calculation.py:125-162): forward pass with saved activations + backward pass to the waveform, for one batch tile.
// Included by api.cu inside its anonymous namespace (it needs w2s_handle / Step / PlanBuilder::plain).
//
// Scope: Wav2Vec2ForCTC -- both front ends (feat_extract_norm = "group" / "layer") and both encoder orders
// (post-LN: facebook/wav2vec2-base-960h, the model the reference runs, and wav2vec2-large-960h; stable-LN: the
// wav2vec2-large-lv60 family), GELU; and Wav2Vec2ConformerForCTC (macaron feed-forwards, relative-position or rotary
// attention, GLU / depthwise / BatchNorm convolution module; swish or GELU).  Only d(output)/d(input) is
// computed: no weight gradients.  Every dense backward contraction dX = dY W runs on the tcgen05 contraction kernels of
// the forward pass with pre-transposed weights; attention backward is one fused tcgen05 kernel (attention_bwd.cu; the
// relative-position conformer: seven batched contractions + row kernels); the normalisation / activation / conv-gather
// steps are CUDA-core kernels (grad.cu).  w2s_grad_rules switches the activation / GLU steps to the reference's DeepLIFT
// handler rules on paired [explained | reference] rows.
#pragma once

struct GradLayerBuf {
  bf16* qkv = nullptr;    // [rows, 3H]   saved q | k | v
  bf16* ctx = nullptr;    // [rows, H]    attention output (fused backward: D_i = dO_i . O_i)
  float* lse = nullptr;   // [n, heads, T] log-sum-exp of the scaled scores (fused backward)
  float* s1 = nullptr;    // [rows, H]    h + attention(h): input of layer_norm
  bf16* u = nullptr;      // [rows, I]    pre-activation of the feed-forward
  float* s2 = nullptr;    // [rows, H]    h1 + ffn(h1): input of final_layer_norm
};

// conformer layer (HF modeling_wav2vec2_conformer.py:568-630): the fp32 residual stream after each of the five sub-blocks
// and the pre-activations the backward pass needs
struct GradConfBuf {
  bf16 *u1 = nullptr, *u2 = nullptr;   // [rows, I]      pre-activations of the two macaron feed-forwards
  bf16* qkv = nullptr;                 // [rows, 3H|4H]  q | k | v  or  q+u | q+v | k | v
  bf16* ctx = nullptr;                 // [rows, H]      attention output  } rotary: the fused attention backward
  float* lse = nullptr;                // [n, heads, T]  log-sum-exp       }
  bf16* raw = nullptr;                 // [rows, 2H]     pointwise_conv1 output, (value, gate) interleaved
  bf16* z = nullptr;                   // [rows, H]      BatchNorm output, the activation's input
  float *r1 = nullptr, *r2 = nullptr, *r3 = nullptr, *r4 = nullptr, *r5 = nullptr;   // [rows, H] each
};

struct GradPlan {
  int n = 0;
  std::vector<Step> steps;
  std::vector<GemmLaunch*> gemms;
  std::vector<PosConvPlan*> posconv;
  std::vector<AttnFaPlan*> attn_fa;
  std::vector<AttnRelPlan*> attn_rel;
  std::vector<AttnBwdPlan*> attn_bwd;
  std::vector<void*> allocs;
  // buffers the entry point reads / snapshots
  float* logits = nullptr;
  float* dA = nullptr;
  bf16* D[2] = {nullptr, nullptr};
  int* frames = nullptr;
  std::map<std::string, std::pair<const void*, size_t>> peek;   // debug: name -> (device buffer, bytes) snapshots
  ~GradPlan() {
    for (auto* f : attn_fa) attention_fa_free(f);
    for (auto* a : attn_rel) attention_rel_free(a);
    for (auto* a : attn_bwd) attention_bwd_free(a);
    for (auto* pc : posconv) posconv_free(pc);
    for (auto* g : gemms) delete g;
    for (void* p : allocs) cudaFree(p);
  }
};

std::string grad_supported(const w2s_handle* h) {
  const w2s_config& c = h->cfg;
  if (c.kind == 2) return "gradient path: WavLMForCTC is not supported (no backward of its gated relative-position bias)";
  if (c.kind == 0) {
    if (c.hidden_act != 0) return "gradient path: Wav2Vec2ForCTC is built for GELU only";
    if (c.num_conv_pos_embeddings % 2) return "gradient path: odd positional-conv kernels are not built";
  } else {
    if (c.position_embeddings_type != 1 && c.position_embeddings_type != 2)
      return "gradient path: the conformer needs relative or rotary position embeddings";
    const int kd = c.conv_depthwise_kernel_size;
    if (kd != 31 && kd != 15 && kd != 7 && kd != 3) return "gradient path: depthwise kernel size must be 31, 15, 7 or 3";
  }
  if (c.hidden_size != c.num_attention_heads * 64) return "gradient path: head_dim must be 64";
  if (c.conv_kernel[0] != 10 || c.conv_dim[0] % 64 || c.conv_dim[0] > 512)
    return "gradient path: conv0 must be k = 10 with 64..512 channels (a multiple of 64)";
  return "";
}

// transposed copies of the dense weights for dX = dY W (once per handle)
std::string grad_prepare_weights(w2s_handle* h) {
  if (h->grad_ready) return "";
  const w2s_config& c = h->cfg;
  const int H = c.hidden_size, I = c.intermediate_size;
  auto tr = [&](const bf16* src, int R, int C, bf16** dst) -> std::string {
    W2S_TRY(dalloc(h->allocs, dst, (size_t)R * C));
    return launch_transpose_bf16(src, *dst, R, C, 0);
  };
  h->gradw.resize(c.num_hidden_layers);
  const bool conf = c.kind == 1, rel = conf && c.position_embeddings_type == 1;
  const int QW = (rel ? 4 : 3) * H;
  for (int l = 0; l < c.num_hidden_layers; ++l) {
    const LayerW& w = h->layers[l];
    GradW& g = h->gradw[l];
    W2S_TRY(tr(w.wqkv, QW, H, &g.wqkvT));      // [3H | 4H][H] -> [H][3H | 4H]
    W2S_TRY(tr(w.wo, H, H, &g.woT));
    W2S_TRY(tr(w.w1, I, H, &g.w1T));           // [I][H] -> [H][I]
    W2S_TRY(tr(w.w2, H, I, &g.w2T));           // [H][I] -> [I][H]
    if (!conf) continue;
    W2S_TRY(tr(w.f2w1, I, H, &g.f2w1T));
    W2S_TRY(tr(w.f2w2, H, I, &g.f2w2T));
    W2S_TRY(tr(w.pw1, 2 * H, H, &g.pw1T));     // (value, gate) interleaved rows -> [H][2H]
    W2S_TRY(tr(w.pw2, H, H, &g.pw2T));
    if (!rel) {                                // rotary: q | k read the rotated input, v the plain one
      W2S_TRY(tr(w.wqkv, 2 * H, H, &g.wqkT));
      W2S_TRY(tr(w.wqkv + (size_t)2 * H * H, H, H, &g.wvT));
    }
    const int kd = c.conv_depthwise_kernel_size;
    W2S_TRY(dalloc(h->allocs, &g.dw_flip, (size_t)kd * H));
    W2S_TRY(launch_flip_taps(w.dw_w, g.dw_flip, kd, H, 0));
  }
  if (conf) {
    W2S_TRY(dalloc(h->allocs, &h->grad_ones, (size_t)H));
    W2S_TRY(dalloc(h->allocs, &h->grad_zeros, (size_t)H, true));
    W2S_TRY(launch_fill_f32(h->grad_ones, 1.0f, H, 0));
  }
  for (int l = 1; l < c.num_conv_layers; ++l)
    W2S_TRY(tr(h->conv_w[l], c.conv_dim[l], c.conv_kernel[l] * c.conv_dim[l - 1], &h->conv_wT[l]));   // [O][kw C] -> [kw C][O]
  const int Cl = c.conv_dim[c.num_conv_layers - 1];
  W2S_TRY(tr(h->fp_w, H, Cl, &h->fp_wT));      // [H][Cl] -> [Cl][H]
  W2S_CUDA_OK(cudaDeviceSynchronize());
  h->grad_ready = true;
  return "";
}

// relative positions: linear_pos(pe) per layer for the current clip length, and its per-head transpose (the W operand of
// d (q + v) = dBD pos_proj); rebuilt when the clip length changes (HF modeling_wav2vec2_conformer.py:159-205, :509-518)
std::string grad_prepare_positions(w2s_handle* h, int T) {
  for (void* p : h->grad_pos_allocs) cudaFree(p);
  h->grad_pos_allocs.clear();
  const w2s_config& c = h->cfg;
  if (c.kind != 1 || c.position_embeddings_type != 1) return "";
  const int H = c.hidden_size, heads = c.num_attention_heads;
  const long long R = 2LL * T - 1, Rp = (R + 63) / 64 * 64;
  bf16* pe = nullptr;
  W2S_TRY(dalloc(h->grad_pos_allocs, &pe, (size_t)R * H));
  W2S_TRY(launch_relpos(T, H, pe, 0));
  for (int l = 0; l < c.num_hidden_layers; ++l) {
    GradW& g = h->gradw[l];
    W2S_TRY(dalloc(h->grad_pos_allocs, &g.pos_proj, (size_t)R * H));
    W2S_TRY(dalloc(h->grad_pos_allocs, &g.pos_projT, (size_t)heads * 64 * Rp, true));
    GemmProblem p = plain_problem(pe, R, H, h->layers[l].wpos, H);
    p.epi.out = g.pos_proj;
    GemmLaunch gl;
    W2S_TRY(gemm_prepare(p, h->num_sms, &gl));
    W2S_TRY(gemm_launch_tc(gl, 0));
    W2S_TRY(launch_head_transpose(g.pos_proj, H, 0, 1, (int)R, (int)Rp, heads, g.pos_projT, 0));
  }
  W2S_CUDA_OK(cudaDeviceSynchronize());
  return "";
}

struct GradBuilder {
  w2s_handle* h;
  GradPlan* plan;
  int n;
  long long L;
  bool debug = false;

  template <typename TT>
  std::string alloc(TT** out, size_t count, bool zero = false) { return dalloc(plan->allocs, out, count, zero); }
  void add(const std::string& name, std::function<std::string(cudaStream_t)> f) {
    plan->steps.push_back(Step{name, std::move(f)});
  }
  std::string add_gemm(const std::string& name, const GemmProblem& p) {
    GemmLaunch* gl = new GemmLaunch();
    plan->gemms.push_back(gl);
    W2S_TRY(gemm_prepare(p, h->num_sms, gl));
    add(name, [gl](cudaStream_t s) { return gemm_launch_tc(*gl, s); });
    plan->steps.back().flops = 2.0 * p.M * (double)p.N * p.K * p.Bz * p.G;
    return "";
  }
  // debug snapshot of a gradient buffer right after the step that produced it
  std::string snap(const std::string& name, const void* src, size_t bytes) {
    if (!debug) return "";
    uint8_t* dst = nullptr;
    W2S_TRY(alloc(&dst, bytes));
    add("snap." + name, [=](cudaStream_t s) -> std::string {
      W2S_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
      return "";
    });
    plan->peek[name] = {dst, bytes};
    return "";
  }

  std::string build() {
    const w2s_config& c = h->cfg;
    const int H = c.hidden_size, I = c.intermediate_size, NL = c.num_hidden_layers, NC = c.num_conv_layers;
    const int C0 = c.conv_dim[0];
    // NB: every value a step lambda uses must be a LOCAL of this function (captured by value): the builder itself is gone
    // by the time the steps run
    std::vector<int> Tl;
    const int T = (int)num_frames(c, L, &Tl);
    if (T <= 0) return "clip shorter than the conv receptive field";
    const long long rows = (long long)n * T;
    const int nn = n;
    w2s_handle* hh = h;
    const bool conf = c.kind == 1;
    const bool rel = conf && c.position_embeddings_type == 1, rotary = conf && c.position_embeddings_type == 2;
    const int QW = (rel ? 4 : 3) * H;                       // q | k | v  or  q+u | q+v | k | v
    const int q_off = 0, k_off = QW - 2 * H, v_off = QW - H;
    const int eact = c.hidden_act == 1 ? ACT_SWISH : ACT_GELU;   // the conformer encoder's activation
    // DeepLIFT handler rules of the reference (custom_shap_handlers.py:35-80; w2s_grad_rules): rows are [explained | reference]
    // halves.  bit 0: SiLU modules use the rescale multiplier (shap's nonlinear_1d); LayerNorm / GroupNorm are linear_1d =
    // the ordinary gradient, and so is every module shap does not know (GELUActivation, the attention matmuls).  bit 1: the
    // GLU placeholder rule.  The reference rows get no seed (head_bwd), so their gradients stay zero.
    const int rules = h->grad_rules;
    if (rules && (n % 2)) return "grad_rules: paired rows need an even number of rows per call (and at most 32)";
    const int rescale_act = (rules & 1) && eact == ACT_SWISH ? 1 : 0, glu_placeholder = (rules & 2) ? 1 : 0;
    const int active_rows = rules ? n / 2 : -1;

    // ---- buffers ------------------------------------------------------------------------------------------------
    std::vector<bf16*> u(NC), y(NC);
    for (int l = 0; l < NC; ++l) {
      W2S_TRY(alloc(&u[l], (size_t)n * Tl[l] * c.conv_dim[l]));
      W2S_TRY(alloc(&y[l], (size_t)n * Tl[l] * c.conv_dim[l]));
    }
    const bool layer = c.feat_extract_norm == 1, stable = !conf && c.do_stable_layer_norm != 0;
    std::vector<bf16*> cpre(NC, nullptr);   // layer-norm front end: conv + bias, the input of the per-frame LayerNorm
    float* ln_rstd0 = nullptr;              // and conv0's per-frame rstd
    if (layer) {
      for (int l = 1; l < NC; ++l) W2S_TRY(alloc(&cpre[l], (size_t)n * Tl[l] * c.conv_dim[l]));
      W2S_TRY(alloc(&ln_rstd0, (size_t)n * Tl[0]));
    }
    float *gn_a = nullptr, *gn_b = nullptr;
    bf16* gn_wb = nullptr;
    W2S_TRY(alloc(&gn_a, (size_t)n * C0));
    W2S_TRY(alloc(&gn_b, (size_t)n * C0));
    W2S_TRY(alloc(&gn_wb, (size_t)n * C0 * 32));
    const int Cl = c.conv_dim[NC - 1];
    bf16 *fpn = nullptr, *h0 = nullptr, *hp = nullptr, *upos = nullptr, *hb = nullptr, *h1 = nullptr, *ctx = nullptr, *ffn = nullptr;
    float* pre0 = nullptr;
    const int G = c.num_conv_pos_embedding_groups, kp = c.num_conv_pos_embeddings, cpg = H / G;
    W2S_TRY(alloc(&fpn, (size_t)rows * Cl));
    if (!conf) {
      W2S_TRY(alloc(&h0, (size_t)rows * H));
      W2S_TRY(alloc(&hp, (size_t)n * (T + kp) * G * 64));
      W2S_TRY(alloc(&upos, (size_t)rows * H));
    }
    W2S_TRY(alloc(&pre0, (size_t)rows * H));
    W2S_TRY(alloc(&hb, (size_t)rows * H));
    W2S_TRY(alloc(&h1, (size_t)rows * H));
    W2S_TRY(alloc(&ctx, (size_t)rows * H));
    W2S_TRY(alloc(&ffn, (size_t)rows * I));
    W2S_TRY(alloc(&plan->logits, (size_t)rows * h->head_ldl));
    // attention backward: one fused tcgen05 kernel (attention_bwd.cu) unless the relative-position term is present or a
    // cross-check form was asked for (w2s_grad_debug bits 1 / 2)
    const bool attn_fused = !rel && !h->grad_attn_simt && !h->grad_attn_unfused;
    // the other forms hold a whole score row per warp (attn_rows_t_kernel, attn_bwd_q_kernel): refuse before launching anything
    if (!attn_fused && T > 1024)
      return std::string("gradient path: ") + (rel ? "the relative-position attention backward" : "the cross-check attention backward") +
             " takes at most 1024 frames (this clip has " + std::to_string(T) + ")";
    const size_t nlse = (size_t)n * c.num_attention_heads * T;
    std::vector<GradLayerBuf> lb(conf ? 0 : NL);
    for (int l = 0; l < NL && !conf; ++l) {
      if (attn_fused) {
        W2S_TRY(alloc(&lb[l].ctx, (size_t)rows * H));
        W2S_TRY(alloc(&lb[l].lse, nlse));
      }
      W2S_TRY(alloc(&lb[l].qkv, (size_t)rows * 3 * H));
      W2S_TRY(alloc(&lb[l].s1, (size_t)rows * H));
      W2S_TRY(alloc(&lb[l].u, (size_t)rows * I));
      W2S_TRY(alloc(&lb[l].s2, (size_t)rows * H));
    }
    std::vector<GradConfBuf> cb(conf ? NL : 0);
    bf16 *hrot = nullptr, *dC2 = nullptr;
    for (int l = 0; l < NL && conf; ++l) {
      if (attn_fused) {
        W2S_TRY(alloc(&cb[l].ctx, (size_t)rows * H));
        W2S_TRY(alloc(&cb[l].lse, nlse));
      }
      W2S_TRY(alloc(&cb[l].u1, (size_t)rows * I));
      W2S_TRY(alloc(&cb[l].u2, (size_t)rows * I));
      W2S_TRY(alloc(&cb[l].qkv, (size_t)rows * QW));
      W2S_TRY(alloc(&cb[l].raw, (size_t)rows * 2 * H));
      W2S_TRY(alloc(&cb[l].z, (size_t)rows * H));
      for (float** r : {&cb[l].r1, &cb[l].r2, &cb[l].r3, &cb[l].r4, &cb[l].r5}) W2S_TRY(alloc(r, (size_t)rows * H));
    }
    if (conf) {
      W2S_TRY(alloc(&hrot, (size_t)rows * H));
      W2S_TRY(alloc(&dC2, (size_t)rows * H));
    }
    // backward
    float *dA = nullptr, *dS = nullptr, *dT = nullptr, *attn_stats = nullptr, *dFp = nullptr, *m12 = nullptr, *gtap = nullptr;
    bf16 *dS16 = nullptr, *dF = nullptr, *dC = nullptr, *dQKV = nullptr, *dcol = nullptr;
    W2S_TRY(alloc(&dA, (size_t)rows * H));
    W2S_TRY(alloc(&dS, (size_t)rows * H));
    if (stable || conf) W2S_TRY(alloc(&dT, (size_t)rows * H));
    W2S_TRY(alloc(&dS16, (size_t)rows * H));
    W2S_TRY(alloc(&dF, (size_t)rows * I));
    W2S_TRY(alloc(&dC, (size_t)rows * H));
    W2S_TRY(alloc(&dQKV, (size_t)rows * QW));
    W2S_TRY(alloc(&attn_stats, (size_t)rows * c.num_attention_heads * 3));
    // attention backward on the tensor cores: [n, heads, T, Tp] score-shaped buffers and per-head transposes, zero padding
    const int heads = c.num_attention_heads;
    const int Tp = (T + 63) / 64 * 64;
    const size_t nsc = (size_t)n * heads * T * Tp, ntr = (size_t)n * heads * 64 * Tp;
    float *aS = nullptr, *adP = nullptr;
    bf16 *aP = nullptr, *aPT = nullptr, *adS = nullptr, *adST = nullptr, *aQT = nullptr, *aKT = nullptr, *adOT = nullptr;
    const bool attn_tc = !h->grad_attn_simt;
    float *adelta = nullptr, *adq = nullptr;
    if (attn_fused) {
      W2S_TRY(alloc(&adelta, nlse));
      W2S_TRY(alloc(&adq, (size_t)rows * H));
    }
    if (conf && !attn_tc) return "gradient path: the CUDA-core attention backward covers Wav2Vec2ForCTC only";
    const int Rp = (2 * T - 1 + 63) / 64 * 64;             // relative positions 2T'-1, padded like Tp
    float* aBD = nullptr;
    bf16* adBD = nullptr;
    if (rel) {
      W2S_TRY(alloc(&aBD, (size_t)n * heads * T * Rp));
      W2S_TRY(alloc(&adBD, (size_t)n * heads * T * Rp));
    }
    if (attn_tc && !attn_fused) {
      W2S_TRY(alloc(&aS, nsc));
      W2S_TRY(alloc(&adP, nsc));
      W2S_TRY(alloc(&aP, nsc, true));
      W2S_TRY(alloc(&aPT, nsc, true));
      W2S_TRY(alloc(&adS, nsc, true));
      W2S_TRY(alloc(&adST, nsc, true));
      W2S_TRY(alloc(&aQT, ntr, true));
      W2S_TRY(alloc(&aKT, ntr, true));
      W2S_TRY(alloc(&adOT, ntr, true));
    }
    W2S_TRY(alloc(&dFp, (size_t)rows * Cl));
    size_t dmax = 0, colmax = 0;
    for (int l = 0; l < NC; ++l) {
      dmax = std::max(dmax, (size_t)n * Tl[l] * c.conv_dim[l]);
      if (l >= 1) colmax = std::max(colmax, (size_t)n * Tl[l] * c.conv_kernel[l] * c.conv_dim[l - 1]);
    }
    W2S_TRY(alloc(&plan->D[0], dmax));
    W2S_TRY(alloc(&plan->D[1], dmax));
    W2S_TRY(alloc(&dcol, colmax));
    W2S_TRY(alloc(&m12, (size_t)n * C0 * (3 + 2 * 32)));   // launch_conv0_bwd scratch: coefficients + 32 time-chunk partial sums
    W2S_TRY(alloc(&gtap, (size_t)n * Tl[0] * c.conv_kernel[0]));
    W2S_TRY(alloc(&plan->frames, (size_t)n));
    plan->dA = dA;

    // ================================ forward, activations saved =================================================
    {
      Conv0Params cp{};
      cp.dyn = h->dyn_dev;
      cp.n = n; cp.L = (int)L; cp.T0 = Tl[0]; cp.C = C0; cp.kw = c.conv_kernel[0]; cp.stride = c.conv_stride[0];
      cp.w = h->conv0_w; cp.bias = layer ? h->conv0_b : nullptr; cp.gamma = h->norm0_g; cp.beta = h->norm0_b;
      cp.gn_a = gn_a; cp.gn_b = gn_b; cp.gn_wb = gn_wb;
      cp.ln_wbar = h->ln0_wbar; cp.ln_gram = h->ln0_gram; cp.ln_wb = h->ln0_wb;
      cp.ln_bmean = h->ln0_bmean; cp.ln_b2mean = h->ln0_b2mean; cp.ln_wb48 = h->ln0_wb48; cp.ln_rstd_out = ln_rstd0;
      cp.out = u[0];
      cp.pre_act = 1;   // store the normalised pre-activation; GELU follows as its own step
      if (layer && !h->ln0_wb48) return "gradient path: the layer-norm conv0 needs the tensor-core form (64..512 channels)";
      if (!layer) add("conv0_stats", [=](cudaStream_t s) { return launch_conv0_stats(cp, s); });
      add("conv0", [=](cudaStream_t s) { return launch_conv0(cp, layer, s); });
      const long long ne = (long long)n * Tl[0] * C0;
      bf16 *uu = u[0], *yy = y[0];
      add("conv0_gelu", [=](cudaStream_t s) { return launch_gelu_fwd(uu, yy, ne, s); });
      W2S_TRY(snap("f.convu0", u[0], sizeof(bf16) * (size_t)ne));
    }
    for (int l = 1; l < NC; ++l) {
      const int Cin = c.conv_dim[l - 1], Cout = c.conv_dim[l], kw = c.conv_kernel[l], st = c.conv_stride[l];
      const int Tin = Tl[l - 1], Tout = Tl[l];
      if ((st * Cin) % 64) return "conv layer " + std::to_string(l) + ": stride * in_channels must be a multiple of 64";
      GemmProblem p;
      p.a = y[l - 1]; p.a_cols = (long long)st * Cin; p.a_rows = (Tin + st - 1) / st; p.a_batches = n;
      p.a_row_stride = (long long)st * Cin; p.a_batch_stride = (long long)Tin * Cin;
      p.a_kb_per_row = st * Cin / 64; p.a_g_col = 0;
      p.w = h->conv_w[l]; p.M = Tout; p.N = Cout; p.K = kw * Cin; p.Bz = n; p.G = 1;
      p.epi.bias = h->conv_b[l];
      p.epi.act = ACT_NONE;
      p.epi.out = layer ? cpre[l] : u[l]; p.epi.ldb = (long long)Tout * Cout; p.epi.ldm = Cout;
      W2S_TRY(add_gemm("conv" + std::to_string(l), p));
      const long long ne = (long long)n * Tout * Cout;
      bf16 *uu = u[l], *yy = y[l];
      if (layer) {
        const bf16* cc = cpre[l];
        const float *lg = h->conv_ln_g[l], *lb2 = h->conv_ln_b[l];
        const long long lrows = (long long)n * Tout;
        add("conv" + std::to_string(l) + "_ln",
            [=](cudaStream_t s) { return launch_layernorm(cc, 0, lrows, Cout, lg, lb2, 1e-5f, ACT_NONE, uu, nullptr, s); });
      }
      add("conv" + std::to_string(l) + "_gelu", [=](cudaStream_t s) { return launch_gelu_fwd(uu, yy, ne, s); });
      W2S_TRY(snap("f.convu" + std::to_string(l), u[l], sizeof(bf16) * (size_t)ne));
    }
    {
      bf16* y6 = y[NC - 1];
      const float *g = h->fp_ln_g, *b = h->fp_ln_b;
      const float eps = c.layer_norm_eps;
      add("featproj_ln", [=](cudaStream_t s) { return launch_layernorm(y6, 0, rows, Cl, g, b, eps, ACT_NONE, fpn, nullptr, s); });
      GemmProblem p = PlanBuilder::plain(fpn, rows, Cl, h->fp_w, H);
      p.epi.bias = h->fp_b; p.epi.out = h0;
      if (conf) {   // the conformer has no positional conv: the projection IS the fp32 residual stream
        p.epi.out = pre0; p.epi.out_fp32 = 1;
      }
      W2S_TRY(add_gemm("featproj", p));
      W2S_TRY(snap("f.conv" + std::to_string(NC - 1), y6, sizeof(bf16) * (size_t)rows * Cl));
      if (conf) W2S_TRY(snap("f.h0", pre0, sizeof(float) * (size_t)rows * H));
      else W2S_TRY(snap("f.h0", h0, sizeof(bf16) * (size_t)rows * H));
    }
    if (!conf) {
      add("pos_pad", [=](cudaStream_t s) { return launch_pos_pad(h0, nn, T, H, G, kp, hp, s, kp / 2); });
      EpiParams e;
      e.bias = h->pos_b; e.act = ACT_NONE; e.out = upos; e.out_fp32 = 0;
      e.ldg = cpg; e.ldb = (long long)T * H; e.ldm = H;
      if (!posconv_supported(H, G, kp)) return "gradient path: positional conv shape not supported by the tcgen05 kernel";
      PosConvPlan* pc = nullptr;
      W2S_TRY(posconv_prepare(hp, h->pos_w, n, T, H, G, kp, e, h->num_sms, &pc));
      plan->posconv.push_back(pc);
      add("pos_conv", [=](cudaStream_t s) { return posconv_launch(pc, s); });
      add("pos_add", [=](cudaStream_t s) { return launch_add_gelu(h0, upos, pre0, rows * H, s); });
      const float *g = h->enc_ln_g, *b = h->enc_ln_b;
      const float eps = c.layer_norm_eps;
      if (!stable) {
        add("encoder_ln", [=](cudaStream_t s) { return launch_layernorm(pre0, 1, rows, H, g, b, eps, ACT_NONE, hb, nullptr, s); });
        W2S_TRY(snap("f.layer0", hb, sizeof(bf16) * (size_t)rows * H));
      }
    }
    AttnParams ap{};
    ap.ctx = ctx; ap.B = n; ap.T = T; ap.Tp = (T + 63) / 64 * 64; ap.H = H;
    ap.heads = c.num_attention_heads; ap.hd = 64;
    ap.ld = QW; ap.q_off = q_off; ap.qv_off = rel ? H : 0; ap.k_off = k_off; ap.v_off = v_off;
    ap.scale = 0.125f;
    const float eps = c.layer_norm_eps;
    const float ceps = 1e-5f;   // the conformer layer's LayerNorms use the nn.LayerNorm default
    // ---- conformer layers: five residual sub-blocks, the fp32 stream saved after each ---------------------------------
    for (int l = 0; l < NL && conf; ++l) {
      const LayerW& w = h->layers[l];
      const GradConfBuf B = cb[l];
      const std::string ls = "L" + std::to_string(l) + ".";
      const float* rin = l == 0 ? pre0 : cb[l - 1].r5;
      auto macaron = [&](const std::string& nm, const float* x, const float* lg, const float* lbias, const bf16* w1,
                         const float* b1, const bf16* w2, const float* b2, bf16* usave, float* rout) -> std::string {
        add(nm + "ln", [=](cudaStream_t s) { return launch_layernorm(x, 1, rows, H, lg, lbias, ceps, ACT_NONE, hb, nullptr, s); });
        GemmProblem p = PlanBuilder::plain(hb, rows, H, w1, I);
        p.epi.bias = b1; p.epi.out = usave;
        W2S_TRY(add_gemm(nm + "ffn1", p));
        add(nm + "act", [=](cudaStream_t s) { return launch_act_fwd(usave, ffn, rows * I, eact, s); });
        GemmProblem q = PlanBuilder::plain(ffn, rows, I, w2, H);
        q.epi.bias = b2; q.epi.alpha = 0.5f; q.epi.residual = x; q.epi.res_fp32 = 1; q.epi.out = rout; q.epi.out_fp32 = 1;
        return add_gemm(nm + "ffn2", q);
      };
      W2S_TRY(macaron(ls + "mac1_", rin, w.lnf1_g, w.lnf1_b, w.w1, w.b1, w.w2, w.b2, B.u1, B.r1));
      {
        const float *g = w.ln1_g, *b = w.ln1_b;
        const float* x = B.r1;
        add(ls + "attn_ln", [=](cudaStream_t s) { return launch_layernorm(x, 1, rows, H, g, b, ceps, ACT_NONE, hb, nullptr, s); });
      }
      if (rotary) {
        const int base = c.rotary_embedding_base;
        add(ls + "rotary", [=](cudaStream_t s) { return launch_rotary(hb, rows, T, H, 64, base, hrot, s); });
        GemmProblem p = PlanBuilder::plain(hrot, rows, H, w.wqkv, 2 * H);
        p.epi.bias = w.bqkv; p.epi.out = B.qkv; p.epi.ldm = 3 * H;
        W2S_TRY(add_gemm(ls + "qk", p));
        GemmProblem v = PlanBuilder::plain(hb, rows, H, w.wqkv + (size_t)2 * H * H, H);
        v.epi.bias = w.bqkv + 2 * H; v.epi.out = B.qkv + 2 * H; v.epi.ldm = 3 * H;
        W2S_TRY(add_gemm(ls + "v", v));
      } else {
        GemmProblem p = PlanBuilder::plain(hb, rows, H, w.wqkv, QW);
        p.epi.bias = w.bqkv; p.epi.out = B.qkv;
        W2S_TRY(add_gemm(ls + "qkv", p));
      }
      {
        AttnParams lp = ap;
        lp.qkv = B.qkv;
        if (rel) {
          lp.pos_proj = h->gradw[l].pos_proj;
          AttnRelPlan* rp = nullptr;
          W2S_TRY(attention_rel_prepare(lp, &rp));
          plan->attn_rel.push_back(rp);
          add(ls + "attention", [=](cudaStream_t s) { return attention_rel_launch(rp, s); });
        } else {
          if (attn_fused) {
            lp.ctx = B.ctx;
            lp.lse = B.lse;
          }
          AttnFaPlan* afl = nullptr;
          W2S_TRY(attention_fa_prepare(lp, h->num_sms, &afl));
          plan->attn_fa.push_back(afl);
          add(ls + "attention", [=](cudaStream_t s) { return attention_fa_launch(afl, s); });
        }
      }
      {
        GemmProblem p = PlanBuilder::plain(attn_fused ? B.ctx : ctx, rows, H, w.wo, H);
        p.epi.bias = w.bo; p.epi.residual = B.r1; p.epi.res_fp32 = 1; p.epi.out = B.r2; p.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "out_proj", p));
      }
      {   // convolution module: LN -> pointwise -> GLU -> depthwise + BatchNorm -> activation -> pointwise (+ residual)
        const float *g = w.lnc_g, *b = w.lnc_b;
        const float* x = B.r2;
        add(ls + "conv_ln", [=](cudaStream_t s) { return launch_layernorm(x, 1, rows, H, g, b, ceps, ACT_NONE, hb, nullptr, s); });
        GemmProblem p = PlanBuilder::plain(hb, rows, H, w.pw1, 2 * H);
        p.epi.out = B.raw;
        W2S_TRY(add_gemm(ls + "pw1", p));
        const bf16* raw = B.raw;
        bf16* z = B.z;
        add(ls + "glu", [=](cudaStream_t s) { return launch_glu_fwd(raw, h1, rows * H, s); });
        const int kd = c.conv_depthwise_kernel_size;
        const float *dw = w.dw_w, *sc = w.dw_scale, *sh = w.dw_shift;
        add(ls + "depthwise", [=](cudaStream_t s) { return launch_depthwise(h1, nn, T, H, kd, dw, sc, sh, ACT_NONE, z, s); });
        add(ls + "conv_act", [=](cudaStream_t s) { return launch_act_fwd(z, ctx, rows * H, eact, s); });
        GemmProblem q = PlanBuilder::plain(ctx, rows, H, w.pw2, H);
        q.epi.residual = B.r2; q.epi.res_fp32 = 1; q.epi.out = B.r3; q.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "pw2", q));
      }
      W2S_TRY(macaron(ls + "mac2_", B.r3, w.lnf2_g, w.lnf2_b, w.f2w1, w.f2b1, w.f2w2, w.f2b2, B.u2, B.r4));
      {
        const float *g = w.lnfin_g, *b = w.lnfin_b;
        const float* x = B.r4;
        float* r5 = B.r5;
        add(ls + "final_ln", [=](cudaStream_t s) { return launch_layernorm(x, 1, rows, H, g, b, ceps, ACT_NONE, nullptr, r5, s); });
        W2S_TRY(snap("f.layer" + std::to_string(l + 1), r5, sizeof(float) * (size_t)rows * H));
      }
    }
    for (int l = 0; l < NL && !conf; ++l) {
      const LayerW& w = h->layers[l];
      const GradLayerBuf B = lb[l];
      const std::string ls = "L" + std::to_string(l) + ".";
      // stable-LN (pre-LN) layers: r1 = residual stream entering the layer (fp32), s1 = r1 + attention(LN1(r1)),
      // s2 = s1 + ffn(LN2(s1)); post-LN layers: s1 = hb + attention(hb), h1 = LN1(s1), s2 = h1 + ffn(h1), hb' = LN2(s2)
      const float* r1 = l == 0 ? pre0 : lb[l - 1].s2;
      if (stable) {
        const float *g = w.ln1_g, *b = w.ln1_b;
        add(ls + "ln1", [=](cudaStream_t s) { return launch_layernorm(r1, 1, rows, H, g, b, eps, ACT_NONE, hb, nullptr, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(hb, rows, H, w.wqkv, 3 * H);
        p.epi.bias = w.bqkv; p.epi.out = B.qkv;
        W2S_TRY(add_gemm(ls + "qkv", p));
      }
      {
        AttnParams lp = ap;
        lp.qkv = B.qkv;
        if (attn_fused) {
          lp.ctx = B.ctx;
          lp.lse = B.lse;
        }
        AttnFaPlan* afl = nullptr;
        W2S_TRY(attention_fa_prepare(lp, h->num_sms, &afl));
        plan->attn_fa.push_back(afl);
        add(ls + "attention", [=](cudaStream_t s) { return attention_fa_launch(afl, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(attn_fused ? B.ctx : ctx, rows, H, w.wo, H);
        p.epi.bias = w.bo;
        if (stable) {
          p.epi.residual = r1; p.epi.res_fp32 = 1;
        } else {
          p.epi.residual = hb; p.epi.res_fp32 = 0;
        }
        p.epi.out = B.s1; p.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "out_proj", p));
      }
      {
        const float *g = stable ? w.ln2_g : w.ln1_g, *b = stable ? w.ln2_b : w.ln1_b;
        const float* in = B.s1;
        add(ls + (stable ? "ln2" : "ln1"),
            [=](cudaStream_t s) { return launch_layernorm(in, 1, rows, H, g, b, eps, ACT_NONE, h1, nullptr, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(h1, rows, H, w.w1, I);
        p.epi.bias = w.b1; p.epi.act = ACT_NONE; p.epi.out = B.u;
        W2S_TRY(add_gemm(ls + "ffn1", p));
        bf16* uu = B.u;
        add(ls + "ffn_gelu", [=](cudaStream_t s) { return launch_gelu_fwd(uu, ffn, rows * I, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(ffn, rows, I, w.w2, H);
        p.epi.bias = w.b2;
        if (stable) {
          p.epi.residual = B.s1; p.epi.res_fp32 = 1;
        } else {
          p.epi.residual = h1; p.epi.res_fp32 = 0;
        }
        p.epi.out = B.s2; p.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "ffn2", p));
      }
      if (!stable) {
        const float *g = w.ln2_g, *b = w.ln2_b;
        const float* in = B.s2;
        add(ls + "ln2", [=](cudaStream_t s) { return launch_layernorm(in, 1, rows, H, g, b, eps, ACT_NONE, hb, nullptr, s); });
        W2S_TRY(snap("f.layer" + std::to_string(l + 1), hb, sizeof(bf16) * (size_t)rows * H));
      }
    }
    const float* last_stream = conf ? cb[NL - 1].r5 : (stable ? lb[NL - 1].s2 : nullptr);
    if (stable || conf) {   // the encoder's LayerNorm comes last (Wav2Vec2EncoderStableLayerNorm, Wav2Vec2ConformerEncoder)
      const float *g = h->enc_ln_g, *b = h->enc_ln_b;
      const float* in = last_stream;
      add("encoder_ln", [=](cudaStream_t s) { return launch_layernorm(in, 1, rows, H, g, b, eps, ACT_NONE, hb, nullptr, s); });
    }
    {
      GemmProblem p = PlanBuilder::plain(hb, rows, H, h->head_w, h->head_ldl);
      p.epi.bias = h->head_b; p.epi.out = plan->logits; p.epi.out_fp32 = 1;
      W2S_TRY(add_gemm("lm_head", p));
      W2S_TRY(snap("f.logits", plan->logits, sizeof(float) * (size_t)rows * h->head_ldl));
    }

    // ================================ backward to the waveform ===================================================
    // attention backward of one layer: (saved q | k | v, dC = d ctx) -> dQKV; shared by both encoder orders
    // (pos_proj / pos_projT: the conformer's relative-position term, S += shift((q + v) pos_proj^T); null otherwise)
    auto add_attention_bwd = [&](const std::string& ls, const bf16* saved_qkv, const bf16* pos_proj, const bf16* pos_projT,
                                 const bf16* saved_ctx, const float* saved_lse) -> std::string {
      if (attn_fused) {
        AttnParams bp = ap;
        bp.qkv = saved_qkv;
        AttnBwdPlan* abp = nullptr;
        W2S_TRY(attention_bwd_prepare(bp, dC, saved_lse, adelta, adq, dQKV, h->num_sms, &abp));
        plan->attn_bwd.push_back(abp);
        add(ls + "attention_bwd", [=](cudaStream_t s) { return attention_bwd_launch(abp, dC, saved_ctx, q_off, s); });
        plan->steps.back().flops = 10.0 * T * (double)T * H * n;   // five T' x T' x 64 contractions per head
      } else if (!attn_tc) {
        const bf16* q = saved_qkv;
        add(ls + "attention_bwd", [=](cudaStream_t s) { return launch_attn_bwd(q, dC, nn, T, H, heads, 0.125f, dQKV, attn_stats, s); });
      } else {
        const bf16* qkv = saved_qkv;
        // operands per (coalition b, head g): columns g*64 of a [rows, ld] buffer, or row block g*T of a [n, heads, T, Tp] one
        auto from_rows = [&](const bf16* base, int ld) {   // A = 64 columns of head g, K = 64
          GemmProblem p;
          p.a = base; p.a_cols = ld; p.a_rows = T; p.a_batches = n; p.a_row_stride = ld; p.a_batch_stride = (long long)T * ld;
          p.a_kb_per_row = 1; p.a_g_col = 64;
          p.M = T; p.K = 64; p.Bz = n; p.G = heads;
          return p;
        };
        auto from_scores = [&](const bf16* base) {        // A = [T, Tp] block of (b, g), K = Tp
          GemmProblem p;
          p.a = base; p.a_cols = Tp; p.a_rows = (long long)heads * T; p.a_batches = n; p.a_row_stride = Tp;
          p.a_batch_stride = (long long)heads * T * Tp; p.a_kb_per_row = Tp / 64; p.a_g_col = 0; p.a_g_row = T;
          p.M = T; p.K = Tp; p.Bz = n; p.G = heads;
          return p;
        };
        auto w_rows_of = [&](GemmProblem& p, const bf16* base, int ld) {   // W = the T rows of head g in a [rows, ld] buffer
          p.w = base; p.w_row_stride = ld; p.w_g_stride = 64; p.w_batch_stride = (long long)T * ld; p.w_rows = T; p.N = Tp;
        };
        auto w_transposed = [&](GemmProblem& p, const bf16* base) {        // W = [64, Tp] block of (b, g)
          p.w = base; p.w_row_stride = Tp; p.w_g_stride = 64LL * Tp; p.w_batch_stride = (long long)heads * 64 * Tp; p.N = 64;
        };
        auto score_out = [&](GemmProblem& p, float* out, float alpha) {
          p.epi.out = out; p.epi.out_fp32 = 1; p.epi.alpha = alpha;
          p.epi.ldg = (long long)T * Tp; p.epi.ldb = (long long)heads * T * Tp; p.epi.ldm = Tp;
        };
        auto qkv_out = [&](GemmProblem& p, bf16* out, float alpha) {
          p.epi.out = out; p.epi.out_fp32 = 0; p.epi.alpha = alpha;
          p.epi.ldg = 64; p.epi.ldb = (long long)T * QW; p.epi.ldm = QW;
        };
        {
          GemmProblem p = from_rows(qkv + q_off, QW);            // S = scale Q K^T
          w_rows_of(p, qkv + k_off, QW);
          score_out(p, aS, 0.125f);
          W2S_TRY(add_gemm(ls + "attn_scores", p));
        }
        if (pos_proj) {                                          // + scale (q + v) . pos_proj[T - 1 - i + j]
          GemmProblem p = from_rows(qkv + H, QW);
          p.w = pos_proj; p.w_row_stride = H; p.w_g_stride = 64; p.w_batch_stride = 0; p.w_rows = 2 * T - 1; p.N = Rp;
          p.epi.out = aBD; p.epi.out_fp32 = 1; p.epi.alpha = 0.125f;
          p.epi.ldg = (long long)T * Rp; p.epi.ldb = (long long)heads * T * Rp; p.epi.ldm = Rp;
          W2S_TRY(add_gemm(ls + "attn_pos_scores", p));
        }
        const float* bd = pos_proj ? aBD : nullptr;   // the rel-shift is folded into the softmax kernel's row read
        add(ls + "attn_softmax", [=](cudaStream_t s) { return launch_attn_softmax_t(aS, nn * heads, T, Tp, aP, aPT, s, bd, Rp); });
        {
          GemmProblem p = from_rows(dC, H);                      // dP = dO V^T
          w_rows_of(p, qkv + v_off, QW);
          score_out(p, adP, 1.0f);
          W2S_TRY(add_gemm(ls + "attn_dp", p));
        }
        add(ls + "attn_ds", [=](cudaStream_t s) { return launch_attn_ds_t(aP, adP, nn * heads, T, Tp, adS, adST, s); });
        add(ls + "attn_transposes", [=](cudaStream_t s) -> std::string {
          W2S_TRY(launch_head_transpose(qkv, QW, q_off, nn, T, Tp, heads, aQT, s));
          W2S_TRY(launch_head_transpose(qkv, QW, k_off, nn, T, Tp, heads, aKT, s));
          return launch_head_transpose(dC, H, 0, nn, T, Tp, heads, adOT, s);
        });
        {
          GemmProblem p = from_scores(adS);                      // dQ = scale dS K
          w_transposed(p, aKT);
          qkv_out(p, dQKV + q_off, 0.125f);
          W2S_TRY(add_gemm(ls + "attn_dq", p));
        }
        if (pos_proj) {                                          // d (q + v) = scale unshift(dS) pos_proj
          add(ls + "attn_rel_unshift", [=](cudaStream_t s) { return launch_rel_unshift(adS, adBD, nn * heads, T, Tp, Rp, s); });
          GemmProblem p;
          p.a = adBD; p.a_cols = Rp; p.a_rows = (long long)heads * T; p.a_batches = n; p.a_row_stride = Rp;
          p.a_batch_stride = (long long)heads * T * Rp; p.a_kb_per_row = Rp / 64; p.a_g_col = 0; p.a_g_row = T;
          p.M = T; p.K = Rp; p.Bz = n; p.G = heads;
          p.w = pos_projT; p.w_row_stride = Rp; p.w_g_stride = 64LL * Rp; p.w_batch_stride = 0; p.N = 64;
          qkv_out(p, dQKV + H, 0.125f);
          W2S_TRY(add_gemm(ls + "attn_dqv", p));
        }
        {
          GemmProblem p = from_scores(adST);                     // dK = scale dS^T Q
          w_transposed(p, aQT);
          qkv_out(p, dQKV + k_off, 0.125f);
          W2S_TRY(add_gemm(ls + "attn_dk", p));
        }
        {
          GemmProblem p = from_scores(aPT);                      // dV = P^T dO
          w_transposed(p, adOT);
          qkv_out(p, dQKV + v_off, 1.0f);
          W2S_TRY(add_gemm(ls + "attn_dv", p));
        }
      }
      return "";
    };
    {
      const float* lg = plan->logits;
      const int ldl = h->head_ldl, V = c.vocab_size;
      const bf16* hw = h->head_w;
      const int* fr = plan->frames;
      float* seed = (stable || conf) ? dT : dA;
      // per-row target frame (w2s_grad_waveforms), or an upstream gradient over all frames (w2s_vjp_waveforms)
      // or the transcript log-likelihood of w2s_grad_transcripts, whose frame slots carry the transcript indices
      add("head_bwd", [=](cudaStream_t s) {
        if (hh->grad_gout) return launch_head_vjp(lg, ldl, V, hw, nn, T, H, hh->grad_gout, seed, hh->grad_out_val, s);
        if (hh->grad_ctc)
          return launch_ctc_seed(lg, ldl, V, hw, nn, T, H, hh->ctc_labels, hh->ctc_offsets, fr, hh->ctc_blank, hh->ctc_smax,
                                 hh->ctc_alpha, hh->ctc_lse, hh->ctc_dz, ldl, seed, hh->grad_out_val, s);
        return launch_head_bwd(lg, ldl, V, hw, nn, T, H, fr, seed, hh->grad_out_val, s, active_rows);
      });
      if (stable || conf) {   // final encoder LayerNorm: dA = d (residual stream after the last layer)
        const float* g = h->enc_ln_g;
        const float* x = last_stream;
        add("encoder_ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(dT, x, 1, rows, H, g, eps, nullptr, dA, nullptr, s); });
      }
      W2S_TRY(snap("layer" + std::to_string(NL), dA, sizeof(float) * rows * H));
    }
    // ---- conformer layers, backward.  gc = gradient of the fp32 stream at the current point, go = the other buffer; every
    // sub-block is  stream' = stream + f(LN(stream)):  d stream = d stream' + LN^T(f^T(d stream')), written to `go`, then swapped
    float *gc = dA, *go = dS;
    for (int l = NL - 1; l >= 0 && conf; --l) {
      const LayerW& w = h->layers[l];
      const GradW& gw = h->gradw[l];
      const GradConfBuf B = cb[l];
      const std::string ls = "B" + std::to_string(l) + ".";
      const float* rin = l == 0 ? pre0 : cb[l - 1].r5;
      auto ln_back = [&](const std::string& nm, const float* dy, const float* x, const float* gamma, const float* addend) {
        float *dst = go;
        add(nm, [=](cudaStream_t s) { return launch_ln_bwd(dy, x, 1, rows, H, gamma, ceps, addend, dst, dS16, s); });
        std::swap(gc, go);
      };
      auto macaron_back = [&](const std::string& nm, const bf16* w2T, const bf16* w1T, const bf16* usave, const float* x,
                              const float* gamma) -> std::string {
        GemmProblem p = PlanBuilder::plain(dS16, rows, H, w2T, I);      // dS16 = bf16 copy of gc
        p.epi.alpha = 0.5f; p.epi.out = dF;
        W2S_TRY(add_gemm(nm + "ffn2_bwd", p));
        add(nm + "act_bwd", [=](cudaStream_t s) { return launch_act_bwd(usave, dF, rows * I, eact, nullptr, H, s, rescale_act); });
        GemmProblem q = PlanBuilder::plain(dF, rows, I, w1T, H);
        q.epi.out = dT; q.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(nm + "ffn1_bwd", q));
        ln_back(nm + "ln_bwd", dT, x, gamma, gc);
        return "";
      };
      ln_back(ls + "final_ln_bwd", gc, B.r4, w.lnfin_g, nullptr);                              // gc = d r4
      W2S_TRY(macaron_back(ls + "mac2_", gw.f2w2T, gw.f2w1T, B.u2, B.r3, w.lnf2_g));            // gc = d r3
      {
        GemmProblem p = PlanBuilder::plain(dS16, rows, H, gw.pw2T, H);
        p.epi.out = dC;
        W2S_TRY(add_gemm(ls + "pw2_bwd", p));
        const bf16 *z = B.z, *raw = B.raw;
        const float* sc = w.dw_scale;
        const int kd = c.conv_depthwise_kernel_size;
        const float *flip = gw.dw_flip, *ones = h->grad_ones, *zeros = h->grad_zeros;
        add(ls + "conv_act_bwd", [=](cudaStream_t s) { return launch_act_bwd(z, dC, rows * H, eact, sc, H, s, rescale_act); });
        add(ls + "depthwise_bwd", [=](cudaStream_t s) { return launch_depthwise(dC, nn, T, H, kd, flip, ones, zeros, ACT_NONE, dC2, s); });
        add(ls + "glu_bwd", [=](cudaStream_t s) { return launch_glu_bwd(raw, dC2, dQKV, rows * H, s, glu_placeholder); });
        GemmProblem q = PlanBuilder::plain(dQKV, rows, 2 * H, gw.pw1T, H);
        q.epi.out = dT; q.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "pw1_bwd", q));
        ln_back(ls + "conv_ln_bwd", dT, B.r2, w.lnc_g, gc);                                     // gc = d r2
      }
      {
        GemmProblem p = PlanBuilder::plain(dS16, rows, H, gw.woT, H);
        p.epi.out = dC;
        W2S_TRY(add_gemm(ls + "out_proj_bwd", p));
        W2S_TRY(add_attention_bwd(ls, B.qkv, rel ? gw.pos_proj : nullptr, rel ? gw.pos_projT : nullptr, B.ctx, B.lse));
        if (rotary) {   // q | k came from the rotated input, v from the plain one
          GemmProblem qk = PlanBuilder::plain(dQKV, rows, 2 * H, gw.wqkT, H);
          qk.a_row_stride = 3 * H;
          qk.epi.out = hrot;
          W2S_TRY(add_gemm(ls + "qk_bwd", qk));
          const int base = c.rotary_embedding_base;
          add(ls + "rotary_bwd", [=](cudaStream_t s) { return launch_rotary(hrot, rows, T, H, 64, base, dC2, s, 1); });
          GemmProblem v = PlanBuilder::plain(dQKV + 2 * H, rows, H, gw.wvT, H);
          v.a_row_stride = 3 * H;
          v.epi.residual = dC2; v.epi.res_fp32 = 0; v.epi.out = dT; v.epi.out_fp32 = 1;
          W2S_TRY(add_gemm(ls + "v_bwd", v));
        } else {
          GemmProblem q = PlanBuilder::plain(dQKV, rows, QW, gw.wqkvT, H);
          q.epi.out = dT; q.epi.out_fp32 = 1;
          W2S_TRY(add_gemm(ls + "qkv_bwd", q));
        }
        ln_back(ls + "attn_ln_bwd", dT, B.r1, w.ln1_g, gc);                                     // gc = d r1
      }
      W2S_TRY(macaron_back(ls + "mac1_", gw.w2T, gw.w1T, B.u1, rin, w.lnf1_g));                 // gc = d (layer input)
      W2S_TRY(snap("layer" + std::to_string(l), gc, sizeof(float) * rows * H));
    }
    for (int l = NL - 1; l >= 0 && stable; --l) {
      // invariant: dA = d s2_l (gradient of the residual stream leaving layer l)
      const LayerW& w = h->layers[l];
      const GradW& gw = h->gradw[l];
      const GradLayerBuf B = lb[l];
      const std::string ls = "B" + std::to_string(l) + ".";
      const float* r1 = l == 0 ? pre0 : lb[l - 1].s2;
      add(ls + "cast", [=](cudaStream_t s) { return launch_grad_cast(dA, nullptr, dS16, rows * H, s); });
      {
        GemmProblem p = PlanBuilder::plain(dS16, rows, H, gw.w2T, I);
        p.epi.out = dF;
        W2S_TRY(add_gemm(ls + "ffn2_bwd", p));
        const bf16* uu = B.u;
        add(ls + "gelu_bwd", [=](cudaStream_t s) { return launch_gelu_bwd(uu, dF, rows * I, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(dF, rows, I, gw.w1T, H);
        p.epi.out = dT; p.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "ffn1_bwd", p));
      }
      {   // d s1 = d s2 + LN2^T (d h1)
        const float* g = w.ln2_g;
        const float* x = B.s1;
        add(ls + "ln2_bwd", [=](cudaStream_t s) { return launch_ln_bwd(dT, x, 1, rows, H, g, eps, dA, dS, dS16, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(dS16, rows, H, gw.woT, H);
        p.epi.out = dC;
        W2S_TRY(add_gemm(ls + "out_proj_bwd", p));
      }
      W2S_TRY(add_attention_bwd(ls, B.qkv, nullptr, nullptr, B.ctx, B.lse));
      {
        GemmProblem p = PlanBuilder::plain(dQKV, rows, 3 * H, gw.wqkvT, H);
        p.epi.out = dT; p.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "qkv_bwd", p));
      }
      {   // d r1 = d s1 + LN1^T (d hb)
        const float* g = w.ln1_g;
        add(ls + "ln1_bwd", [=](cudaStream_t s) { return launch_ln_bwd(dT, r1, 1, rows, H, g, eps, dS, dA, nullptr, s); });
      }
      W2S_TRY(snap("layer" + std::to_string(l), dA, sizeof(float) * rows * H));
    }
    for (int l = NL - 1; l >= 0 && !stable && !conf; --l) {
      const LayerW& w = h->layers[l];
      const GradW& gw = h->gradw[l];
      const GradLayerBuf B = lb[l];
      const std::string ls = "B" + std::to_string(l) + ".";
      {
        const float* g = w.ln2_g;
        const float* x = B.s2;
        add(ls + "ln2_bwd", [=](cudaStream_t s) { return launch_ln_bwd(dA, x, 1, rows, H, g, eps, nullptr, dS, dS16, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(dS16, rows, H, gw.w2T, I);
        p.epi.out = dF;
        W2S_TRY(add_gemm(ls + "ffn2_bwd", p));
        const bf16* uu = B.u;
        add(ls + "gelu_bwd", [=](cudaStream_t s) { return launch_gelu_bwd(uu, dF, rows * I, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(dF, rows, I, gw.w1T, H);
        p.epi.residual = dS; p.epi.res_fp32 = 1; p.epi.out = dA; p.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "ffn1_bwd", p));
      }
      {
        const float* g = w.ln1_g;
        const float* x = B.s1;
        add(ls + "ln1_bwd", [=](cudaStream_t s) { return launch_ln_bwd(dA, x, 1, rows, H, g, eps, nullptr, dS, dS16, s); });
      }
      {
        GemmProblem p = PlanBuilder::plain(dS16, rows, H, gw.woT, H);
        p.epi.out = dC;
        W2S_TRY(add_gemm(ls + "out_proj_bwd", p));
      }
      W2S_TRY(add_attention_bwd(ls, B.qkv, nullptr, nullptr, B.ctx, B.lse));
      {
        GemmProblem p = PlanBuilder::plain(dQKV, rows, 3 * H, gw.wqkvT, H);
        p.epi.residual = dS; p.epi.res_fp32 = 1; p.epi.out = dA; p.epi.out_fp32 = 1;
        W2S_TRY(add_gemm(ls + "qkv_bwd", p));
      }
      W2S_TRY(snap("layer" + std::to_string(l), dA, sizeof(float) * rows * H));
    }
    if (conf) {
      // the layer stack read the feature projection directly: d h0 = gc
      W2S_TRY(snap("h0", gc, sizeof(float) * rows * H));
      const float* src = gc;
      add("h0_cast", [=](cudaStream_t s) { return launch_grad_cast(src, nullptr, dS16, rows * H, s); });
    } else {
      // encoder input: hb0 = LN(pre0), pre0 = h0 + gelu(pos_conv(h0))
      const float* g = h->enc_ln_g;
      if (stable)   // the residual stream enters the first layer un-normalised: d pre0 = dA
        add("pre0_copy", [=](cudaStream_t s) -> std::string {
          W2S_CUDA_OK(cudaMemcpyAsync(dS, dA, sizeof(float) * rows * H, cudaMemcpyDeviceToDevice, s));
          return "";
        });
      else
        add("encoder_ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(dA, pre0, 1, rows, H, g, eps, nullptr, dS, nullptr, s); });
      add("pos_gelu_bwd", [=](cudaStream_t s) { return launch_grad_cast(dS, upos, dS16, rows * H, s); });
      add("pos_pad_bwd", [=](cudaStream_t s) { return launch_pos_pad(dS16, nn, T, H, G, kp, hp, s, kp / 2 - 1); });
      EpiParams e;
      e.act = ACT_NONE; e.residual = dS; e.res_fp32 = 1; e.out = dA; e.out_fp32 = 1;
      e.ldg = cpg; e.ldb = (long long)T * H; e.ldm = H;
      PosConvPlan* pc = nullptr;
      W2S_TRY(posconv_prepare(hp, h->pos_w_bwd, n, T, H, G, kp, e, h->num_sms, &pc));
      plan->posconv.push_back(pc);
      add("pos_conv_bwd", [=](cudaStream_t s) { return posconv_launch(pc, s); });
      W2S_TRY(snap("h0", dA, sizeof(float) * rows * H));
      add("h0_cast", [=](cudaStream_t s) { return launch_grad_cast(dA, nullptr, dS16, rows * H, s); });
    }
    {
      GemmProblem p = PlanBuilder::plain(dS16, rows, H, h->fp_wT, Cl);
      p.epi.out = dFp; p.epi.out_fp32 = 1;
      W2S_TRY(add_gemm("featproj_bwd", p));
      const float* gl = h->fp_ln_g;
      const bf16* y6 = y[NC - 1];
      bf16* d6 = plan->D[(NC - 1) & 1];
      add("featproj_ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(dFp, y6, 0, rows, Cl, gl, eps, nullptr, nullptr, d6, s); });
      W2S_TRY(snap("conv" + std::to_string(NC - 1), d6, sizeof(bf16) * rows * Cl));
      const bf16* u6 = u[NC - 1];
      add("conv" + std::to_string(NC - 1) + "_gelu_bwd", [=](cudaStream_t s) { return launch_gelu_bwd(u6, d6, rows * Cl, s); });
    }
    for (int l = NC - 1; l >= 1; --l) {
      // D[l & 1] holds d u_l [n, T_l, C_l]; contraction with the transposed filters, then gather to d u_(l-1)
      const int Cin = c.conv_dim[l - 1], Cout = c.conv_dim[l], kw = c.conv_kernel[l], st = c.conv_stride[l];
      const int Tin = Tl[l - 1], Tout = Tl[l];
      bf16* dul = plan->D[l & 1];
      bf16* dprev = plan->D[(l - 1) & 1];
      if (layer) {   // through the per-frame LayerNorm: d (conv + bias) from d u_l, in place
        const bf16* cc = cpre[l];
        const float* lg = h->conv_ln_g[l];
        const long long lrows = (long long)n * Tout;
        add("conv" + std::to_string(l) + "_ln_bwd",
            [=](cudaStream_t s) { return launch_ln_bwd(dul, cc, 0, lrows, Cout, lg, 1e-5f, nullptr, nullptr, dul, s, 0); });
      }
      GemmProblem p = PlanBuilder::plain(dul, (long long)n * Tout, Cout, h->conv_wT[l], kw * Cin);
      p.epi.out = dcol;
      W2S_TRY(add_gemm("conv" + std::to_string(l) + "_bwd", p));
      const bf16* up = u[l - 1];
      add("conv" + std::to_string(l) + "_gather",
          [=](cudaStream_t s) { return launch_conv_gather(dcol, nn, Tin, Tout, Cin, kw, st, up, dprev, s); });
      W2S_TRY(snap("convu" + std::to_string(l - 1), dprev, sizeof(bf16) * (size_t)n * Tin * Cin));
    }
    {
      const bf16* du0 = plan->D[0];
      const bf16* u0 = u[0];
      const int T0 = Tl[0], kw = c.conv_kernel[0], st = c.conv_stride[0];
      const float *w0 = h->conv0_w, *gam = h->norm0_g, *bet = h->norm0_b;
      const long long LL = L;
      add("conv0_bwd", [=](cudaStream_t s) {
        if (layer) return launch_conv0_ln_bwd(du0, u0, ln_rstd0, nn, LL, T0, C0, kw, st, w0, gam, bet, gtap, hh->grad_out, LL, s);
        return launch_conv0_bwd(du0, u0, nn, LL, T0, C0, kw, st, w0, gn_a, gam, bet, m12, gtap, hh->grad_out, LL, s);
      });
    }
    return "";
  }
};

std::string get_grad_plan(w2s_handle* h, int n, long long L, GradPlan** out) {
  if (h->grad_L != L || h->grad_debug_built != h->grad_debug || h->grad_rules_built != h->grad_rules) {
    cudaDeviceSynchronize();
    h->grad_plans.clear();
    h->grad_rules_built = h->grad_rules;
    if (h->grad_L != L || h->grad_pos_allocs.empty()) W2S_TRY(grad_prepare_positions(h, (int)num_frames(h->cfg, L, nullptr)));
    h->grad_L = L;
    h->grad_debug_built = h->grad_debug;
  }
  auto it = h->grad_plans.find(n);
  if (it != h->grad_plans.end()) {
    *out = it->second.get();
    return "";
  }
  std::shared_ptr<GradPlan> pl(new GradPlan());
  pl->n = n;
  GradBuilder b{h, pl.get(), n, L};
  b.debug = h->grad_debug;
  W2S_TRY(b.build());
  *out = pl.get();
  h->grad_plans[n] = pl;
  return "";
}

// rows in tiles of `tile`; per tile: argument block, target frames, forward + backward
std::string run_grad(w2s_handle* h, const float* x, long long ld, long long L, int64_t n, const int32_t* frames_host,
                     const float* gout, float* grad, float* out_val, cudaStream_t s) {
  W2S_TRY(grad_supported(h));
  W2S_TRY(grad_prepare_weights(h));
  const int64_t T = num_frames(h->cfg, L, nullptr);
  if (T <= 0) return "clip shorter than the conv receptive field";
  if (h->grad_ctc) {   // transcript indices, checked by w2s_grad_transcripts; seed scratch for one tile
    const long long tile_rows = n < h->grad_tile ? n : h->grad_tile;
    auto grow = [&](float** p, long long* cap, long long need) -> std::string {
      if (*cap >= need) return "";
      W2S_CUDA_OK(cudaStreamSynchronize(s));   // earlier calls may still use the old scratch
      if (*p) cudaFree(*p);
      *p = nullptr;
      *cap = 0;
      W2S_CUDA_OK(cudaMalloc((void**)p, sizeof(float) * need));
      *cap = need;
      return "";
    };
    W2S_TRY(grow(&h->ctc_alpha, &h->ctc_alpha_cap, tile_rows * T * h->ctc_smax));
    W2S_TRY(grow(&h->ctc_lse, &h->ctc_lse_cap, tile_rows * T));
    W2S_TRY(grow(&h->ctc_dz, &h->ctc_dz_cap, tile_rows * T * h->head_ldl));
  }
  if (frames_host) {
    for (int64_t i = 0; i < n && !h->grad_ctc; ++i)
      if (frames_host[i] < 0 || frames_host[i] >= T)
        return "target frame " + std::to_string(frames_host[i]) + " outside the clip's " + std::to_string(T) + " frames";
    if (!h->grad_frames_pinned) {
      W2S_CUDA_OK(cudaHostAlloc(&h->grad_frames_pinned, sizeof(int32_t) * w2s_handle::kFrameSlots * h->grad_tile, cudaHostAllocDefault));
      for (auto& e : h->grad_frames_done) W2S_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
  }
  const int tile = h->grad_tile;
  if (h->grad_rules && (n > tile || n % 2))
    return "grad_rules: paired [explained | reference] rows must come as one tile (an even number of rows, at most " +
           std::to_string(tile) + ")";
  for (int64_t k0 = 0; k0 < n; k0 += tile) {
    const int nt = (int)((n - k0) < tile ? (n - k0) : tile);
    GradPlan* pl = nullptr;
    W2S_TRY(get_grad_plan(h, nt, L, &pl));
    DynArgs d{};
    d.x = x + k0 * ld; d.ld = ld;
    set_dyn_kernel<<<1, 1, 0, s>>>(h->dyn_dev, d);
    if (frames_host) {
      const unsigned slot = h->grad_frames_next++ % w2s_handle::kFrameSlots;
      W2S_CUDA_OK(cudaEventSynchronize(h->grad_frames_done[slot]));   // the copy that last read this slot (no-op when unused)
      int32_t* src = h->grad_frames_pinned + (size_t)slot * h->grad_tile;
      std::memcpy(src, frames_host + k0, sizeof(int32_t) * nt);
      W2S_CUDA_OK(cudaMemcpyAsync(pl->frames, src, sizeof(int) * nt, cudaMemcpyHostToDevice, s));
      W2S_CUDA_OK(cudaEventRecord(h->grad_frames_done[slot], s));
    }
    h->grad_out = grad + k0 * L;
    h->grad_gout = gout ? gout + k0 * T : nullptr;
    h->grad_out_val = out_val ? out_val + k0 * (gout ? T : 1) : nullptr;
    for (const Step& st : pl->steps) {
      ProfRec rec;
      if (h->profiling) {
        rec.name = "grad." + st.name;
        rec.flops = st.flops;
        rec.bytes = st.bytes;
        cudaEventCreate(&rec.e0);
        cudaEventCreate(&rec.e1);
        cudaEventRecord(rec.e0, s);
      }
      std::string e = st.run(s);
      if (h->profiling) {
        cudaEventRecord(rec.e1, s);
        h->prof.push_back(rec);
      }
      if (!e.empty()) return st.name + ": " + e;
    }
    h->launches += (long long)pl->steps.size() + 1 + (h->grad_ctc ? 1 : 0);   // the CTC seed step launches two kernels
  }
  return "";
}
