// CTC forward-backward over one row of frame logits (the output W2S_OUT_CTC and its gradient seed), one warp per
// (row, transcript).  HF computes the same quantity as -Wav2Vec2ForCTC(x, labels=y).loss with reduction "sum":
// log_softmax in fp32, then torch.nn.functional.ctc_loss (HF wav2vec2/modeling_wav2vec2.py, Wav2Vec2ForCTC.forward).
//
// Extended labels l'_s, s = 0 .. S-1, S = 2U + 1: blank at even s, y_{(s-1)/2} at odd s.  The recursion runs in the log
// domain in fp32; -inf marks unreachable states and never meets another -inf in a subtraction.  The S states are spread
// over the 32 lanes in contiguous blocks of k = ceil(S / 32); lane i owns [i k, min(S, i k + k)) and its two neighbour
// states come from the previous (alpha) or next (beta) lane through shared memory.  Every value is produced by one fixed
// sequence of operations that depends only on the row's logits, so it is bit-reproducible for any batch position.
#pragma once
#include "common.cuh"

namespace w2s {

constexpr int CTC_MAX_U = 512;                 // W2S_MAX_TRANSCRIPT
constexpr int CTC_MAX_S = 2 * CTC_MAX_U + 1;   // extended states

__device__ __forceinline__ float ctc_lae2(float a, float b) {
  const float m = fmaxf(a, b);
  if (m == -INFINITY) return -INFINITY;
  return m + logf(expf(a - m) + expf(b - m));
}
__device__ __forceinline__ float ctc_lae3(float a, float b, float c) {
  const float m = fmaxf(a, fmaxf(b, c));
  if (m == -INFINITY) return -INFINITY;
  return m + logf(expf(a - m) + expf(b - m) + expf(c - m));
}

// extended label of state s, and whether the skip transition s-2 -> s is allowed (s odd, s >= 3, y differs from y before)
__device__ __forceinline__ int ctc_label(const int* __restrict__ lab, int blank, int s) {
  return (s & 1) ? __ldg(lab + (s >> 1)) : blank;
}
__device__ __forceinline__ bool ctc_skip(const int* __restrict__ lab, int s) {
  return (s & 1) && s >= 3 && __ldg(lab + (s >> 1)) != __ldg(lab + (s >> 1) - 1);
}

// log-sum-exp over the vocabulary of one frame held one-per-lane (logit[j] = entry lane + 32 j, -inf past V); the same
// fixed shuffle tree on every lane, so every lane holds the same value
template <int J>
__device__ __forceinline__ float ctc_frame_lse(const float (&logit)[J], int V, int lane) {
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j)
    if (lane + 32 * j < V) mx = fmaxf(mx, logit[j]);
  mx = warp_max(mx);
  float se = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j)
    if (lane + 32 * j < V) se += expf(logit[j] - mx);
  return mx + logf(warp_sum(se));
}

// log p_CTC(y | frames).  frame(t, logit) loads frame t one-per-lane (as ctc_frame_lse takes it) and returns a pointer
// through which the frame's logits are indexed by vocabulary id.  alpha: this warp's shared scratch of S floats.  When
// alpha_out is given, alpha_t(s) is also stored at alpha_out[t * S + s] and lse_t at lse_out[t] (the gradient seed).
// Every lane returns the result.
template <int J, class Frame>
__device__ float ctc_forward_warp(int T, int V, const int* __restrict__ lab, int U, int blank, int lane, float* alpha,
                                  Frame frame, float* __restrict__ alpha_out = nullptr, float* __restrict__ lse_out = nullptr) {
  const int S = 2 * U + 1;
  const int k = (S + 31) >> 5;
  const int s0 = lane * k, s1 = min(S, s0 + k);
  for (int t = 0; t < T; ++t) {
    float logit[J];
    const float* z = frame(t, logit);
    const float lse = ctc_frame_lse(logit, V, lane);
    if (t == 0) {
      for (int s = s0; s < s1; ++s) alpha[s] = s < 2 ? z[ctc_label(lab, blank, s)] - lse : -INFINITY;
    } else {
      // neighbours owned by the previous lane, read before anyone writes; own states updated from the top down, so
      // alpha[s - 1] and alpha[s - 2] are still those of frame t - 1 when state s reads them
      const float p1 = (s0 < s1 && s0 >= 1) ? alpha[s0 - 1] : -INFINITY;
      const float p2 = (s0 < s1 && s0 >= 2) ? alpha[s0 - 2] : -INFINITY;
      __syncwarp();
      for (int s = s1 - 1; s >= s0; --s) {
        const float a = alpha[s];
        const float b = s - 1 >= s0 ? alpha[s - 1] : p1;
        const float c = ctc_skip(lab, s) ? (s - 2 >= s0 ? alpha[s - 2] : (s - 2 == s0 - 1 ? p1 : p2)) : -INFINITY;
        const float m = ctc_lae3(a, b, c);
        alpha[s] = m == -INFINITY ? -INFINITY : m + (z[ctc_label(lab, blank, s)] - lse);
      }
    }
    if (alpha_out) {
      for (int s = s0; s < s1; ++s) alpha_out[(long long)t * S + s] = alpha[s];
      if (lane == 0) lse_out[t] = lse;
    }
    __syncwarp();
  }
  const float r = S >= 2 ? ctc_lae2(alpha[S - 1], alpha[S - 2]) : alpha[S - 1];
  __syncwarp();   // alpha may be reused by the caller's next item
  return r;
}

// frames a transcript needs: one per label, plus one blank between each pair of equal adjacent labels
inline int ctc_frames_needed(const int32_t* y, int U) {
  int need = U;
  for (int u = 1; u < U; ++u) need += y[u] == y[u - 1];
  return need;
}

}  // namespace w2s
