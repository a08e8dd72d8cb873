// Recognition errors of one row's greedy transcript against a reference (the output W2S_OUT_ERRORS), one warp per
// (row, reference): the Levenshtein distance over labels or over words, see include/w2s.h.
//
// Greedy decode: per frame a warp argmax, the lowest id among equal maxima (torch.argmax / numpy.argmax), then repeats
// collapsed and blanks dropped.  The hypothesis is consumed as a stream of symbols -- every emitted label, or every
// finished word -- and each symbol advances the edit distance by one column, so nothing bounds T'.
//
// Edit distance: Myers' bit-parallel recurrence in Hyyro's form over the reference's m <= 512 units, held as one 512-bit
// vector pair (VP, VN) of vertical deltas, 32 units per lane in lanes 0 .. 15 (lanes 16 .. 31 hold units past 512 that
// nothing reads).  One column is a few bit operations per lane; the two cross-lane parts are the 512-bit addition, whose
// carries come from a carry-lookahead over the lanes' generate / propagate ballots, and the one-unit shift of the
// horizontal deltas, whose top bits travel by ballot.  Every value above unit m only ever depends on units below it, so the
// unused units never reach the result.  At the end D[m][n] = n + sum_i (VP_i - VN_i) over the m units.
//
// Words: a hypothesis word is buffered in the warp's shared row (only up to the longest reference word: a longer one
// cannot match) and compared label by label against the reference's distinct words, one per lane; its symbol is the
// index of the equal distinct word, or -1 (a word that matches no reference word).
//
// Every value is one fixed sequence of integer and compare operations on the row's logits: bit-identical for any batch
// position, tile or GPU count.
#pragma once
#include "common.cuh"
#include "../../include/w2s.h"

namespace w2s {

constexpr int ERR_LANES = 16;   // 32-bit words of a match mask: 512 units = W2S_MAX_TRANSCRIPT
constexpr int ERR_HDR = 8;      // ints per reference header

// Tables of the references (host-built, error_tables in api.cu), one int32 array `tab`:
//   header d at tab[ERR_HDR d]: m (units), the tab index of its first match-mask row, the tab index of its first
//   distinct-word record, the number of distinct words, the length of its longest word (words unit), then zeros;
//   distinct-word record j: (tab index of its labels, length);
//   match-mask rows of ERR_LANES words: bit i % 32 of word i / 32 set when reference unit i is the row's symbol (a label
//   id, or a distinct-word index).

// argmax over the vocabulary of one frame held one-per-lane (logit[j] = entry lane + 32 j); ties go to the lowest id
template <int J>
__device__ __forceinline__ int err_argmax(const float (&logit)[J], int V, int lane) {
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j)
    if (lane + 32 * j < V) mx = fmaxf(mx, logit[j]);
  mx = warp_max(mx);
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const unsigned b = __ballot_sync(0xffffffffu, lane + 32 * j < V && logit[j] == mx);
    if (b) return 32 * j + __ffs(b) - 1;
  }
  return 0;   // only for NaN rows
}

// one column of the edit-distance matrix for a hypothesis symbol whose match mask over this lane's 32 units is eq
__device__ __forceinline__ void err_step(uint32_t eq, uint32_t& vp, uint32_t& vn, int lane) {
  const uint32_t x = eq | vn;
  // (x & vp) + vp over 512 bits: lane k's carry-in is 1 when some lower lane generates a carry that every lane in
  // between propagates -- bit k of (g + (g | p)) ^ p, g and p never both set in one lane
  const uint32_t s = (x & vp) + vp;
  const unsigned g = __ballot_sync(0xffffffffu, s < vp);
  const unsigned p = __ballot_sync(0xffffffffu, s == 0xffffffffu);
  const uint32_t d0 = ((s + (((g + (g | p)) ^ p) >> lane & 1u)) ^ vp) | x;
  const uint32_t hn = vp & d0;
  const uint32_t hp = vn | ~(vp | d0);
  // horizontal deltas shifted up by one unit: lane k takes lane k - 1's top bit; above unit 0 the delta is +1
  const unsigned tp = __ballot_sync(0xffffffffu, hp >> 31);
  const unsigned tn = __ballot_sync(0xffffffffu, hn >> 31);
  const uint32_t hps = (hp << 1) | (((tp << 1) | 1u) >> lane & 1u);
  const uint32_t hns = (hn << 1) | ((tn << 1) >> lane & 1u);
  vn = hps & d0;
  vp = hns | ~(hps | d0);
}

// Edit distance between the greedy transcript of T frames and reference d.  frame(t, logit) loads frame t one-per-lane
// (-inf past V).  wbuf: this warp's shared scratch of at least W2S_MAX_TRANSCRIPT ints (words unit).  Every lane returns
// the result.
template <int J, class Frame>
__device__ int errors_warp(int T, int V, const int* __restrict__ tab, int d, int unit, int blank, int delim, int lane,
                           int* wbuf, Frame frame) {
  const int* hdr = tab + ERR_HDR * d;
  const int m = __ldg(hdr), dw = __ldg(hdr + 2), nd = __ldg(hdr + 3), maxw = __ldg(hdr + 4);
  const uint32_t* rows = reinterpret_cast<const uint32_t*>(tab + __ldg(hdr + 1));
  uint32_t vp = 0xffffffffu, vn = 0u;   // D[i][0] = i: every vertical delta +1
  int n = 0, prev = -1, wlen = 0;       // hypothesis symbols so far, previous frame's argmax, labels of the open word
  auto consume = [&](int sym) {
    const uint32_t eq = sym >= 0 && lane < ERR_LANES ? __ldg(rows + sym * ERR_LANES + lane) : 0u;
    err_step(eq, vp, vn, lane);
    ++n;
  };
  auto end_word = [&]() {
    if (wlen == 0) return;   // empty words (leading, trailing or repeated delimiters) are no words
    __syncwarp();
    int sym = -1;
    for (int j0 = 0; wlen <= maxw && j0 < nd; j0 += 32) {
      const int j = j0 + lane;
      bool same = false;
      if (j < nd) {
        const int st = __ldg(tab + dw + 2 * j);
        same = __ldg(tab + dw + 2 * j + 1) == wlen;
        for (int i = 0; same && i < wlen; ++i) same = __ldg(tab + st + i) == wbuf[i];
      }
      const unsigned b = __ballot_sync(0xffffffffu, same);
      if (b) {
        sym = j0 + __ffs(b) - 1;
        break;
      }
    }
    consume(sym);
    wlen = 0;
    __syncwarp();   // the compare has read the word before the next one is written
  };
  for (int t = 0; t < T; ++t) {
    float logit[J];
    frame(t, logit);
    const int a = err_argmax(logit, V, lane);
    if (a != prev && a != blank) {
      if (unit == W2S_ERR_LABELS) {
        consume(a);
      } else if (a == delim) {
        end_word();
      } else {
        if (wlen < maxw && lane == 0) wbuf[wlen] = a;
        ++wlen;
      }
    }
    prev = a;
  }
  if (unit == W2S_ERR_WORDS) end_word();
  const int lo = 32 * lane;
  const uint32_t keep = m >= lo + 32 ? 0xffffffffu : m > lo ? (1u << (m - lo)) - 1u : 0u;
  const int r = n + (int)__reduce_add_sync(0xffffffffu, (unsigned)(__popc(vp & keep) - __popc(vn & keep)));
  __syncwarp();   // wbuf may be reused by the caller's next item
  return r;
}

}  // namespace w2s
