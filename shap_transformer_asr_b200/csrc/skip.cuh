// Constant-frame skip of the feature encoder (frontend_skip.cu): block lists built on the device per tile.
#pragma once
#include "kernels.cuh"

namespace w2s {

constexpr int SKIP_MAX_LAYERS = 8;

// Layer index l here is conv layer l + 1.  Lists: [0] = count, then entries (coalition << 16) | 128-row block.
struct SkipParams {
  const DynArgs* dyn;                 // keep bits of the tile's coalitions
  const int4* tab;                    // w2s_frontend_blocks rows (segment range, input block range)
  int nl, n, total;                   // layers, coalitions, table rows
  int nb[SKIP_MAX_LAYERS];            // blocks per coalition
  int off[SKIP_MAX_LAYERS];           // first table row of the layer
  int dense[SKIP_MAX_LAYERS];         // 1: the layer's contraction runs dense (every block live, nothing to fill)
  int* live[SKIP_MAX_LAYERS];         // blocks to contract   [1 + n * nb]
  int* fill[SKIP_MAX_LAYERS];         // blocks to copy the representative row into   [1 + n * nb]
  int* rep;                           // [nl][n] representative block (all constant, contracted)
};

std::string launch_skip_lists(const SkipParams& p, cudaStream_t s);
std::string launch_skip_fill(const int* fill, const int* rep, __nv_bfloat16* buf, int T, int C, int num_sms, cudaStream_t s);

}  // namespace w2s
