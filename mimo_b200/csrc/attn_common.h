// Shared declarations of the spatial-attention kernels. mimo_attn_spatial (attn_spatial.cu) picks one by head dim:
//   d + 1 <= 64 : attn_spatial_pp2.cu - two Q tiles per CTA in ping-pong, two softmax threads per query row
//   dp <= 128   : attn_spatial_pp.cu  - two Q tiles per CTA in ping-pong, one softmax thread per query row
//   otherwise   : attn_spatial.cu     - one Q tile per CTA, head dim up to 192
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

namespace mimo {

constexpr int BQ = 128;                 // query rows per tile
constexpr int BKV = 128;                // keys per tile
constexpr int kChunkBytes = 128 * 128;  // one 64-element-wide (128 B) chunk of a 128-row tile

struct AttnArgs {
  int lq, lb, heads, d, dp;  // dp = d rounded up to 16
  int n_self_tiles, n_bank_tiles;
  float scale_log2;
  const int* bank_index;
  void* out;
  long long ld_out;
};

// two Q tiles per CTA (grid.x = ceil(lq / 256)); dp <= 128
int launch_attn_pp(bool bf16, const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const CUtensorMap& bk,
                   const CUtensorMap& bv, const AttnArgs& a, int n, cudaStream_t st);

// two softmax threads per query row, row sum by the tensor pipe (attn_spatial_pp2.cu); d + 1 <= 64
int launch_attn_pp2(bool bf16, const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const CUtensorMap& bk,
                    const CUtensorMap& bv, const AttnArgs& a, int n, cudaStream_t st);

}  // namespace mimo
