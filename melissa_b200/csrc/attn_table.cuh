// Table-mode attention convolution on the tensor cores (discrete node features), see attn_table.cu.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace mls {

constexpr int kAttnUcap = 1024;      // distinct feature keys per pass the pair-logit table is sized for
constexpr int kAttnMaxRows = 62;     // node rows per tile (one 64-wide K panel of the weight matrix, 2 columns for the bias)

struct AttnTableArgs {
  // projection tables over all feature keys (MLS_FWD_DISCRETE_FEATURES)
  const __nv_bfloat16* t_P;  // [n_keys][ldp]  GATv2 [x_l | x_r], Transformer [q | k | v]
  int ldp;
  const float* t_ab;         // GATv2 [n_keys][2H]: <att_h, x_l>, <att_h, x_r>
  const float* att;          // GATv2 [H*C]
  const float* bias;         // GATv2 conv bias [H*C]; NULL for the Transformer conv
  int transformer;
  // this pass
  const uint32_t* key;       // [rows] feature key of every node row
  int N, H, n_graphs;
  const uint16_t* csr_ptr;   // [graphs][N+1]
  const uint8_t* csr_src;    // [graphs][csr_stride(N)]
  // optional "needed" row map (ctrl_need_list_kernel): x_out row of every node row, -1 = nobody reads this node's
  // conv output (its softmax weights are not even built)
  const int* xrow;
  // CSR lists of graph g live at index graph_id[g * gid_stride] (topology cache of a static graph pool), else at g
  const int* graph_id;
  int gid_stride;
  __nv_bfloat16* x_out;      // [rows][H*C] relu(conv)  (or [needed rows][H*C] with xrow)
  // HL-DGN: pool_mode >= 0 (enum MlsPool): instead of x_out, z[graph][z_col + H*C] = pool over the graph's nodes of
  // relu(conv) * dm, dm = obs column 7 (one graph per tile)
  int pool_mode;
  __nv_bfloat16* z;
  int ldz, z_col;
  const float* obs;
  long long obs_stride;
  // scratch (workspace)
  uint32_t* used_bits;       // [n_keys / 32] bitmap marked by feature_key_kernel, cleared here
  int n_keys;
  uint16_t* cid_of_key;      // [n_keys] compact id of a key present in this pass (0xFFFF otherwise)
  uint32_t* key_of_cid;      // [kAttnUcap]
  uint16_t* row_cid;         // [rows] compact id of every node row
  int* n_used;               // [1] number of distinct keys; > kAttnUcap: the caller's gather kernel runs instead
  void* Vh;                  // [kAttnUcap][H*C] fp16 value rows of the present keys (by compact id)
  float* E;                  // [kAttnUcap][kAttnUcap][4] base-2 logits of (target key, source key) for the 4 heads
  // x_out (pool_mode < 0): per-tile records written by the pre-pass, attn_table_record_bytes() bytes, and
  // {padded entry count, needed targets} of every tile
  unsigned char* rec;
  int2* tile_idx;            // [tiles]
};

// scratch bytes behind `E`
inline size_t attn_table_pair_bytes() { return (size_t)kAttnUcap * kAttnUcap * 4 * sizeof(float); }
inline size_t attn_table_value_bytes() { return (size_t)kAttnUcap * 512 * 2; }
// true when this (N, H) can take the tensor-core path at all
inline bool attn_table_supported(int N, int H) { return N >= 1 && N <= kAttnMaxRows && H == 4; }

// bytes behind `rec` for a pass of n_graphs graphs of N nodes
size_t attn_table_record_bytes(int N, int n_graphs);
int attn_table_conv_launch(const AttnTableArgs& a, int sm_count, cudaStream_t st);

}  // namespace mls
