// Second attention convolution (conv2) of L-DGN / DGN-R on the compacted row sets, see conv2_attn.cu.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace mls {

constexpr int kConv2MaxNodes = 64;   // graphs of up to 64 nodes: one 64-row K panel of sources, up to 64 targets

struct Conv2Args {
  // source side, one row per NEEDED node (a controlling node or a source of one), fp16:
  //   GATv2 [x_l] (lds >= H*C), Transformer [k | v] (lds >= 2*H*C)
  const __half* Ps;
  int lds;
  // target side, one row per controlling node (slot order), fp16: GATv2 x_r, Transformer q
  const __half* Pt;
  int ldt;
  const float* as;       // GATv2 [needed rows][H]: <att_h, x_l[row, h]>
  const float* bt;       // GATv2 [slots][H]:       <att_h, x_r[slot, h]>
  const float* att;      // GATv2 [H*C]
  const float* bias;     // GATv2 conv bias [H*C]; NULL for the Transformer conv
  int transformer;
  int N, H, n_graphs;
  // row sets and edge lists (ctrl_need_list_kernel): the slots / needed rows / edge entries of graph g are consecutive
  //   gmeta[g] = {first slot, controlling nodes, first other needed row, needed rows, first edge entry, edge entries, 0, 0}
  //   needed rows are ordered [controlling nodes by slot][the others]: source k of graph g (compact index, controlling
  //   nodes first) lives in row first slot + k for k < controlling nodes, else gmeta[2] + k - controlling nodes
  //   eabs[slot] = position of the slot's first edge entry (its entries run to the next slot's, the last to the block end)
  //   eent[e]    = compact source index (rank in the graph's needed list) | target index within the graph << 8;
  //                the GATv2 self loop is an ordinary entry; blocks start 16-byte aligned
  const int* gmeta;
  const int* eabs;
  const uint16_t* eent;
  // output: relu(conv2)[slot] as bf16 at z[slot][z_col + h*C ...]
  __nv_bfloat16* z;
  int ldz, z_col;
};

inline bool conv2_attn_supported(int N, int H) { return N >= 1 && N <= kConv2MaxNodes && H >= 1; }
int conv2_attn_launch(const Conv2Args& a, int sm_count, cudaStream_t st);

}  // namespace mls
