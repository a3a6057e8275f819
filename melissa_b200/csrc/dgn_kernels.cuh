// Device kernels shared by the fp32 and bf16 forward paths of the DGN Q-networks.
//
// Math follows the reference networks and the third-party ops they call:
//   graph_env/env/utils/networks/common.py:31-63  (obs split, radius_graph, ctrl index)
//   graph_env/env/utils/networks/{l_dgn.py:117-149, dgn_r.py:98-127, hl_dgn.py:97-117}
//   PyG GATv2Conv / TransformerConv / softmax / global_*_pool, torch_cluster radius,
//   tianshou MLP + DQNPolicy.forward / exploration_noise  (SURVEY.md Appendix B).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

// bf16 tensor-core path (dgn_forward_bf16.cu)
size_t dgn_workspace_bytes_bf16(const MlsNetDesc* d, int n_graphs);
int dgn_forward_bf16(const MlsNetDesc* d, const MlsNetWeights* w, const MlsForwardArgs* a, void* stream);
int dgn_prepare_bf16(const MlsNetDesc* d, const MlsNetWeights* w, int flags, void* workspace, size_t workspace_bytes, void* stream);
size_t dgn_csr_cache_bytes(const MlsNetDesc* d, int n_pool_graphs);
int dgn_csr_cache_build(const MlsNetDesc* d, const float* pos_obs, int64_t obs_stride, int n_pool_graphs, void* cache, size_t cache_bytes,
                        void* stream);

namespace mls {

constexpr int kC = 128;                 // channels per head the edge kernels are written for
constexpr int kMaxNbr = 32;             // torch_cluster radius_graph max_num_neighbors
// radius_graph(loop=False) keeps the first max_num_neighbors + 1 hits and then drops the self hit: a node that is not among
// the first 33 hits of its own scan (index > 32 with more than 33 nodes in reach) keeps 33 sources, one more than
// max_num_neighbors.  A source list therefore holds up to kMaxList entries (plus the GATv2 self loop where that is added).
constexpr int kMaxList = kMaxNbr + 1;
// bytes of one graph's CSR source lists (uint8 ids), a multiple of 16: N * 32 while no node can have 33 sources (N <= 33),
// else N * 33 rounded up
__host__ __device__ constexpr int csr_stride(int N) { return N <= kMaxList ? N * kMaxNbr : (N * kMaxList + 15) & ~15; }
__device__ __forceinline__ float r2_threshold() { return (float)(0.2 * 0.2); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Neighbour set of target node i in graph with node rows at `g_obs` (N rows of 8 floats):
// radius_graph(pos, r=0.2, loop=False, max_num_neighbors=32) -- candidates scanned in index
// order, kept while fma(dy,dy,dx*dx) < r*r in fp32, scan stops after 33 hits (self
// included), self dropped.  Warp-cooperative; result words are warp-uniform.
template <int W>
__device__ __forceinline__ void radius_neighbours(const float* __restrict__ g_obs, int N, int i, int lane,
                                                  uint32_t (&nb)[W], const int stride = 8) {
  // `stride` floats between node rows: 8 for observation rows, 2 for a staged (x, y) array
  const float xi = g_obs[i * stride + 0], yi = g_obs[i * stride + 1];
  const float thr = r2_threshold();
  int total = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const int j = w * 32 + lane;
    bool hit = false;
    if (j < N) {
      const float dx = g_obs[j * stride + 0] - xi, dy = g_obs[j * stride + 1] - yi;
      const float d2 = __fmaf_rn(dy, dy, __fmul_rn(dx, dx));
      hit = d2 < thr;
    }
    nb[w] = __ballot_sync(0xffffffffu, hit);
    total += __popc(nb[w]);
  }
  if (total > kMaxNbr + 1) {          // keep the first 33 hits in index order
    int keep = kMaxNbr + 1;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      const int c = __popc(nb[w]);
      if (c <= keep) { keep -= c; }
      else {
        uint32_t m = nb[w], out = 0;
        for (int t = 0; t < keep; ++t) { out |= m & (0u - m); m &= m - 1; }
        nb[w] = out;
        keep = 0;
      }
    }
  }
#pragma unroll
  for (int w = 0; w < W; ++w) if (w == (i >> 5)) nb[w] &= ~(1u << (i & 31));
}

struct ActArgsB {
  float eps;
  uint64_t seed, offset;
  const double* rand3;
  const unsigned long long* offset_dev;   // optional device-side addend (round counter under CUDA-graph replay)
  uint64_t row0;                          // added to the row index that keys the Philox draw (sub-batch calls)
};
__device__ __forceinline__ int select_action_b(float q0, float q1, const ActArgsB& a, uint64_t row) {
  int act = q1 > q0 ? 1 : 0;
  if (fabsf(a.eps) > 1e-8f) {
    double ue, u0, u1;
    if (a.rand3) { ue = a.rand3[row * 3 + 0]; u0 = a.rand3[row * 3 + 1]; u1 = a.rand3[row * 3 + 2]; }
    else {
      Philox4 r = philox4x32_10(a.seed, row + a.row0, a.offset + (a.offset_dev ? *a.offset_dev : 0ull));
      ue = u01_from_u32x2(r.v[0], r.v[1]);
      u0 = (double)r.v[2] * (1.0 / 4294967296.0);
      u1 = (double)r.v[3] * (1.0 / 4294967296.0);
    }
    if (ue < (double)a.eps) act = (u1 + 1.0) > (u0 + 1.0) ? 1 : 0;
  }
  return act;
}

// Output layer of the 128-wide dueling heads for one row t, from the three dot products of its rectified last hidden layer
// (d_q0 = <relu(hq), wq[0]>, d_v = <relu(hv), wv>, d_q1 = <relu(hq), wq[1]>): biases, dueling combination, output row
// mapping and action.  Same outputs as head_out_bf16_kernel.
struct HeadOut {
  const float *bq, *bv;
  const int* idx;             // out_mode 0 / 1: row t is node row idx[t] of the pass
  int64_t row0;               // first node row of the pass (out_mode 0 / 1)
  int per_graph_N;
  float* q_out;
  int8_t* act_out;
  int out_mode;               // 0: per node row, 1: per graph (of the node row), 2: row t (HL-DGN graph rows, no action)
  ActArgsB aa;
};
__device__ __forceinline__ void head_final_row(int t, float d_q0, float d_v, float d_q1, const HeadOut& h) {
  const float s0 = d_q0 + h.bq[0], sv = d_v + h.bv[0], s1 = d_q1 + h.bq[1];
  const float mean = (s0 + s1) / 2.0f;
  const float o0 = (s0 - mean) + sv, o1 = (s1 - mean) + sv;
  int64_t orow;
  if (h.out_mode == 0) orow = h.row0 + h.idx[t];
  else if (h.out_mode == 1) orow = h.row0 / h.per_graph_N + h.idx[t] / h.per_graph_N;
  else orow = t;
  h.q_out[orow * 2 + 0] = o0;
  h.q_out[orow * 2 + 1] = o1;
  if (h.act_out && h.out_mode != 2) h.act_out[orow] = (int8_t)select_action_b(o0, o1, h.aa, (uint64_t)orow);
}

}  // namespace mls
