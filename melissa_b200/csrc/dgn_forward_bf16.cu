// bf16 tensor-core forward of DGN-R / L-DGN / HL-DGN (sm_100a).
//
// Dense layers run on the tcgen05 GEMM (gemm_tcgen05.cu) with fused bias / ReLU / decision-maker
// row mask (and the linear parts of the GATv2 logits); the attention convolutions run one CTA per
// (graph, head) with that head's operands staged in shared memory (every x_l / x_r / k / v row is
// read from global memory once per head instead of once per edge) over CSR neighbour lists built
// once per pass; controlling-node snapshots and the HL-DGN graph pooling are written by the same
// kernels.  The only activations in global memory are bf16 rows in a workspace that is reused
// pass after pass (a pass = mls_dgn_chunk_graphs() graphs).
//
// Accumulation is fp32 everywhere; activations and weights are rounded to bf16
// (tolerance stated in tests/test_networks_gpu.py).  Reference math: see dgn_forward.cu.
#include <algorithm>

#include "dgn_kernels.cuh"
#include "gemm_tcgen05.cuh"
#include "attn_table.cuh"
#include "conv2_attn.cuh"

namespace mls {

typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------ weight preparation
struct CvtJob {
  const float* src;   // [rows, cols] fp32 row major
  bf16* dst;          // destination matrix base
  int rows, cols, ld_dst, row_off, col_off;
};
struct CvtJobs {
  CvtJob j[8];
  int n;
};
__global__ void cvt_weights_kernel(const CvtJobs jobs) {
  const CvtJob jb = jobs.j[blockIdx.y];
  const long long total = (long long)jb.rows * jb.cols;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(t / jb.cols), c = (int)(t - (long long)r * jb.cols);
    jb.dst[(size_t)(r + jb.row_off) * jb.ld_dst + c + jb.col_off] = __float2bfloat16_rn(jb.src[t]);
  }
}
struct CatJobs {
  const float* src[12];
  float* dst[12];
  int n[12];
  int count;
};
__global__ void cat_bias_kernel(const CatJobs jobs) {
  const int k = blockIdx.y;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < jobs.n[k]; t += gridDim.x * blockDim.x) jobs.dst[k][t] = jobs.src[k][t];
}

// ------------------------------------------------------------------------------ encoder layer 0
// h = relu(W0 f + b0), f = obs cols 2..6.  16 threads per node row (8 channels each, one 16 B store),
// W0 / b0 in shared memory.
__global__ void __launch_bounds__(256) enc0_bf16_kernel(const float* __restrict__ obs, int64_t obs_stride, int N, int rows, int in_dim,
                                                        const float* __restrict__ w0, const float* __restrict__ b0, int hidden,
                                                        bf16* __restrict__ h) {
  __shared__ float w_s[kC * 5 + kC];
  for (int t = threadIdx.x; t < hidden * in_dim; t += 256) w_s[t] = w0[t];
  for (int t = threadIdx.x; t < hidden; t += 256) w_s[kC * 5 + t] = b0[t];
  __syncthreads();
  const int per_row = hidden / 8;                      // threads per row
  const int rows_per_cta = 256 / per_row;
  const int r = blockIdx.x * rows_per_cta + threadIdx.x / per_row;
  if (r >= rows) return;
  const int c0 = (threadIdx.x % per_row) * 8;
  const int g = r / N, i = r - g * N;
  const float* f = obs + (int64_t)g * obs_stride + i * 8 + 2;
  float fv[5];
#pragma unroll
  for (int k = 0; k < 5; ++k) fv[k] = k < in_dim ? f[k] : 0.f;
  uint32_t packed[4];
#pragma unroll
  for (int c = 0; c < 8; c += 2) {
    float a0 = w_s[kC * 5 + c0 + c], a1 = w_s[kC * 5 + c0 + c + 1];
    for (int k = 0; k < in_dim; ++k) {
      a0 = fmaf(w_s[(c0 + c) * in_dim + k], fv[k], a0);
      a1 = fmaf(w_s[(c0 + c + 1) * in_dim + k], fv[k], a1);
    }
    __nv_bfloat162 p = __floats2bfloat162_rn(fmaxf(a0, 0.f), fmaxf(a1, 0.f));
    packed[c >> 1] = *reinterpret_cast<uint32_t*>(&p);
  }
  *reinterpret_cast<uint4*>(h + (size_t)r * hidden + c0) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
}

// ------------------------------------------------------------------------------ discrete-feature table
// The encoder input of a node is five small integers (obs cols 2..6: degree, messages transmitted, last
// action, interested, has-message; reference graph.py:263-269), so x0 = encoder(f) and the conv1
// projections [x_l | x_r] (or [q | k | v]) take only a few thousand distinct values.  In "discrete
// features" mode they are computed ONCE per forward for every possible key and the conv1 attention
// kernel gathers its rows from that table (L2 resident) instead of a per-node GEMM result in HBM.
//   key = ((((deg << 6) | msgs) << 1 | action) << 1 | interested) << 1 | has_message
__device__ __forceinline__ void key_decode(uint32_t key, float (&f)[5]) {
  f[4] = (float)(key & 1u); f[3] = (float)((key >> 1) & 1u); f[2] = (float)((key >> 2) & 1u);
  f[1] = (float)((key >> 3) & 63u); f[0] = (float)(key >> 9);
}
__global__ void feature_key_kernel(const float* __restrict__ obs, int64_t obs_stride, int N, int rows, int degbits,
                                   uint32_t* __restrict__ key, int* __restrict__ errors, uint32_t* __restrict__ used_bits) {
  extern __shared__ uint32_t s_bits[];         // (1 << degbits) * 16 words when used_bits != NULL
  const int n_words = (1 << degbits) * 16;
  if (used_bits) {
    for (int w = threadIdx.x; w < n_words; w += blockDim.x) s_bits[w] = 0;
    __syncthreads();
  }
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < rows) {
    const int g = r / N, i = r - g * N;
    const float* f = obs + (int64_t)g * obs_stride + i * 8 + 2;
    const float deg = f[0], msgs = f[1], act = f[2], intr = f[3], hm = f[4];
    const bool ok = deg >= 0.f && deg < (float)(1 << degbits) && deg == floorf(deg) && msgs >= 0.f && msgs < 64.f &&
                    msgs == floorf(msgs) && (act == 0.f || act == 1.f) && (intr == 0.f || intr == 1.f) && (hm == 0.f || hm == 1.f);
    uint32_t k = 0;
    if (ok) k = (((((uint32_t)deg << 6) | (uint32_t)msgs) << 1 | (uint32_t)act) << 1 | (uint32_t)intr) << 1 | (uint32_t)hm;
    else if (errors) atomicAdd(errors, 1);
    key[r] = k;
    if (used_bits) atomicOr(&s_bits[k >> 5], 1u << (k & 31));   // keys present in this pass (attn_table.cu compacts them)
  }
  if (used_bits) {
    __syncthreads();
    for (int w = threadIdx.x; w < n_words; w += blockDim.x) {
      const uint32_t b = s_bits[w];
      if (b && (used_bits[w] & b) != b) atomicOr(&used_bits[w], b);
    }
  }
}
__global__ void __launch_bounds__(256) enc0_keys_kernel(int n_keys, int in_dim, const float* __restrict__ w0,
                                                        const float* __restrict__ b0, int hidden, bf16* __restrict__ h) {
  __shared__ float w_s[kC * 5 + kC];
  for (int t = threadIdx.x; t < hidden * in_dim; t += 256) w_s[t] = w0[t];
  for (int t = threadIdx.x; t < hidden; t += 256) w_s[kC * 5 + t] = b0[t];
  __syncthreads();
  const int per_row = hidden / 8, rows_per_cta = 256 / per_row;
  const int r = blockIdx.x * rows_per_cta + threadIdx.x / per_row;
  if (r >= n_keys) return;
  const int c0 = (threadIdx.x % per_row) * 8;
  float fv[5];
  key_decode((uint32_t)r, fv);
  uint32_t packed[4];
#pragma unroll
  for (int c = 0; c < 8; c += 2) {
    float a0 = w_s[kC * 5 + c0 + c], a1 = w_s[kC * 5 + c0 + c + 1];
    for (int k = 0; k < in_dim; ++k) {
      a0 = fmaf(w_s[(c0 + c) * in_dim + k], fv[k], a0);
      a1 = fmaf(w_s[(c0 + c + 1) * in_dim + k], fv[k], a1);
    }
    __nv_bfloat162 p = __floats2bfloat162_rn(fmaxf(a0, 0.f), fmaxf(a1, 0.f));
    packed[c >> 1] = *reinterpret_cast<uint32_t*>(&p);
  }
  *reinterpret_cast<uint4*>(h + (size_t)r * hidden + c0) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
}

// ------------------------------------------------------------------------------ graph CSR
// radius_graph(pos, r=0.2, loop=False, max_num_neighbors=32) once per chunk and graph, as source
// lists per target: csr_ptr[g][N+1] (uint16 offsets into the graph's list), csr_src[g][csr_stride(N)] (uint8
// source node ids, index order; up to 33 per target, see kMaxList).  Self loops are NOT stored (GATv2 adds its own).  The lists are
// shared by all heads and by both conv layers.  One CTA per graph.
template <int W>
__global__ void __launch_bounds__(256) graph_csr_kernel(const float* __restrict__ obs, int64_t obs_stride, int N, int n_graphs,
                                                        uint16_t* __restrict__ csr_ptr, uint8_t* __restrict__ csr_src,
                                                        uint32_t* __restrict__ adj_out) {
  extern __shared__ __align__(16) unsigned char csm[];
  uint32_t* s_mask = reinterpret_cast<uint32_t*>(csm);      // [N][W]
  int* s_ptr = reinterpret_cast<int*>(s_mask + (size_t)N * W);   // [N+1]
  float* s_pos = reinterpret_cast<float*>(s_ptr + N + 1);   // [N][2]: one trip to global memory for the positions
  const int g = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const float* g_obs = obs + (int64_t)g * obs_stride;
  for (int t = threadIdx.x; t < 2 * N; t += blockDim.x) s_pos[t] = g_obs[(t >> 1) * 8 + (t & 1)];
  __syncthreads();
  for (int i = warp; i < N; i += nwarps) {
    uint32_t nb[W];
    radius_neighbours<W>(s_pos, N, i, lane, nb, 2);
    int deg = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      deg += __popc(nb[w]);
      if (lane == w) s_mask[i * W + w] = nb[w];
    }
    if (lane == 0) s_ptr[i + 1] = deg;
  }
  __syncthreads();
  if (warp == 0) {                                          // exclusive scan of the degrees
    int run = 0;
    for (int c0 = 0; c0 < N; c0 += 32) {
      const int idx = c0 + lane;
      int v = idx < N ? s_ptr[idx + 1] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
      }
      if (idx < N) s_ptr[idx + 1] = run + v;
      run += __shfl_sync(0xffffffffu, v, 31);
    }
    if (lane == 0) s_ptr[0] = 0;
  }
  __syncthreads();
  uint16_t* gp = csr_ptr + (size_t)g * (N + 1);
  uint8_t* gs = csr_src + (size_t)g * csr_stride(N);
  for (int t = threadIdx.x; t <= N; t += blockDim.x) gp[t] = (uint16_t)s_ptr[t];
  if (adj_out) for (int t = threadIdx.x; t < N * W; t += blockDim.x) adj_out[(size_t)g * N * W + t] = s_mask[t];   // source masks per target
  for (int i = warp; i < N; i += nwarps) {
    int off = s_ptr[i];
#pragma unroll
    for (int w = 0; w < W; ++w) {
      const uint32_t m = s_mask[i * W + w];
      if ((m >> lane) & 1u) gs[off + __popc(m & ((1u << lane) - 1u))] = (uint8_t)(w * 32 + lane);
      off += __popc(m);
    }
  }
}

// ------------------------------------------------------------------------------ attention convolutions
struct EdgeArgs {
  const bf16* P;          // [rows, ldp] projections: GATv2 [x_l | x_r], Transformer [q | k | v]
  int ldp;
  const float* obs;       // chunk base
  int64_t obs_stride;
  int N, H, n_graphs;
  const uint16_t* csr_ptr; // [graphs][N+1]
  const uint8_t* csr_src;  // [graphs][csr_stride(N)]
  const float* ab;        // GATv2: [rows][2H] = (<att_h, x_l[row,h]>, <att_h, x_r[row,h]>) from the projection GEMM
  const uint32_t* row_key; // optional [rows]: P / ab are tables indexed by row_key[row] (discrete-feature mode), else by row
  const float* att;       // GATv2 [H*C]
  const float* bias;      // GATv2 [H*C]
  bf16* x_out;            // [rows, H*C] relu(conv) for every node, or NULL
  const int* slot;        // [rows] index of the node in the controlling list, -1 if none; or NULL
  bf16* z;                // snapshot destination rows [*, ldz], written at column z_col for slot >= 0; or NULL
  int ldz, z_col;
  int ctrl_only;          // compute only nodes with slot >= 0
  int pool_mode;          // >= 0: HL-DGN pooling of relu(conv)*dm into z[g][H*C] (enum MlsPool); -1 none
  // optional compact target side (conv2: only controlling nodes are targets).  Pt row (slot of node i) holds the
  // target projection (GATv2 x_r, Transformer q) of node i, bt[slot][H] the <att, x_r> dots; the slots of graph g
  // are gfirst[g] .. gfirst[g] + gcnt[g] - 1 in node order.  P then holds only the source side:
  // GATv2 [x_l] (ab = [rows][H]), Transformer [k | v].
  const bf16* Pt;
  int ldpt;
  const float* bt;
  const int* gfirst;
  const int* gcnt;
  const int* idx;         // [slots] node row of every slot (compact mode: the warps walk the target list, evenly split)
  const int* run_if_gt;   // optional device int: the kernel only runs when *run_if_gt > run_thresh
  int run_thresh;         // (fallback behind the tensor-core table kernel, attn_table.cu)
  // "needed" row sets (ctrl_need_list_kernel): xrow[node row] = compact row of a node that some later stage reads, -1 else.
  //   xrow_out: x_out rows are written at xrow_out[row]; targets with -1 are skipped altogether (conv1)
  //   xrow_src: P / ab hold one row per needed node, indexed by xrow_src[row] (conv2, compact target mode)
  const int* xrow_out;
  const int* xrow_src;
  // CSR lists of graph g live at index graph_id[g * gid_stride] (topology cache of a static graph pool), else at g
  const int* graph_id;
  int gid_stride;
};

// CTA size: 128 threads, 5-6 CTAs per SM (register bound), so that the staging of one CTA overlaps the compute of the
// others.  The operands are staged as bf16 (2-3 x 12.8 KB for 50-node graphs), shared memory is no longer the limit.
template <bool TRANSFORMER> struct EdgeCfg {
  static constexpr int kThreads = 128;
  static constexpr int kMinCtas = TRANSFORMER ? 6 : 5;      // measured: 5 CTAs (96 registers) beat 4 by 9 % for GATv2, 6 spill
};


__device__ __forceinline__ void edge_cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void edge_cp_async_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// 8 bf16 -> two float4 (exact: a bf16 is the upper half of an fp32)
__device__ __forceinline__ void bf16x8_to_f32(const uint4 u, float4& lo, float4& hi) {
  lo = make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
  hi = make_float4(__uint_as_float(u.z << 16), __uint_as_float(u.z & 0xffff0000u), __uint_as_float(u.w << 16), __uint_as_float(u.w & 0xffff0000u));
}
__device__ __forceinline__ uint32_t pack_bf16x2_rn(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// One CTA per (graph, head).
//   phase 0  stage the head's operands in shared memory as raw bf16 rows with cp.async, together with the graph's
//            CSR block and the per-node scalars
//   phase 1  one warp per target, FOUR neighbours per round (two lane groups x two independent chains), SIXTEEN
//            lanes per neighbour (8 channels each); the target's 8 channels stay in registers, every neighbour
//            row is read from shared memory exactly once and serves both its logit and its contribution to the
//            output (single-pass softmax in base 2: running max / denominator, same value as PyG's
//            exp(e - max) / (sum + 1e-16) up to rounding); the two lane groups are combined with 9 shuffles and
//            group 0 writes 256 contiguous bytes per target.
//              GATv2:       e_ij = 0.6 (a_j + b_i) + 0.4 sum_c att_c |x_l[j,c] + x_r[i,c]|   (leaky_relu(s,.2) = .6 s + .4 |s|)
//              Transformer: e_ij = <q_i, k_j> / sqrt(C)
template <bool TRANSFORMER>
__global__ void __launch_bounds__(EdgeCfg<TRANSFORMER>::kThreads, EdgeCfg<TRANSFORMER>::kMinCtas) edge_bf16_kernel(const EdgeArgs a) {
  constexpr int kEdgeThreads = EdgeCfg<TRANSFORMER>::kThreads, kEdgeWarps = kEdgeThreads / 32;
  extern __shared__ __align__(16) unsigned char esm[];
  const int N = a.N, H = a.H, HC = H * kC;
  // operands staged as raw bf16 rows (cp.async, converted at use: a bf16 is the upper half of an fp32)
  bf16* stT = reinterpret_cast<bf16*>(esm);                                      // [N][kC]  x_r or q (target side)
  bf16* stA = stT + N * kC;                                                      // [N][kC]  x_l or k (source side)
  bf16* stB = stA + N * kC;                                                      // [N][kC]  v (Transformer)
  float* s_a = reinterpret_cast<float*>(stB + (TRANSFORMER ? N * kC : 0));       // [N] <att, x_l[j]> * 0.6 log2e
  float* s_b = s_a + N;                                                          // [N] <att, x_r[i]> * 0.6 log2e
  float* s_dm = s_b + N;                                                         // [N]
  int* s_slot = reinterpret_cast<int*>(s_dm + N);                                // [N]
  float* poolbuf = reinterpret_cast<float*>(s_slot + N);                         // [warps][kC]  (16 B aligned: 4N floats before it)
  uint8_t* s_src = reinterpret_cast<uint8_t*>(poolbuf + (a.pool_mode >= 0 ? kEdgeWarps * kC : 0));     // [csr_stride(N)] (16 B aligned)
  uint16_t* s_ptr = reinterpret_cast<uint16_t*>(s_src + csr_stride(N));          // [N+1]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (a.run_if_gt && *a.run_if_gt <= a.run_thresh) return;
  // one (graph, head) per CTA; the fallback launch behind the table kernel uses a small grid and strides
  for (int blk = blockIdx.x; blk < a.n_graphs * H; blk += gridDim.x) {
  if (blk != (int)blockIdx.x) __syncthreads();
  const int g = blk / H, h = blk - g * H;
  const float* g_obs = a.obs + (int64_t)g * a.obs_stride;
  const size_t base = (size_t)g * N;
  const size_t cg = a.graph_id ? (size_t)a.graph_id[(size_t)g * a.gid_stride] : (size_t)g;
  constexpr float kLog2e = 1.4426950408889634f;
  // ---------------------------------------------------------------- phase 0
  {
    const bool compact = a.Pt != nullptr;
    const int src_col = (TRANSFORMER && !compact ? HC : 0) + h * kC;
    const int val_col = (compact ? HC : 2 * HC) + h * kC;  // Transformer values
    const int tgt_col = (TRANSFORMER ? 0 : HC) + h * kC;
    // everything big is copied asynchronously (no registers, all loads in flight at once); the only chained
    // global access is (first, cnt) -> the compact target rows, and it overlaps the rest
    int first = 0, cnt = N;
    if (compact) { first = a.gfirst[g]; cnt = a.gcnt[g]; }
    const uint32_t sT32 = (uint32_t)__cvta_generic_to_shared(stT), sA32 = (uint32_t)__cvta_generic_to_shared(stA);
    const uint32_t sB32 = (uint32_t)__cvta_generic_to_shared(stB);
    for (int t = tid; t < N * 16; t += kEdgeThreads) {
      const int j = t >> 4, c = t & 15;                     // 16 chunks of 16 B per 128-channel row
      size_t pr = base + j;
      if (a.xrow_src) { const int xr = a.xrow_src[base + j]; if (xr < 0) continue; pr = (size_t)xr; }   // never read: not a source of a target
      else if (a.row_key) pr = (size_t)a.row_key[base + j];
      const bf16* row = a.P + pr * a.ldp;
      edge_cp_async16(sA32 + j * (kC * 2) + c * 16, row + src_col + c * 8);
      if (TRANSFORMER) edge_cp_async16(sB32 + j * (kC * 2) + c * 16, row + val_col + c * 8);
      if (!compact) edge_cp_async16(sT32 + j * (kC * 2) + c * 16, row + tgt_col + c * 8);
    }
    {
      const uint32_t sS32 = (uint32_t)__cvta_generic_to_shared(s_src);      // the graph's whole list block (16 B aligned)
      const uint8_t* gs = a.csr_src + cg * csr_stride(N);
      for (int t = tid; t < csr_stride(N) / 16; t += kEdgeThreads) edge_cp_async16(sS32 + t * 16, gs + t * 16);
    }
    const uint16_t* gp = a.csr_ptr + cg * (N + 1);
    for (int t = tid; t <= N; t += kEdgeThreads) s_ptr[t] = gp[t];
    for (int t = tid; t < N; t += kEdgeThreads) {
      s_slot[t] = a.slot ? a.slot[base + t] : -1;
      if (!compact) s_dm[t] = g_obs[t * 8 + 7];
      if (!TRANSFORMER) {
        size_t pr = a.row_key ? (size_t)a.row_key[base + t] : base + t;
        if (a.xrow_src) { const int xr = a.xrow_src[base + t]; pr = xr < 0 ? 0 : (size_t)xr; }
        if (compact) s_a[t] = a.ab[pr * H + h] * (0.6f * kLog2e);
        else {
          s_a[t] = a.ab[pr * (2 * H) + h] * (0.6f * kLog2e);
          s_b[t] = a.ab[pr * (2 * H) + H + h] * (0.6f * kLog2e);
        }
      }
    }
    if (compact) {                                          // target rows of the graph's controlling nodes: consecutive slots
      for (int t = tid; t < cnt * 16; t += kEdgeThreads) {
        const int k = t >> 4, c = t & 15;
        edge_cp_async16(sT32 + k * (kC * 2) + c * 16, a.Pt + (size_t)(first + k) * a.ldpt + h * kC + c * 8);
      }
      int* s_tl = reinterpret_cast<int*>(s_dm);            // target list (s_dm is only read by the pooling variant)
      for (int k = tid; k < cnt; k += kEdgeThreads) {
        s_tl[k] = a.idx[first + k] - (int)base;
        if (!TRANSFORMER) s_b[k] = a.bt[(size_t)(first + k) * H + h] * (0.6f * kLog2e);
      }
    }
  }
  const int grp = lane >> 4, sub = lane & 15;               // neighbour slot of the round / 8-channel slice of the head
  const int och = sub * 8;
  float bias8[8], attn[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    bias8[c] = TRANSFORMER ? 0.f : a.bias[h * kC + och + c];
    attn[c] = TRANSFORMER ? 0.f : a.att[h * kC + och + c] * (0.4f * kLog2e);
  }
  edge_cp_async_wait();
  __syncthreads();
  // ---------------------------------------------------------------- phase 1
  const float tr_scale = kLog2e / sqrtf((float)kC);
  const bf16* stV = TRANSFORMER ? stB : stA;
  const int self = TRANSFORMER ? 0 : 1;                     // GATv2: slot 0 of every target is its self loop
  float pool[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) pool[c] = a.pool_mode == MLS_POOL_MAX ? -INFINITY : 0.f;
  const int n_targets = a.Pt ? a.gcnt[g] : N;               // compact mode: only the controlling nodes, split evenly over the warps
  for (int tk = warp; tk < n_targets; tk += kEdgeWarps) {
    const int i = a.Pt ? reinterpret_cast<const int*>(s_dm)[tk] : tk;
    const int sl = s_slot[i];
    if (a.ctrl_only && sl < 0) continue;
    long long orow = (long long)(base + i);
    if (a.xrow_out) { orow = a.xrow_out[base + i]; if (orow < 0) continue; }
    const int r0 = s_ptr[i];
    const int d = (int)s_ptr[i + 1] - r0 + self;            // warp uniform, <= kMaxList + 1
    const int ti = a.Pt ? tk : i;                           // row of the target side in stT / s_b
    float tg[8];                                            // the target's 8 channels stay in registers
    {
      float4 lo4, hi4;
      bf16x8_to_f32(reinterpret_cast<const uint4*>(stT + ti * kC)[sub], lo4, hi4);
      tg[0] = lo4.x; tg[1] = lo4.y; tg[2] = lo4.z; tg[3] = lo4.w; tg[4] = hi4.x; tg[5] = hi4.y; tg[6] = hi4.z; tg[7] = hi4.w;
    }
    const float b_i = TRANSFORMER ? 0.f : s_b[ti];
    float mx = -INFINITY, den = 0.f;
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
    for (int kb = 0; kb < d; kb += 4) {                     // 4 neighbours per pass: two lane groups x two independent chains
      const int k0 = kb + grp, k1 = kb + 2 + grp;
      const bool v0 = k0 < d, v1 = k1 < d;
      int j0 = i, j1 = i;
      if (v0 && k0 >= self) j0 = s_src[r0 + k0 - self];
      if (v1) j1 = s_src[r0 + k1 - self];                   // k1 >= 2 > self
      float x0[8], x1[8];
      {
        float4 l0, h0, l1, h1;
        bf16x8_to_f32(reinterpret_cast<const uint4*>(stA + j0 * kC)[sub], l0, h0);
        bf16x8_to_f32(reinterpret_cast<const uint4*>(stA + j1 * kC)[sub], l1, h1);
        x0[0] = l0.x; x0[1] = l0.y; x0[2] = l0.z; x0[3] = l0.w; x0[4] = h0.x; x0[5] = h0.y; x0[6] = h0.z; x0[7] = h0.w;
        x1[0] = l1.x; x1[1] = l1.y; x1[2] = l1.z; x1[3] = l1.w; x1[4] = h1.x; x1[5] = h1.y; x1[6] = h1.z; x1[7] = h1.w;
      }
      float pa0 = 0.f, pb0 = 0.f, pa1 = 0.f, pb1 = 0.f;     // two partial sums per chain: shorter FFMA dependency
#pragma unroll
      for (int c = 0; c < 8; c += 2) {
        if (TRANSFORMER) {
          pa0 = fmaf(x0[c], tg[c], pa0); pb0 = fmaf(x0[c + 1], tg[c + 1], pb0);
          pa1 = fmaf(x1[c], tg[c], pa1); pb1 = fmaf(x1[c + 1], tg[c + 1], pb1);
        } else {
          pa0 = fmaf(attn[c], fabsf(x0[c] + tg[c]), pa0); pb0 = fmaf(attn[c + 1], fabsf(x0[c + 1] + tg[c + 1]), pb0);
          pa1 = fmaf(attn[c], fabsf(x1[c] + tg[c]), pa1); pb1 = fmaf(attn[c + 1], fabsf(x1[c + 1] + tg[c + 1]), pb1);
        }
      }
      float e0 = pa0 + pb0, e1 = pa1 + pb1;
#pragma unroll
      for (int o = 1; o < 16; o <<= 1) {
        e0 += __shfl_xor_sync(0xffffffffu, e0, o);
        e1 += __shfl_xor_sync(0xffffffffu, e1, o);
      }
      e0 = TRANSFORMER ? e0 * tr_scale : e0 + (s_a[j0] + b_i);
      e1 = TRANSFORMER ? e1 * tr_scale : e1 + (s_a[j1] + b_i);
      if (!v0) e0 = -INFINITY;
      if (!v1) e1 = -INFINITY;
      float m_r = fmaxf(e0, e1);
      m_r = fmaxf(m_r, __shfl_xor_sync(0xffffffffu, m_r, 16));
      if (kb > 0 && m_r > mx) {                             // only targets with more than 4 entries get here (warp uniform)
        const float resc = fast_ex2(mx - m_r);
        den *= resc;
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] *= resc;
      }
      mx = fmaxf(mx, m_r);
      const float p0 = fast_ex2(e0 - mx), p1 = fast_ex2(e1 - mx);   // 0 for padded slots
      den += p0 + p1;                                       // per-group partial
      if (TRANSFORMER) {
        float4 l0, h0, l1, h1;
        bf16x8_to_f32(reinterpret_cast<const uint4*>(stV + j0 * kC)[sub], l0, h0);
        bf16x8_to_f32(reinterpret_cast<const uint4*>(stV + j1 * kC)[sub], l1, h1);
        x0[0] = l0.x; x0[1] = l0.y; x0[2] = l0.z; x0[3] = l0.w; x0[4] = h0.x; x0[5] = h0.y; x0[6] = h0.z; x0[7] = h0.w;
        x1[0] = l1.x; x1[1] = l1.y; x1[2] = l1.z; x1[3] = l1.w; x1[4] = h1.x; x1[5] = h1.y; x1[6] = h1.z; x1[7] = h1.w;
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[c] = fmaf(p1, x1[c], fmaf(p0, x0[c], acc[c]));
    }
    // combine the two lane groups (both end up with the full sums; group 0 writes)
    den += __shfl_xor_sync(0xffffffffu, den, 16);
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], 16);
    const float inv_den = fast_rcp(den + 1e-16f);           // isolated Transformer node: acc = 0 -> output 0
    float o[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) o[c] = fmaxf(fmaf(acc[c], inv_den, bias8[c]), 0.f);
    if (grp == 0) {
      uint4 ov;
      ov.x = pack_bf16x2_rn(o[0], o[1]); ov.y = pack_bf16x2_rn(o[2], o[3]); ov.z = pack_bf16x2_rn(o[4], o[5]); ov.w = pack_bf16x2_rn(o[6], o[7]);
      if (a.x_out) *reinterpret_cast<uint4*>(a.x_out + (size_t)orow * HC + h * kC + och) = ov;     // 16 lanes: 256 contiguous bytes
      if (a.z && sl >= 0 && a.pool_mode < 0) *reinterpret_cast<uint4*>(a.z + (size_t)sl * a.ldz + a.z_col + h * kC + och) = ov;
    }
    if (a.pool_mode >= 0) {
      const float dm = s_dm[i];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float v = o[c] * dm;
        pool[c] = a.pool_mode == MLS_POOL_MAX ? fmaxf(pool[c], v) : pool[c] + v;
      }
    }
  }
  if (a.pool_mode >= 0) {      // HL-DGN: z[g] = pool_i(relu(conv)[i] * dm[i])  (hl_dgn.py:103-108)
    if (grp == 0) {
      *reinterpret_cast<float4*>(poolbuf + warp * kC + och) = make_float4(pool[0], pool[1], pool[2], pool[3]);
      *reinterpret_cast<float4*>(poolbuf + warp * kC + och + 4) = make_float4(pool[4], pool[5], pool[6], pool[7]);
    }
    __syncthreads();
    if (tid < kC) {
      const int used = N < kEdgeWarps ? N : kEdgeWarps;        // warps that own at least one node
      float r = poolbuf[tid];
      for (int w2 = 1; w2 < used; ++w2) {
        const float v = poolbuf[w2 * kC + tid];
        r = a.pool_mode == MLS_POOL_MAX ? fmaxf(r, v) : r + v;
      }
      if (a.pool_mode == MLS_POOL_MEAN) r = r / (float)N;
      a.z[(size_t)g * a.ldz + a.z_col + h * kC + tid] = __float2bfloat16_rn(r);
    }
  }
  }
}

// ------------------------------------------------------------------------------ controlling nodes + needed rows
// One warp per graph.
//   controlling list: idx[slot] = node row, slot[node row] = slot or -1; the slots of a graph's controlling nodes are
//     consecutive, in node order (gfirst / gcnt; one atomic reservation per graph)
//   needed rows (two-conv models, adj != NULL): the network reads conv2 only at the controlling nodes
//     (l_dgn.py:133-139), so conv2's sources -- and therefore the only rows of relu(conv1) anybody reads -- are the
//     controlling nodes themselves (self loop, snapshot) and their radius-graph sources.  The needed rows are ordered
//     [all controlling nodes, in slot order][the other needed nodes]: a controlling node's needed row IS its slot, so
//     relu(conv1) of a controlling node is written once and x1[0 : count) doubles as the snapshot matrix.  Here the other
//     needed nodes get xrow = -2 - j (j from a counter of their own, ncount); need_rows_fixup_kernel turns that into
//     count + j once the total number of controlling nodes is known, and builds nidx[r] = node row of needed row r.
// mode 1 (agent-observation rows, one controlling node per graph): slot of graph g is g.
template <int W>
__global__ void ctrl_need_list_kernel(const uint8_t* __restrict__ ctrl_mask, const float* __restrict__ obs, int64_t obs_stride,
                                      int N, int n_graphs, int mode, const uint32_t* __restrict__ adj,
                                      const int* __restrict__ graph_id, int gid_stride, int* __restrict__ idx,
                                      int* __restrict__ slot, int* __restrict__ count, int* __restrict__ gfirst,
                                      int* __restrict__ gcnt, int* __restrict__ nidx, int* __restrict__ xrow,
                                      int* __restrict__ ncount, int* __restrict__ nfirst, int* __restrict__ ncnt,
                                      const uint16_t* __restrict__ csr_ptr, const uint8_t* __restrict__ csr_src, int self_loops,
                                      int* __restrict__ ecount, int* __restrict__ eabs, uint16_t* __restrict__ eent,
                                      int* __restrict__ gmeta) {
  const int lane = threadIdx.x & 31;
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (g >= n_graphs) return;
  uint32_t cw[W];
  int total = 0;
  if (mode == 1) {
    float c = obs[(int64_t)g * obs_stride + (int64_t)N * 8];
    c = fminf(fmaxf(c, 0.f), (float)(N - 1));
    const int ci = (int)(long long)c;
#pragma unroll
    for (int w = 0; w < W; ++w) cw[w] = (ci >> 5) == w ? 1u << (ci & 31) : 0u;
    total = 1;
  } else {
#pragma unroll
    for (int w = 0; w < W; ++w) {
      const int i = w * 32 + lane;
      cw[w] = __ballot_sync(0xffffffffu, i < N && ctrl_mask[(size_t)g * N + i] != 0);
      total += __popc(cw[w]);
    }
  }
  int s = 0;
  if (mode == 1) {
    s = g;
    if (g == 0 && lane == 0) *count = n_graphs;
  } else {
    if (lane == 0 && total) s = atomicAdd(count, total);
    s = __shfl_sync(0xffffffffu, s, 0);
  }
  if (lane == 0) { gfirst[g] = s; gcnt[g] = total; }
  const int slot0 = s;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const int i = w * 32 + lane;
    if (i < N) {
      const bool c = (cw[w] >> lane) & 1u;
      const int t = s + __popc(cw[w] & ((1u << lane) - 1));
      if (c) idx[t] = g * N + i;
      slot[(size_t)g * N + i] = c ? t : -1;
    }
    s += __popc(cw[w]);
  }
  if (!adj) return;
  const uint32_t* ga = adj + (graph_id ? (size_t)graph_id[(size_t)g * gid_stride] : (size_t)g) * N * W;
  uint32_t nw[W];
#pragma unroll
  for (int w = 0; w < W; ++w) nw[w] = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const int i = w * 32 + lane;
    if ((cw[w] >> lane) & 1u) {
#pragma unroll
      for (int v = 0; v < W; ++v) nw[v] |= ga[(size_t)i * W + v];
    }
  }
  int nn = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    nw[w] = __reduce_or_sync(0xffffffffu, nw[w]) | cw[w];
    nn += __popc(nw[w]);
  }
  const int nalloc = nn - total;
  int ns = 0;
  if (lane == 0 && nalloc) ns = atomicAdd(ncount, nalloc);
  ns = __shfl_sync(0xffffffffu, ns, 0);
  if (lane == 0) { nfirst[g] = ns; ncnt[g] = nn; }
  int run_c = slot0, run_o = ns;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const int i = w * 32 + lane;
    const uint32_t ow = nw[w] & ~cw[w], below = (1u << lane) - 1;
    if (i < N) {
      int r = -1;
      if ((cw[w] >> lane) & 1u) r = run_c + __popc(cw[w] & below);
      else if ((ow >> lane) & 1u) r = -2 - (run_o + __popc(ow & below));
      xrow[(size_t)g * N + i] = r;
    }
    run_c += __popc(cw[w]);
    run_o += __popc(ow);
  }
  if (!eent) return;
  // conv2 edge list of the graph, shared by the heads: per controlling node (slot order) one entry per incoming edge
  // (the GATv2 self loop first), entry = compact source index (rank in the needed list) | target index << 8; the
  // graph's block starts 16-byte aligned, eabs[slot] = absolute position of the slot's first entry
  const size_t cg = graph_id ? (size_t)graph_id[(size_t)g * gid_stride] : (size_t)g;
  const uint16_t* gp = csr_ptr + cg * (N + 1);
  const uint8_t* gs = csr_src + cg * csr_stride(N);
  int etot = 0;
  int r0v[W], dv[W], offv[W];
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const int i = w * 32 + lane;
    const bool c = (cw[w] >> lane) & 1u;
    r0v[w] = 0; dv[w] = 0;
    if (c) { r0v[w] = gp[i]; dv[w] = (int)gp[i + 1] - r0v[w]; }
    const int v = c ? dv[w] + self_loops : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    offv[w] = etot + incl - v;
    etot += __shfl_sync(0xffffffffu, incl, 31);
  }
  int e0 = 0;
  if (lane == 0 && etot) e0 = atomicAdd(ecount, (etot + 7) & ~7);          // 8 entries of 2 bytes = 16 bytes
  e0 = __shfl_sync(0xffffffffu, e0, 0);
  if (lane == 0) {
    int* gm = gmeta + (size_t)g * 8;
    gm[0] = slot0; gm[1] = total; gm[2] = ns; gm[3] = nn; gm[4] = e0; gm[5] = etot; gm[6] = 0; gm[7] = 0;
  }
  int tk_base = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const int i = w * 32 + lane;
    if ((cw[w] >> lane) & 1u) {
      const int tk = tk_base + __popc(cw[w] & ((1u << lane) - 1));
      int pos = e0 + offv[w];
      eabs[slot0 + tk] = pos;
      auto rank_of = [&](int j) {                        // controlling nodes first (rank among them), then the other needed nodes
        const int jw = j >> 5;
        const uint32_t below = (1u << (j & 31)) - 1u;
        int r = 0;
        const bool jc = (cw[jw] >> (j & 31)) & 1u;
#pragma unroll
        for (int v = 0; v < W; ++v) {
          const uint32_t m = v < jw ? 0xffffffffu : (v == jw ? below : 0u);
          r += __popc((jc ? cw[v] : (nw[v] & ~cw[v])) & m);
        }
        return jc ? r : total + r;
      };
      if (self_loops) eent[pos++] = (uint16_t)(rank_of(i) | (tk << 8));
      for (int k = 0; k < dv[w]; ++k) eent[pos + k] = (uint16_t)(rank_of(gs[r0v[w] + k]) | (tk << 8));
    }
    tk_base += __popc(cw[w]);
  }
}

// Final needed rows (see ctrl_need_list_kernel).  One thread per node row: -2 - j -> count + j, nidx[row] = node
// row; one thread per graph: first non-controlling needed row of the graph (gmeta[2]) made absolute; thread 0: ncount (the
// other needed nodes so far) -> total number of needed rows.
__global__ void need_rows_fixup_kernel(int* __restrict__ xrow, int* __restrict__ nidx, int* __restrict__ gmeta, const int* __restrict__ count,
                                       const int* __restrict__ ncount, int* __restrict__ ntotal, int rows, int n_graphs) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = *count;
  if (t < rows) {
    int r = xrow[t];
    if (r <= -2) { r = c + (-2 - r); xrow[t] = r; }
    if (r >= 0) nidx[r] = t;
  }
  if (gmeta && t < n_graphs) gmeta[(size_t)t * 8 + 2] += c;
  if (t == 0) *ntotal = *ncount + c;
}

// z[t][0:hidden] = x0[idx[t]]  (encoder snapshot, l_dgn.py:121-122)
__global__ void gather_x0_kernel(const int* __restrict__ idx, const int* __restrict__ count, const bf16* __restrict__ x0,
                                 const uint32_t* __restrict__ row_key, int hidden, bf16* __restrict__ z, int ldz) {
  // grid-stride over the compacted controlling rows (their count is only known on the device: most of a grid sized for
  // every node row would exit at once)
  const int n = *count;
  for (int t = blockIdx.x * blockDim.y + threadIdx.y; t < n; t += gridDim.x * blockDim.y) {
    const size_t r = row_key ? (size_t)__ldg(row_key + __ldg(idx + t)) : (size_t)__ldg(idx + t);
    for (int c = threadIdx.x * 8; c < hidden; c += blockDim.x * 8)
      *reinterpret_cast<uint4*>(z + (size_t)t * ldz + c) = __ldg(reinterpret_cast<const uint4*>(x0 + (size_t)r * hidden + c));
  }
}

// last head layer + dueling + action; hid row = [Q hidden (hh) | V hidden (hh)] in bf16
__global__ void head_out_bf16_kernel(const bf16* __restrict__ hid, int hh, const int* __restrict__ idx, const int* __restrict__ count,
                                     int max_rows, const float* __restrict__ wq, const float* __restrict__ bq,
                                     const float* __restrict__ wv, const float* __restrict__ bv, int64_t row0, int per_graph_N,
                                     float* __restrict__ q_out, int8_t* __restrict__ act_out, int out_mode, ActArgsB aa) {
  const int lane = threadIdx.x & 31;
  const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n = count ? min(*count, max_rows) : max_rows;
  if (t >= n) return;
  const bf16* hq = hid + (size_t)t * 2 * hh;
  const bf16* hv = hq + hh;
  float s0 = 0.f, s1 = 0.f, sv = 0.f;
  for (int c = lane; c < hh; c += 32) {
    const float q = __bfloat162float(hq[c]), v = __bfloat162float(hv[c]);
    s0 = fmaf(q, wq[c], s0);
    s1 = fmaf(q, wq[hh + c], s1);
    sv = fmaf(v, wv[c], sv);
  }
  s0 = warp_sum(s0) + bq[0]; s1 = warp_sum(s1) + bq[1]; sv = warp_sum(sv) + bv[0];
  if (lane == 0) {
    const float mean = (s0 + s1) / 2.0f;
    const float o0 = (s0 - mean) + sv, o1 = (s1 - mean) + sv;
    int64_t orow;
    if (out_mode == 0) orow = row0 + idx[t];
    else if (out_mode == 1) orow = row0 / per_graph_N + idx[t] / per_graph_N;
    else orow = t;
    q_out[orow * 2 + 0] = o0;
    q_out[orow * 2 + 1] = o1;
    if (act_out && out_mode != 2) act_out[orow] = (int8_t)select_action_b(o0, o1, aa, (uint64_t)orow);
  }
}

// Network without dueling heads: q = out_linear(latent) (l_dgn.py:88-90,149) on the bf16 latent rows.  One warp per row.
// With x1 (L-DGN / DGN-R) the snapshot columns [hid, hid + HC) of latent row t are x1 row t, the rest come from z.
__global__ void head_linear_b_kernel(const bf16* __restrict__ z, int latent, const bf16* __restrict__ x1, int hid, int HC,
                                     const int* __restrict__ idx, const int* __restrict__ count,
                                     int max_rows, const float* __restrict__ w, const float* __restrict__ b, int64_t row0, int per_graph_N,
                                     float* __restrict__ q_out, int8_t* __restrict__ act_out, int out_mode, ActArgsB aa) {
  const int lane = threadIdx.x & 31;
  const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n = count ? min(*count, max_rows) : max_rows;
  if (t >= n) return;
  const bf16* zr = z + (size_t)t * latent;
  const bf16* xr = x1 ? x1 + (size_t)t * HC : nullptr;
  float s0 = 0.f, s1 = 0.f;
  for (int c = lane; c < latent; c += 32) {
    const bool snap = x1 && c >= hid && c < hid + HC;
    const float v = __bfloat162float(snap ? xr[c - hid] : zr[c]);
    s0 = fmaf(v, w[c], s0);
    s1 = fmaf(v, w[latent + c], s1);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
  s0 += b[0]; s1 += b[1];
  if (lane == 0) {
    int64_t orow;
    if (out_mode == 0) orow = row0 + idx[t];
    else if (out_mode == 1) orow = row0 / per_graph_N + idx[t] / per_graph_N;
    else orow = t;
    q_out[orow * 2 + 0] = s0;
    q_out[orow * 2 + 1] = s1;
    if (act_out && out_mode != 2) act_out[orow] = (int8_t)select_action_b(s0, s1, aa, (uint64_t)orow);
  }
}

__global__ void hl_scatter_b_kernel(const float* __restrict__ qg, const uint8_t* __restrict__ ctrl_mask, int N, int n_graphs,
                                    int64_t graph0, int mode, float* __restrict__ q_out, int8_t* __restrict__ act_out, ActArgsB aa) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (mode == 1) {
    if (t >= n_graphs) return;
    const float o0 = qg[t * 2], o1 = qg[t * 2 + 1];
    const int64_t orow = graph0 + t;
    q_out[orow * 2] = o0; q_out[orow * 2 + 1] = o1;
    if (act_out) act_out[orow] = (int8_t)select_action_b(o0, o1, aa, (uint64_t)orow);
    return;
  }
  if (t >= (int64_t)n_graphs * N) return;
  if (!ctrl_mask[t]) return;
  const int64_t g = t / N, orow = graph0 * N + t;
  const float o0 = qg[g * 2], o1 = qg[g * 2 + 1];
  q_out[orow * 2] = o0; q_out[orow * 2 + 1] = o1;
  if (act_out) act_out[orow] = (int8_t)select_action_b(o0, o1, aa, (uint64_t)orow);
}

}  // namespace mls

// ================================================================================== host
namespace {
using namespace mls;

size_t al(size_t v, size_t a = 1024) { return (v + a - 1) / a * a; }

int degree_bits(int n_nodes) { int b = 1; while ((1 << b) < n_nodes) ++b; return b; }
int table_keys(int n_nodes) { return (1 << degree_bits(n_nodes)) * 512; }     // deg | 6 bits msgs | 3 flag bits

struct WsB {
  // ---- packed parameters + feature tables (mls_dgn_prepare; offsets independent of the number of graphs)
  bf16 *w_enc1, *w_c1, *w_c2, *w_h0, *w_h1;
  float *b_c1, *b_c2, *b_h0, *b_h1;
  float *hv1, *hv2;           // output-layer dot vectors [2*hh] each
  float *att1, *att2;
  bf16 *t_h, *t_x0, *t_P;     // discrete-feature tables: [n_keys][hid], [n_keys][hid], [n_keys][nproj*HC]
  float* t_ab;                // [n_keys][2H]
  // ---- per pass
  bf16 *h, *x0, *P, *x1, *z;
  bf16 *hid1, *hid2;          // hidden layers of dueling heads that are not 128 wide (the fused head keeps them on chip)
  float* qg;
  int *idx, *slot, *count, *gfirst, *gcnt;
  int *nidx, *xrow, *ncount, *nfirst, *ncnt;   // needed rows (conv2 sources)
  int* ntotal;                                 // controlling + other needed rows (ncount counts the others only)
  int *ecount, *eabs, *gmeta;                  // conv2 edge lists (conv2_attn.cu)
  uint16_t* eent;
  uint16_t* csr_ptr;
  uint8_t* csr_src;
  uint32_t* adjm;             // [graphs][N][W] radius-graph source masks
  float* ab;
  uint32_t* key;              // [R]
  // tensor-core table attention (attn_table.cu)
  uint32_t* used;             // [n_keys / 32] bitmap
  uint16_t* cid_of_key;       // [n_keys]
  uint32_t* key_of_cid;       // [kAttnUcap]
  int* n_used;
  uint16_t* row_cid;          // [R]
  float* pairE;               // [kAttnUcap][kAttnUcap][4]
  void* Vh;                   // [kAttnUcap][512] fp16
  unsigned char* rec;         // per-tile records of the conv1 pre-pass (attn_table_record_bytes)
  int2* tile_idx;             // [tiles]
};

size_t carve_b(const MlsNetDesc* d, int Gc, unsigned char* base, WsB* ws) {
  const size_t R = al((size_t)Gc * d->n_nodes, 128);
  const int hid = d->hidden, HC = d->hidden * d->heads, hh2 = 2 * d->head_hidden;
  const bool hl = d->kind == MLS_NET_HL_DGN;
  const int nproj = d->kind == MLS_NET_DGN_R ? 3 : 2;
  const int latent = hl ? HC : hid + 2 * HC;
  const size_t T = hl ? al((size_t)Gc, 128) : R;
  const int Wn = mls_words_per_row(d->n_nodes);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = al(off + bytes); return o; };
  // parameters and tables first: their offsets must not depend on Gc (MLS_FWD_PREPARED)
  const size_t o_we = take((size_t)hid * hid * 2), o_wc1 = take((size_t)nproj * HC * hid * 2);
  const size_t o_wc2 = take(hl ? 0 : (size_t)nproj * HC * HC * 2), o_wh0 = take((size_t)hh2 * latent * 2);
  const size_t o_wh1 = take((size_t)hh2 * hh2 * 2);
  const size_t o_bc1 = take((size_t)nproj * HC * 4), o_bc2 = take((size_t)nproj * HC * 4), o_bh0 = take(hh2 * 4), o_bh1 = take(hh2 * 4);
  const size_t o_hv1 = take(hh2 * 4), o_hv2 = take(hh2 * 4);
  const size_t o_att1 = take((size_t)2 * HC * 4), o_att2 = take((size_t)2 * HC * 4);
  const size_t KT = (size_t)table_keys(d->n_nodes);
  const size_t o_th = take(KT * hid * 2), o_tx0 = take(KT * hid * 2), o_tP = take(KT * nproj * HC * 2), o_tab = take(KT * 2 * d->heads * 4);
  // per pass
  const size_t o_h = take(R * hid * 2), o_x0 = take(R * hid * 2), o_P = take(R * nproj * HC * 2);
  const size_t hid_bytes = d->head_hidden == 128 ? 0 : T * hh2 * 2;
  const size_t o_x1 = take(hl ? 0 : R * HC * 2), o_z = take(T * latent * 2), o_h1 = take(hid_bytes), o_h2 = take(hid_bytes);
  const size_t o_qg = take((size_t)Gc * 8), o_idx = take(R * 4), o_slot = take(R * 4), o_cnt = take(16);
  const bool c2 = !hl && conv2_attn_supported(d->n_nodes, d->heads);
  const size_t o_eabs = take(c2 ? R * 4 : 0), o_gmeta = take(c2 ? (size_t)Gc * 32 : 0);
  const size_t o_eent = take(c2 ? (R * (kMaxList + 1) + (size_t)Gc * 8 + 64) * 2 : 0);   // sources + GATv2 self loop
  const size_t o_gf = take((size_t)Gc * 4), o_gc = take((size_t)Gc * 4);
  const size_t o_nidx = take(hl ? 0 : R * 4), o_xrow = take(hl ? 0 : R * 4), o_nf = take(hl ? 0 : (size_t)Gc * 4), o_nc = take(hl ? 0 : (size_t)Gc * 4);
  const size_t o_cptr = take(((size_t)Gc * (d->n_nodes + 1) + 64) * 2), o_csrc = take((size_t)Gc * csr_stride(d->n_nodes) + 64);
  const size_t o_adjm = take(hl ? 0 : (size_t)Gc * d->n_nodes * Wn * 4);
  const size_t o_ab = take(R * 2 * d->heads * 4);
  const size_t o_key = take(R * 4);
  const bool mma_ok = attn_table_supported(d->n_nodes, d->heads);
  const size_t o_used = take(KT), o_cok = take(KT * 2), o_koc = take(kAttnUcap * 4), o_nu = take(4);
  const size_t o_pe = take(mma_ok ? attn_table_pair_bytes() : 0), o_rcid = take(R * 2), o_vh = take(mma_ok ? attn_table_value_bytes() : 0);
  const size_t o_rec = take(mma_ok && !hl ? attn_table_record_bytes(d->n_nodes, Gc) : 0), o_tix = take(mma_ok && !hl ? ((size_t)Gc + 1) * 8 : 0);
  if (ws) {
    auto B = [&](size_t o) { return reinterpret_cast<bf16*>(base + o); };
    auto F = [&](size_t o) { return reinterpret_cast<float*>(base + o); };
    auto I = [&](size_t o) { return reinterpret_cast<int*>(base + o); };
    ws->w_enc1 = B(o_we); ws->w_c1 = B(o_wc1); ws->w_c2 = B(o_wc2); ws->w_h0 = B(o_wh0); ws->w_h1 = B(o_wh1);
    ws->b_c1 = F(o_bc1); ws->b_c2 = F(o_bc2); ws->b_h0 = F(o_bh0); ws->b_h1 = F(o_bh1);
    ws->hv1 = F(o_hv1); ws->hv2 = F(o_hv2);
    ws->h = B(o_h); ws->x0 = B(o_x0); ws->P = B(o_P); ws->x1 = B(o_x1); ws->z = B(o_z); ws->hid1 = B(o_h1); ws->hid2 = B(o_h2);
    ws->qg = F(o_qg);
    ws->idx = I(o_idx); ws->slot = I(o_slot); ws->count = I(o_cnt); ws->ncount = I(o_cnt) + 1; ws->ecount = I(o_cnt) + 2; ws->ntotal = I(o_cnt) + 3;
    ws->eabs = I(o_eabs); ws->gmeta = I(o_gmeta); ws->eent = reinterpret_cast<uint16_t*>(base + o_eent);
    ws->gfirst = I(o_gf); ws->gcnt = I(o_gc);
    ws->nidx = I(o_nidx); ws->xrow = I(o_xrow); ws->nfirst = I(o_nf); ws->ncnt = I(o_nc);
    ws->csr_ptr = reinterpret_cast<uint16_t*>(base + o_cptr); ws->csr_src = base + o_csrc;
    ws->adjm = reinterpret_cast<uint32_t*>(base + o_adjm);
    ws->ab = F(o_ab); ws->att1 = F(o_att1); ws->att2 = F(o_att2);
    ws->t_h = B(o_th); ws->t_x0 = B(o_tx0); ws->t_P = B(o_tP); ws->t_ab = F(o_tab); ws->key = reinterpret_cast<uint32_t*>(base + o_key);
    ws->used = reinterpret_cast<uint32_t*>(base + o_used); ws->cid_of_key = reinterpret_cast<uint16_t*>(base + o_cok);
    ws->key_of_cid = reinterpret_cast<uint32_t*>(base + o_koc); ws->n_used = reinterpret_cast<int*>(base + o_nu);
    ws->pairE = F(o_pe); ws->row_cid = reinterpret_cast<uint16_t*>(base + o_rcid); ws->Vh = base + o_vh;
    ws->rec = (mma_ok && !hl) ? base + o_rec : nullptr; ws->tile_idx = (mma_ok && !hl) ? reinterpret_cast<int2*>(base + o_tix) : nullptr;
  }
  return off;
}

template <bool TR>
int launch_edge(cudaStream_t st, const EdgeArgs& ea) {
  constexpr int kEdgeThreads = EdgeCfg<TR>::kThreads, kEdgeWarps = kEdgeThreads / 32;
  const size_t smem = (size_t)ea.N * kC * 2 * (TR ? 3 : 2) + (size_t)ea.N * 4 * 4 + (ea.pool_mode >= 0 ? kEdgeWarps * kC * 4 : 0) +
                      ((size_t)ea.N + 1) * 2 + (size_t)csr_stride(ea.N) + 16;
  static size_t configured = 0;
  if (smem > 227 * 1024) {
    mls_set_error("bf16 attention kernel needs %zu bytes of shared memory for %d nodes (max 232448): use precision fp32", smem, ea.N);
    return MLS_ERR_UNSUPPORTED;
  }
  if (smem > configured) {
    if (smem > 48 * 1024)
      MLS_CUDA(cudaFuncSetAttribute(edge_bf16_kernel<TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // ask for the largest shared-memory carveout: the default split only fits 2 of these CTAs per SM
    MLS_CUDA(cudaFuncSetAttribute(edge_bf16_kernel<TR>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    configured = smem;
  }
  int grid = ea.n_graphs * ea.H;
  if (ea.run_if_gt && grid > 148 * 4) grid = 148 * 4;      // normally exits at once
  edge_bf16_kernel<TR><<<grid, kEdgeThreads, smem, st>>>(ea);
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}

int edge_dispatch(cudaStream_t st, const EdgeArgs& ea, bool tr) {
  return tr ? launch_edge<true>(st, ea) : launch_edge<false>(st, ea);
}

// radius_graph lists (+ source bitmasks) of n_graphs graphs whose positions sit in obs-style rows
int launch_csr(cudaStream_t st, const float* obs, int64_t obs_stride, int N, int n_graphs, uint16_t* csr_ptr, uint8_t* csr_src,
               uint32_t* adjm) {
  const int Wn = mls_words_per_row(N);
  const size_t csm = (size_t)N * Wn * 4 + ((size_t)N + 1) * 4 + (size_t)N * 8;
  const int thr = N <= 64 ? 64 : 256;           // small graphs: more, smaller CTAs (fewer threads idle at the barriers)
  switch (Wn) {
    case 1: graph_csr_kernel<1><<<n_graphs, thr, csm, st>>>(obs, obs_stride, N, n_graphs, csr_ptr, csr_src, adjm); break;
    case 2: graph_csr_kernel<2><<<n_graphs, thr, csm, st>>>(obs, obs_stride, N, n_graphs, csr_ptr, csr_src, adjm); break;
    case 4: graph_csr_kernel<4><<<n_graphs, thr, csm, st>>>(obs, obs_stride, N, n_graphs, csr_ptr, csr_src, adjm); break;
    default: graph_csr_kernel<8><<<n_graphs, thr, csm, st>>>(obs, obs_stride, N, n_graphs, csr_ptr, csr_src, adjm); break;
  }
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}

struct CsrCache {          // layout of the topology cache buffer
  uint16_t* ptr;
  uint8_t* src;
  uint32_t* adjm;
};
size_t carve_cache(int N, int G, unsigned char* base, CsrCache* c) {
  const int Wn = mls_words_per_row(N);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = al(off + bytes); return o; };
  const size_t o_p = take(((size_t)G * (N + 1) + 64) * 2), o_s = take((size_t)G * csr_stride(N) + 64), o_a = take((size_t)G * N * Wn * 4);
  if (c) { c->ptr = reinterpret_cast<uint16_t*>(base + o_p); c->src = base + o_s; c->adjm = reinterpret_cast<uint32_t*>(base + o_a); }
  return off;
}

// weights -> bf16 (stacked the way the GEMMs consume them), biases stay fp32; with `tables` the discrete-feature
// tables (encoder output + conv1 projections of every feature key)
int pack_parameters(const MlsNetDesc* d, const MlsNetWeights* w, const WsB& ws, bool tables, int sms, cudaStream_t st) {
  const int N = d->n_nodes, hid = d->hidden, H = d->heads, HC = hid * H, hh = d->head_hidden, hh2 = 2 * hh;
  const bool hl = d->kind == MLS_NET_HL_DGN, tr = d->kind == MLS_NET_DGN_R;
  const int nproj = tr ? 3 : 2;
  const int latent = hl ? HC : hid + 2 * HC;
  CvtJobs cj{};
  int n = 0;
  auto add = [&](const float* src, bf16* dst, int rows, int cols, int ld, int ro, int co) { cj.j[n++] = CvtJob{src, dst, rows, cols, ld, ro, co}; };
  add(w->enc_w1, ws.w_enc1, hid, hid, hid, 0, 0);
  add(w->c1_wa, ws.w_c1, HC, hid, hid, 0, 0);
  add(w->c1_wb, ws.w_c1, HC, hid, hid, HC, 0);
  if (tr) add(w->c1_wc, ws.w_c1, HC, hid, hid, 2 * HC, 0);
  cj.n = n;
  cvt_weights_kernel<<<dim3(64, n), 256, 0, st>>>(cj);
  CvtJobs c2{};
  n = 0;
  auto add2 = [&](const float* src, bf16* dst, int rows, int cols, int ld, int ro, int co) { c2.j[n++] = CvtJob{src, dst, rows, cols, ld, ro, co}; };
  if (!hl) {
    add2(w->c2_wa, ws.w_c2, HC, HC, HC, 0, 0);
    add2(w->c2_wb, ws.w_c2, HC, HC, HC, HC, 0);
    if (tr) add2(w->c2_wc, ws.w_c2, HC, HC, HC, 2 * HC, 0);
  }
  const bool dueling = w->out_w == nullptr;
  MLS_CUDA(cudaMemsetAsync(ws.w_h1, 0, (size_t)hh2 * hh2 * 2, st));
  if (dueling) {
    add2(w->q_w0, ws.w_h0, hh, latent, latent, 0, 0);
    add2(w->v_w0, ws.w_h0, hh, latent, latent, hh, 0);
    add2(w->q_w1, ws.w_h1, hh, hh, hh2, 0, 0);       // block diagonal: Q and V hidden layers in one GEMM
    add2(w->v_w1, ws.w_h1, hh, hh, hh2, hh, hh);
  }
  c2.n = n;
  if (n > 0) cvt_weights_kernel<<<dim3(128, n), 256, 0, st>>>(c2);
  CatJobs bj{};
  int m = 0;
  auto addb = [&](const float* src, float* dst, int cnt) { bj.src[m] = src; bj.dst[m] = dst; bj.n[m] = cnt; ++m; };
  addb(w->c1_ba, ws.b_c1, HC); addb(w->c1_bb, ws.b_c1 + HC, HC);
  if (tr) addb(w->c1_bc, ws.b_c1 + 2 * HC, HC);
  if (!tr) { addb(w->c1_att, ws.att1, HC); addb(w->c1_att, ws.att1 + HC, HC); }
  MLS_CUDA(cudaMemsetAsync(ws.hv2, 0, (size_t)hh2 * 4, st));
  if (dueling) {
    addb(w->q_b0, ws.b_h0, hh); addb(w->v_b0, ws.b_h0 + hh, hh);
    addb(w->q_b1, ws.b_h1, hh); addb(w->v_b1, ws.b_h1 + hh, hh);
    // output layer as dot vectors for the epilogue of the last hidden-layer GEMM: [wq[0] | wv], [wq[1] | 0]
    addb(w->q_w2, ws.hv1, hh); addb(w->v_w2, ws.hv1 + hh, hh); addb(w->q_w2 + hh, ws.hv2, hh);
  }
  bj.count = m;
  cat_bias_kernel<<<dim3(2, m), 256, 0, st>>>(bj);
  if (!hl) {
    CatJobs b2{};
    m = 0;
    auto addc = [&](const float* src, float* dst, int cnt) { b2.src[m] = src; b2.dst[m] = dst; b2.n[m] = cnt; ++m; };
    addc(w->c2_ba, ws.b_c2, HC); addc(w->c2_bb, ws.b_c2 + HC, HC);
    if (!tr) { addc(w->c2_att, ws.att2, HC); addc(w->c2_att, ws.att2 + HC, HC); }
    if (tr) addc(w->c2_bc, ws.b_c2 + 2 * HC, HC);
    b2.count = m;
    cat_bias_kernel<<<dim3(2, m), 256, 0, st>>>(b2);
    mls_count_launch();
  }
  mls_count_launch(3);
  MLS_LAUNCH_CHECK();
  if (tables) {
    int rc;
    const int n_keys = table_keys(N);
    const int rows_per_cta = 256 / (hid / 8);
    enc0_keys_kernel<<<(n_keys + rows_per_cta - 1) / rows_per_cta, 256, 0, st>>>(n_keys, d->input_dim, w->enc_w0, w->enc_b0, hid, ws.t_h);
    mls_count_launch();
    GemmEpilogue e0{ws.t_x0, hid, w->enc_b1, nullptr, 0, N, 1, nullptr, nullptr};
    if ((rc = gemm_bf16_launch(ws.t_h, hid, ws.w_enc1, hid, GemmShape{n_keys, hid, hid, nullptr}, e0, sms, st))) return rc;
    GemmEpilogue e1{ws.t_P, nproj * HC, ws.b_c1, nullptr, 0, N, 0, tr ? nullptr : ws.att1, tr ? nullptr : ws.t_ab};
    if ((rc = gemm_bf16_launch(ws.t_x0, hid, ws.w_c1, hid, GemmShape{n_keys, nproj * HC, hid, nullptr}, e1, sms, st))) return rc;
  }
  return MLS_OK;
}

int sm_count_of_current_device(int* sms) {
  int dev = 0;
  MLS_CUDA(cudaGetDevice(&dev));
  MLS_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
  return MLS_OK;
}

}  // namespace

#include <stdlib.h>
int bf16_chunk_graphs(const MlsNetDesc* d, int n_graphs) {
  // Up to 12800 128-row GEMM tiles (1.64 M node rows, ~16 GB of bf16 workspace) per pass: 32768 episodes of
  // 50 nodes go through in one pass.  Measured on B200 (profiles/r01_chunk_sweep.txt): every pass costs the
  // ramp/drain of ~20 kernels, so fewer, larger passes win (one pass 6.36 ms/round, three passes 6.56 ms),
  // and L2-sized chunks (148 tiles) are 35 % slower.  MLS_BF16_CHUNK_TILES overrides.
  static int tiles = 0;
  if (!tiles) {
    const char* e = getenv("MLS_BF16_CHUNK_TILES");
    tiles = e ? atoi(e) : 12800;
    if (tiles < 1) tiles = 12800;
  }
  int gc = (tiles * 128) / d->n_nodes;
  if (gc < 1) gc = 1;
  return n_graphs < gc ? n_graphs : gc;
}

size_t dgn_workspace_bytes_bf16(const MlsNetDesc* d, int n_graphs) {
  return carve_b(d, bf16_chunk_graphs(d, n_graphs), nullptr, nullptr);
}

int dgn_prepare_bf16(const MlsNetDesc* d, const MlsNetWeights* w, int flags, void* workspace, size_t workspace_bytes, void* stream) {
  MLS_CHECK_ARG(d->hidden % 64 == 0 && d->head_hidden % 64 == 0, "bf16 path needs hidden sizes that are multiples of 64");
  MLS_CHECK_ARG(workspace && workspace_bytes >= carve_b(d, 1, nullptr, nullptr), "workspace too small");
  int sms = 0, rc;
  if ((rc = sm_count_of_current_device(&sms))) return rc;
  WsB ws;
  carve_b(d, 1, (unsigned char*)workspace, &ws);           // the packed region does not depend on the graph count
  return pack_parameters(d, w, ws, (flags & MLS_FWD_DISCRETE_FEATURES) != 0, sms, reinterpret_cast<cudaStream_t>(stream));
}

size_t dgn_csr_cache_bytes(const MlsNetDesc* d, int n_pool_graphs) { return carve_cache(d->n_nodes, n_pool_graphs, nullptr, nullptr); }

int dgn_csr_cache_build(const MlsNetDesc* d, const float* pos_obs, int64_t obs_stride, int n_pool_graphs, void* cache, size_t cache_bytes,
                        void* stream) {
  MLS_CHECK_ARG(cache && cache_bytes >= carve_cache(d->n_nodes, n_pool_graphs, nullptr, nullptr), "topology cache buffer too small");
  CsrCache c;
  carve_cache(d->n_nodes, n_pool_graphs, (unsigned char*)cache, &c);
  return launch_csr(reinterpret_cast<cudaStream_t>(stream), pos_obs, obs_stride, d->n_nodes, n_pool_graphs, c.ptr, c.src, c.adjm);
}

int dgn_forward_bf16(const MlsNetDesc* d, const MlsNetWeights* w, const MlsForwardArgs* a, void* stream) {
  const int N = d->n_nodes, hid = d->hidden, H = d->heads, HC = hid * H, hh = d->head_hidden, hh2 = 2 * hh;
  MLS_CHECK_ARG(hid % 64 == 0 && hh % 64 == 0, "bf16 path needs hidden sizes that are multiples of 64");
  const int Gc = bf16_chunk_graphs(d, a->n_graphs);
  MLS_CHECK_ARG(a->workspace && a->workspace_bytes >= carve_b(d, Gc, nullptr, nullptr), "workspace too small");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int sms = 0, rc;
  if ((rc = sm_count_of_current_device(&sms))) return rc;
  WsB ws;
  carve_b(d, Gc, (unsigned char*)a->workspace, &ws);
  const int Wn = mls_words_per_row(N);
  const bool hl = d->kind == MLS_NET_HL_DGN, tr = d->kind == MLS_NET_DGN_R;
  const int nproj = tr ? 3 : 2;
  const int latent = hl ? HC : hid + 2 * HC;
  ActArgsB aa{a->eps, a->philox_seed, a->philox_offset, a->rand3, reinterpret_cast<const unsigned long long*>(a->philox_offset_dev), a->philox_row0};
  if (a->ctrl_mode == 0) {
    MLS_CUDA(cudaMemsetAsync(a->q, 0, (size_t)a->n_graphs * N * 2 * sizeof(float), st));
    if (a->act) MLS_CUDA(cudaMemsetAsync(a->act, 0xFF, (size_t)a->n_graphs * N, st));
  }
  // discrete-feature mode: encoder + conv1 projections as a table over all feature keys
  const bool use_table = (a->flags & MLS_FWD_DISCRETE_FEATURES) != 0;
  if (!(a->flags & MLS_FWD_PREPARED) && (rc = pack_parameters(d, w, ws, use_table, sms, st))) return rc;
  cudaEvent_t ev0 = reinterpret_cast<cudaEvent_t>(a->prof_start), ev1 = reinterpret_cast<cudaEvent_t>(a->prof_stop);
  bool first_chunk = true;
  auto prof_begin = [&](int which) { if (first_chunk && ev0 && ev1 && a->prof_kernel == which) cudaEventRecord(ev0, st); };
  auto prof_end = [&](int which) { if (first_chunk && ev0 && ev1 && a->prof_kernel == which) cudaEventRecord(ev1, st); };
  const int degbits = degree_bits(N), n_keys = table_keys(N);
  if (use_table) {
    if (a->feature_errors) MLS_CUDA(cudaMemsetAsync(a->feature_errors, 0, sizeof(int), st));
    MLS_CUDA(cudaMemsetAsync(ws.used, 0, (size_t)n_keys / 8, st));
  }
  // conv1 attention through the pair-logit table + tensor-core aggregation (graphs of <= 62 nodes)
  const bool use_mma = use_table && attn_table_supported(N, H) && mls_get_option("attn_mma");
  // conv2 attention with tensor-core aggregation over the compacted row sets (graphs of <= 64 nodes)
  const bool use_c2 = !hl && conv2_attn_supported(N, H) && mls_get_option("conv2_mma");
  // topology cache of a static pool: lists per pool graph, selected by graph id
  CsrCache cache{};
  const bool cached = a->csr_cache && a->graph_ids;
  if (cached) {
    MLS_CHECK_ARG(a->csr_cache_graphs > 0 && a->graph_id_stride > 0, "topology cache: pool size / graph id stride missing");
    carve_cache(N, a->csr_cache_graphs, (unsigned char*)const_cast<void*>(a->csr_cache), &cache);
  }
  for (int g0 = 0; g0 < a->n_graphs; g0 += Gc) {
    const int gc = (a->n_graphs - g0) < Gc ? (a->n_graphs - g0) : Gc;
    const int rows = gc * N;
    const float* obs = a->obs + (int64_t)g0 * a->obs_stride;
    const uint8_t* cm = a->ctrl_mode == 0 ? a->ctrl_mask + (size_t)g0 * N : nullptr;
    const int* gid = cached ? a->graph_ids + (size_t)g0 * a->graph_id_stride : nullptr;
    const int gid_stride = cached ? a->graph_id_stride : 0;
    const uint16_t* csr_ptr = cached ? cache.ptr : ws.csr_ptr;
    const uint8_t* csr_src = cached ? cache.src : ws.csr_src;
    const uint32_t* adjm = cached ? cache.adjm : ws.adjm;
    // radius graph (unless cached), then the controlling-node list and the needed rows
    if (!cached && (rc = launch_csr(st, obs, a->obs_stride, N, gc, ws.csr_ptr, ws.csr_src, hl ? nullptr : ws.adjm))) return rc;
    if (!hl) {
      MLS_CUDA(cudaMemsetAsync(ws.count, 0, 4 * sizeof(int), st));
      const unsigned grid = (unsigned)((gc * 32 + 255) / 256);
#define MLS_LIST(WW) ctrl_need_list_kernel<WW><<<grid, 256, 0, st>>>(cm, obs, a->obs_stride, N, gc, a->ctrl_mode, adjm, gid, gid_stride, ws.idx, \
                                                                      ws.slot, ws.count, ws.gfirst, ws.gcnt, ws.nidx, ws.xrow, ws.ncount, ws.nfirst, ws.ncnt, \
                                                                      csr_ptr, csr_src, tr ? 0 : 1, ws.ecount, ws.eabs, use_c2 ? ws.eent : nullptr, ws.gmeta)
      switch (Wn) { case 1: MLS_LIST(1); break; case 2: MLS_LIST(2); break; case 4: MLS_LIST(4); break; default: MLS_LIST(8); break; }
#undef MLS_LIST
      const int nthr = rows > gc ? rows : gc;
      need_rows_fixup_kernel<<<(nthr + 255) / 256, 256, 0, st>>>(ws.xrow, ws.nidx, use_c2 ? ws.gmeta : nullptr, ws.count, ws.ncount, ws.ntotal, rows, gc);
      mls_count_launch(2);
    }
    // encoder (or, in discrete-feature mode, just the table keys of this pass)
    if (use_table) {
      feature_key_kernel<<<(rows + 1023) / 1024, 1024, use_mma ? (size_t)(n_keys / 32) * 4 : 0, st>>>(
          obs, a->obs_stride, N, rows, degbits, ws.key, reinterpret_cast<int*>(a->feature_errors), use_mma ? ws.used : nullptr);
      mls_count_launch();
    } else {
      const int rows_per_cta = 256 / (hid / 8);
      enc0_bf16_kernel<<<(rows + rows_per_cta - 1) / rows_per_cta, 256, 0, st>>>(obs, a->obs_stride, N, rows, d->input_dim, w->enc_w0,
                                                                                  w->enc_b0, hid, ws.h);
      mls_count_launch();
      GemmEpilogue e{ws.x0, hid, w->enc_b1, nullptr, 0, N, 1, nullptr, nullptr};
      if ((rc = gemm_bf16_launch(ws.h, hid, ws.w_enc1, hid, GemmShape{rows, hid, hid, nullptr}, e, sms, st))) return rc;
      // conv1 projections (table mode: already in ws.t_P for every feature key)
      GemmEpilogue e1{ws.P, nproj * HC, ws.b_c1, nullptr, 0, N, 0, tr ? nullptr : ws.att1, tr ? nullptr : ws.ab};
      prof_begin(MLS_PROF_PROJ1);
      if ((rc = gemm_bf16_launch(ws.x0, hid, ws.w_c1, hid, GemmShape{rows, nproj * HC, hid, nullptr}, e1, sms, st))) return rc;
      prof_end(MLS_PROF_PROJ1);
    }
    // conv1 attention (+ReLU): relu(conv1) of the needed rows (compacted, x1; x1[0 : count) are the controlling nodes'
    // snapshot rows, pre-mask); HL-DGN: graph pooling into z
    {
      EdgeArgs ea{};
      ea.P = use_table ? ws.t_P : ws.P; ea.ldp = nproj * HC; ea.obs = obs; ea.obs_stride = a->obs_stride; ea.N = N; ea.H = H;
      ea.n_graphs = gc; ea.row_key = use_table ? ws.key : nullptr;
      ea.att = w->c1_att; ea.bias = w->c1_bias; ea.csr_ptr = csr_ptr; ea.csr_src = csr_src; ea.ab = use_table ? ws.t_ab : ws.ab;
      ea.graph_id = gid; ea.gid_stride = gid_stride;
      if (hl) { ea.x_out = nullptr; ea.z = ws.z; ea.ldz = latent; ea.z_col = 0; ea.ctrl_only = 0; ea.pool_mode = d->pool; }
      else { ea.x_out = ws.x1; ea.ctrl_only = 0; ea.pool_mode = -1; ea.xrow_out = ws.xrow; }
      prof_begin(MLS_PROF_EDGE1);
      if (use_mma) {
        AttnTableArgs ta{};
        ta.t_P = ws.t_P; ta.ldp = nproj * HC; ta.t_ab = ws.t_ab; ta.att = w->c1_att; ta.bias = tr ? nullptr : w->c1_bias;
        ta.transformer = tr ? 1 : 0; ta.key = ws.key; ta.N = N; ta.H = H; ta.n_graphs = gc; ta.csr_ptr = csr_ptr;
        ta.csr_src = csr_src; ta.graph_id = gid; ta.gid_stride = gid_stride;
        if (hl) { ta.z = ws.z; ta.ldz = latent; ta.z_col = 0; ta.pool_mode = d->pool; ta.obs = obs; ta.obs_stride = a->obs_stride; }
        else { ta.xrow = ws.xrow; ta.x_out = ws.x1; ta.pool_mode = -1; }
        ta.used_bits = ws.used; ta.n_keys = n_keys; ta.cid_of_key = ws.cid_of_key; ta.key_of_cid = ws.key_of_cid;
        ta.n_used = ws.n_used; ta.E = ws.pairE; ta.row_cid = ws.row_cid; ta.Vh = ws.Vh;
        ta.rec = ws.rec; ta.tile_idx = ws.tile_idx;
        if ((rc = attn_table_conv_launch(ta, sms, st))) return rc;
        ea.run_if_gt = ws.n_used; ea.run_thresh = kAttnUcap;      // more distinct keys than the table holds: gather kernel
      }
      if ((rc = edge_dispatch(st, ea, tr))) return rc;
      prof_end(MLS_PROF_EDGE1);
    }
    if (!hl) {
      // conv2 projections on x1 * dm (the row mask commutes with the GEMM, applied in its epilogue), both in one launch
      // over the packed weight rows (Transformer [q; k; v], GATv2 [l; r]).  Source side (GATv2 x_l, Transformer k | v) on
      // the needed rows; target side (GATv2 x_r, Transformer q) on the controlling nodes: x1[0 : count) itself (the x1
      // tile is read once for both).  fp16 outputs for the tensor-core attention.
      const int nsrc = nproj - 1;
      bf16* Psrc = ws.P;                                    // [needed rows][nsrc*HC]
      bf16* Ptgt = ws.P + (size_t)rows * nsrc * HC;         // [count][HC]
      float* dots_t = ws.ab + (size_t)rows * H;             // [count][H]
      GemmEpilogue e{Psrc, nsrc * HC, ws.b_c2, obs, a->obs_stride, N, 0, tr ? nullptr : ws.att2, tr ? nullptr : ws.ab, ws.nidx};
      e.c_fp16 = use_c2 ? 1 : 0;
      e.Ct = Ptgt; e.ldct = HC; e.dots_t = tr ? nullptr : dots_t; e.row_index_t = ws.idx;
      GemmShape sh{rows, nproj * HC, HC, ws.ntotal};
      sh.m_dev_t = ws.count; sh.t_lo = tr ? 0 : HC; sh.t_hi = sh.t_lo + HC;
      prof_begin(MLS_PROF_PROJ2);
      if ((rc = gemm_bf16_launch(ws.x1, HC, ws.w_c2, HC, sh, e, sms, st))) return rc;
      prof_end(MLS_PROF_PROJ2);
      // conv2 attention only where a controlling agent reads it; the result goes straight into z
      prof_begin(MLS_PROF_EDGE2);
      if (use_c2) {
        Conv2Args ca{};
        ca.Ps = reinterpret_cast<const __half*>(Psrc); ca.lds = nsrc * HC; ca.Pt = reinterpret_cast<const __half*>(Ptgt); ca.ldt = HC;
        ca.as = ws.ab; ca.bt = dots_t; ca.att = w->c2_att; ca.bias = tr ? nullptr : w->c2_bias; ca.transformer = tr ? 1 : 0;
        ca.N = N; ca.H = H; ca.n_graphs = gc; ca.gmeta = ws.gmeta; ca.eabs = ws.eabs; ca.eent = ws.eent;
        ca.z = ws.z; ca.ldz = latent; ca.z_col = hid + HC;
        if ((rc = conv2_attn_launch(ca, sms, st))) return rc;
      } else {
        EdgeArgs ea{};
        ea.P = Psrc; ea.ldp = nsrc * HC; ea.obs = obs; ea.obs_stride = a->obs_stride; ea.N = N; ea.H = H; ea.n_graphs = gc;
        ea.Pt = Ptgt; ea.ldpt = HC; ea.bt = dots_t; ea.gfirst = ws.gfirst; ea.gcnt = ws.gcnt; ea.idx = ws.idx;
        ea.att = w->c2_att; ea.bias = w->c2_bias; ea.csr_ptr = csr_ptr; ea.csr_src = csr_src; ea.ab = ws.ab; ea.x_out = nullptr;
        ea.slot = ws.slot; ea.z = ws.z; ea.ldz = latent; ea.z_col = hid + HC; ea.ctrl_only = 1; ea.pool_mode = -1;
        ea.xrow_src = ws.xrow; ea.graph_id = gid; ea.gid_stride = gid_stride;
        if ((rc = edge_dispatch(st, ea, tr))) return rc;
      }
      prof_end(MLS_PROF_EDGE2);
      dim3 blk(16, 16);
      gather_x0_kernel<<<std::min((rows + 15) / 16, sms * 16), blk, 0, st>>>(ws.idx, ws.count, use_table ? ws.t_x0 : ws.x0, use_table ? ws.key : nullptr, hid, ws.z, latent);
      mls_count_launch();
    }
    // dueling head on the tensor cores: [Q0;V0] stacked, then block-diagonal [Q1 0; 0 V1]
    const int head_rows = hl ? gc : rows;
    const int* m_dev = hl ? nullptr : ws.count;
    if (w->out_w) {                                           // no dueling heads: one linear layer on the latent row
      if (!hl) {
        head_linear_b_kernel<<<(rows * 32 + 255) / 256, 256, 0, st>>>(ws.z, latent, ws.x1, hid, HC, ws.idx, ws.count, rows, w->out_w,
                                                                      w->out_b, (int64_t)g0 * N, N, a->q, a->act, a->ctrl_mode, aa);
        mls_count_launch();
      } else {
        head_linear_b_kernel<<<(gc * 32 + 255) / 256, 256, 0, st>>>(ws.z, latent, nullptr, 0, HC, nullptr, nullptr, gc, w->out_w, w->out_b,
                                                                    0, N, ws.qg, nullptr, 2, aa);
        const long long nthr = a->ctrl_mode == 1 ? gc : (long long)gc * N;
        hl_scatter_b_kernel<<<(unsigned)((nthr + 255) / 256), 256, 0, st>>>(ws.qg, cm, N, gc, g0, a->ctrl_mode, a->q, a->act, aa);
        mls_count_launch(2);
      }
    } else {
      GemmShape sh0{head_rows, hh2, latent, m_dev};
      if (!hl) { sh0.A2 = ws.x1; sh0.lda2 = HC; sh0.k2_lo = hid; sh0.k2_hi = hid + HC; }   // snapshot columns come from x1
      prof_begin(MLS_PROF_HEAD0);
      if (hh == 128) {
        // both hidden layers, the output layer and the action in one kernel: the hidden activations stay on chip
        HeadOut ho{w->q_b2, w->v_b2, hl ? nullptr : ws.idx, hl ? 0 : (int64_t)g0 * N, N, hl ? ws.qg : a->q, hl ? nullptr : a->act,
                   hl ? 2 : a->ctrl_mode, aa};
        if ((rc = head_dueling_launch(ws.z, latent, sh0, ws.w_h0, ws.w_h1, HeadVecs{ws.b_h0, ws.b_h1, ws.hv1, ws.hv2}, ho, sms, st))) return rc;
        prof_end(MLS_PROF_HEAD0);
      } else {
        GemmEpilogue e0{ws.hid1, hh2, ws.b_h0, nullptr, 0, N, 1, nullptr, nullptr};
        if ((rc = gemm_bf16_launch(ws.z, latent, ws.w_h0, latent, sh0, e0, sms, st))) return rc;
        prof_end(MLS_PROF_HEAD0);
        GemmEpilogue e1{ws.hid2, hh2, ws.b_h1, nullptr, 0, N, 1, nullptr, nullptr};
        if ((rc = gemm_bf16_launch(ws.hid1, hh2, ws.w_h1, hh2, GemmShape{head_rows, hh2, hh2, m_dev}, e1, sms, st))) return rc;
        if (!hl)
          head_out_bf16_kernel<<<(rows * 32 + 255) / 256, 256, 0, st>>>(ws.hid2, hh, ws.idx, ws.count, rows, w->q_w2, w->q_b2, w->v_w2,
                                                                         w->v_b2, (int64_t)g0 * N, N, a->q, a->act, a->ctrl_mode, aa);
        else
          head_out_bf16_kernel<<<(gc * 32 + 255) / 256, 256, 0, st>>>(ws.hid2, hh, nullptr, nullptr, gc, w->q_w2, w->q_b2, w->v_w2,
                                                                       w->v_b2, 0, N, ws.qg, nullptr, 2, aa);
        mls_count_launch();
      }
      if (hl) {
        const long long nthr = a->ctrl_mode == 1 ? gc : (long long)gc * N;
        hl_scatter_b_kernel<<<(unsigned)((nthr + 255) / 256), 256, 0, st>>>(ws.qg, cm, N, gc, g0, a->ctrl_mode, a->q, a->act, aa);
        mls_count_launch();
      }
    }
    MLS_LAUNCH_CHECK();
    first_chunk = false;
  }
  return MLS_OK;
}
