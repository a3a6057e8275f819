// Attention convolution in discrete-feature mode, on the tensor cores (sm_100a).
//
// With MLS_FWD_DISCRETE_FEATURES every node's encoder output and conv1 projections are rows of small
// tables indexed by the node's feature key (dgn_forward_bf16.cu).  The attention logit of an edge then
// depends only on the pair (target key, source key):
//
//   compact_keys_kernel   keys present in this pass -> dense ids 0..U-1
//   pair_logit_kernel     E[ci][cj][h] = base-2 logit of head h for target key ci, source key cj
//                           GATv2:       0.6 (a_j + b_i) + 0.4 sum_c att_c |x_l[j,c] + x_r[i,c]|
//                           Transformer: <q_i, k_j> / sqrt(C)
//   values_fp16_kernel    value rows x_l[key] / v[key] of the present keys as fp16
//
// The aggregation runs on tcgen05 per tile of G graphs (G*N <= 62 node rows), with the softmax weights
// 2^(e_ij - max_i) / (sum_j + 1e-16) from E as an fp16 weight matrix W_h[target][source] (block diagonal
// over the graphs of a tile) and the value rows of the tile's nodes as the other operand; the aggregation
// over (at most 33) neighbours is done densely because the tensor core does the 64-wide row in 4 instructions.
//
//   attn_table_prep_kernel + attn_table_rows_kernel   L-DGN / DGN-R: relu(conv1) of the needed rows into x1.
//       A pre-pass builds one record per tile (needed targets, softmax weights); the MMA kernel's producers only
//       move data, D[target][channel] = W x V per (tile, head), and the epilogue writes whole x1 rows.
//   attn_table_pool_kernel   HL-DGN: one graph per tile, out^T[channel][target] = V^T x W^T per (tile, head pair),
//       the epilogue pools relu(conv) * dm over the graph's nodes into z.
//
// Reference math: PyG GATv2Conv / TransformerConv as used by l_dgn.py:125,133 and dgn_r.py; softmax
// exp(e - max) / (sum + 1e-16).  Same results as edge_bf16_kernel up to bf16 rounding of the weights.
#include "attn_table.cuh"

#include <cuda_fp16.h>

#include "dgn_kernels.cuh"
#include "tcgen05_ptx.cuh"

namespace mls {

namespace {

typedef __nv_bfloat16 bf16;

// cute::UMMA::SmemDescriptor, SWIZZLE_128B, explicit LBO / SBO (both in 16-byte units)
__device__ __forceinline__ uint64_t make_smem_desc_ex(uint32_t smem_addr, uint32_t lbo16, uint32_t sbo16) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo16 & 0x3FFFu) << 16;
  d |= (uint64_t)(sbo16 & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor with B MN-major (bit 16)
__host__ __device__ constexpr uint32_t make_idesc_bmn(int M, int N) { return make_idesc(M, N) | (1u << 16); }

__global__ void __launch_bounds__(128) umma_mn_probe_kernel(const bf16* __restrict__ A, const bf16* __restrict__ B, float* __restrict__ D,
                                                            int rows_a, int kt, uint32_t lbo16, uint32_t sbo16, uint32_t kadv16) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = smem;                 // 128 rows x 128 B
  unsigned char* sB = smem + 16384;         // 2 panels x 64 rows x 128 B
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 32768);
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 1);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  for (int u = t; u < 128 * 8; u += 128) {
    const int r = u >> 3, c = u & 7;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r < rows_a) v = *reinterpret_cast<const uint4*>(A + (size_t)r * 64 + c * 8);
    *reinterpret_cast<uint4*>(sA + r * 128 + ((c ^ (r & 7)) << 4)) = v;
  }
  for (int u = t; u < 64 * 16; u += 128) {
    const int k = u >> 4, c = u & 15;       // node row k, 16-byte chunk c of its 128 channels
    const int pn = c >> 3, ch = c & 7;
    const uint4 v = *reinterpret_cast<const uint4*>(B + (size_t)k * 128 + c * 8);
    *reinterpret_cast<uint4*>(sB + pn * 8192 + k * 128 + ((ch ^ (k & 7)) << 4)) = v;
  }
  fence_proxy_async();
  if (t == 0) { mbar_init(smem_u32(bar), 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(smem_u32(tslot), 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tslot;
  if (t == 0) {
    const uint32_t idesc = make_idesc_bmn(128, 128);
    const uint64_t da = make_smem_desc(smem_u32(sA)), db = make_smem_desc_ex(smem_u32(sB), lbo16, sbo16);
    for (int k = 0; k < kt / 16; ++k) umma_bf16(tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * kadv16), idesc, k ? 1u : 0u);
    umma_commit(smem_u32(bar));
  }
  mbar_wait(smem_u32(bar), 0);
  tc_fence_after();
  for (int c0 = 0; c0 < 128; c0 += 32) {
    uint32_t v[32];
    tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
    for (int j = 0; j < 32; ++j) D[(size_t)(warp * 32 + lane) * 128 + c0 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}


// ------------------------------------------------------------------------------ key compaction
// used_bits: bitmap over all feature keys, bit set by feature_key_kernel for every key present in this pass.
__global__ void __launch_bounds__(1024) compact_keys_kernel(uint32_t* __restrict__ used_bits, int n_keys, uint16_t* __restrict__ cid_of_key,
                                                            uint32_t* __restrict__ key_of_cid, int* __restrict__ n_used) {
  __shared__ int s_warp[32];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int n_words = n_keys >> 5;
  const int per = (n_words + 1023) / 1024;
  const int w0 = t * per, w1 = min(n_words, w0 + per);
  int cnt = 0;
  for (int w = w0; w < w1; ++w) cnt += __popc(used_bits[w]);
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = s_warp[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += v;
    }
    s_warp[lane] = wi - w;
    if (lane == 31) *n_used = wi;
  }
  __syncthreads();
  int id = s_warp[warp] + incl - cnt;
  for (int w = w0; w < w1; ++w) {
    uint32_t bits = used_bits[w];
    used_bits[w] = 0;                                   // clean for the next pass
    while (bits) {
      const int b = __ffs(bits) - 1;
      bits &= bits - 1;
      const int k = w * 32 + b;
      if (id < kAttnUcap) { cid_of_key[k] = (uint16_t)id; key_of_cid[id] = (uint32_t)k; }
      ++id;
    }
  }
}

__global__ void row_cid_kernel(const uint32_t* __restrict__ key, const uint16_t* __restrict__ cid_of_key, int rows,
                               uint16_t* __restrict__ row_cid) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < rows) row_cid[r] = cid_of_key[key[r]];
}

// Value rows (GATv2 x_l, Transformer v) of the keys present in this pass as fp16, indexed by compact id: exact for
// every bf16 value inside fp16's normal range (saturated beyond +-65504, flushed below 2^-24).
__global__ void values_fp16_kernel(const AttnTableArgs a) {
  const int U = *a.n_used;
  if (U > kAttnUcap) return;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int cid = t >> 6, c = t & 63;                       // 64 chunks of 8 channels per row
  if (cid >= U) return;
  const int vcol = a.transformer ? 2 * a.H * kC : 0;
  const uint4 v = __ldg(reinterpret_cast<const uint4*>(a.t_P + (size_t)a.key_of_cid[cid] * a.ldp + vcol) + c);
  const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&v);
  uint4 o;
  uint32_t* op = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 f = __bfloat1622float2(p[i]);
    f.x = fminf(fmaxf(f.x, -65504.f), 65504.f); f.y = fminf(fmaxf(f.y, -65504.f), 65504.f);
    const __half2 h2 = __floats2half2_rn(f.x, f.y);
    op[i] = *reinterpret_cast<const uint32_t*>(&h2);
  }
  reinterpret_cast<uint4*>(a.Vh)[(size_t)cid * 64 + c] = o;
}

__device__ __forceinline__ void unpack8(const uint4 u, float* f) {
  const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 v = __bfloat1622float2(p[i]); f[2 * i] = v.x; f[2 * i + 1] = v.y; }
}

// ------------------------------------------------------------------------------ pair logits
// One warp per (target key, 32 source keys); lane = (head, 16-channel slice).
__global__ void __launch_bounds__(256) pair_logit_kernel(const AttnTableArgs a) {
  const int U = *a.n_used;
  if (U > kAttnUcap) return;
  constexpr float kLog2e = 1.4426950408889634f;
  const int H = a.H, HC = H * kC;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int h = lane >> 3, sub = lane & 7;
  const int src_col = (a.transformer ? HC : 0) + h * kC + sub * 16;
  const int tgt_col = (a.transformer ? 0 : HC) + h * kC + sub * 16;
  float attn[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) attn[c] = a.transformer ? 1.f : a.att[h * kC + sub * 16 + c] * (0.4f * kLog2e);
  const float tr_scale = kLog2e / sqrtf((float)kC);
  const int nchunk = (U + 31) / 32;
  const int tasks = U * nchunk;
  for (int task = blockIdx.x * 8 + warp; task < tasks; task += gridDim.x * 8) {
    const int ci = task / nchunk, cj0 = (task - ci * nchunk) * 32;
    const uint32_t ki = a.key_of_cid[ci];
    float tg[16];
    {
      const uint4* p = reinterpret_cast<const uint4*>(a.t_P + (size_t)ki * a.ldp + tgt_col);
      unpack8(p[0], tg); unpack8(p[1], tg + 8);
    }
    const float b_i = a.transformer ? 0.f : a.t_ab[(size_t)ki * (2 * H) + H + h] * (0.6f * kLog2e);
    const int cj1 = min(U, cj0 + 32);
    // four source keys in flight (read-only loads: free to move above the previous iterations' table stores)
#pragma unroll 4
    for (int cj = cj0; cj < cj1; ++cj) {
      const uint32_t kj = __ldg(a.key_of_cid + cj);
      float x[16];
      const uint4* p = reinterpret_cast<const uint4*>(a.t_P + (size_t)kj * a.ldp + src_col);
      unpack8(__ldg(p), x); unpack8(__ldg(p + 1), x + 8);
      float pa = 0.f, pb = 0.f;
      if (a.transformer) {
#pragma unroll
        for (int c = 0; c < 16; c += 2) { pa = fmaf(x[c], tg[c], pa); pb = fmaf(x[c + 1], tg[c + 1], pb); }
      } else {
#pragma unroll
        for (int c = 0; c < 16; c += 2) { pa = fmaf(attn[c], fabsf(x[c] + tg[c]), pa); pb = fmaf(attn[c + 1], fabsf(x[c + 1] + tg[c + 1]), pb); }
      }
      float e = pa + pb;
      e += __shfl_xor_sync(0xffffffffu, e, 1);
      e += __shfl_xor_sync(0xffffffffu, e, 2);
      e += __shfl_xor_sync(0xffffffffu, e, 4);
      if (a.transformer) e *= tr_scale;
      else e += __ldg(a.t_ab + (size_t)kj * (2 * H) + h) * (0.6f * kLog2e) + b_i;
      float4 o;
      o.x = __shfl_sync(0xffffffffu, e, 0); o.y = __shfl_sync(0xffffffffu, e, 8);
      o.z = __shfl_sync(0xffffffffu, e, 16); o.w = __shfl_sync(0xffffffffu, e, 24);
      if (lane == 0) reinterpret_cast<float4*>(a.E)[(size_t)ci * kAttnUcap + cj] = o;
    }
  }
}

// ------------------------------------------------------------------------------ graph pooling on the tensor cores
// The MMA is issued transposed, out_h^T[channel][target] = V_h^T x W_h^T, so that M = 128 channels fills the
// tensor core's rows whatever the graph's node count and a warp's 32 TMEM lanes are 32 consecutive channels:
// the pooling over the graph's nodes is a reduction over each lane's registers.
//   A operand = value panels [source][channel]   (MN-major, 128B swizzle)
//   B operand = weight matrix [target][source]   (K-major,  128B swizzle)
// Work item = (tile, head pair).  A stage is 48 KiB (2 weight matrices + 4 value panels), so four stages and four
// producer teams of 3 warps are in flight.
//   warp 0  MMA issuer      warp 1  TMEM allocation      warps 2..9  epilogue (quarter = w & 3, head of the pair = (w - 2) >> 2)
//   warps 10..21  four producer teams of 3 warps; team t builds items t, t+4, ... (item k: tile k >> 1, head pair k & 1)
constexpr int kAHead = 64 * 128;               // weight matrix of one head: 64 targets x 64 sources bf16
constexpr int kBPanel = 64 * 128;              // value panel: 64 sources x 64 channels bf16
constexpr int kMetaSrc = 64 * kMaxNbr;         // CSR source lists of a tile: G * csr_stride(N) <= 2048 for G * N <= 64, N <= 62
static_assert(64 / 33 * csr_stride(33) <= kMetaSrc && csr_stride(62) <= kMetaSrc, "tile CSR lists");
constexpr int kMeta = kMetaSrc + 64 * 2 /*ids*/ + 128 * 2 /*CSR row pointers*/ + 64 * 4 /*dm*/;
constexpr int kPoolThreads = 704;
constexpr int kPoolTeam = 96;
constexpr int kStageA2 = 2 * kAHead;           // 16 KiB
constexpr int kStageB2 = 4 * kBPanel;          // 32 KiB
constexpr int kStage2 = kStageA2 + kStageB2;   // 48 KiB
constexpr int kPoolSmem = 4 * kStage2 + 4 * kMeta + 256 /*barriers*/ + 1024;

__device__ __forceinline__ float f_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float f_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ uint32_t a_off(int i, int j) {      // byte offset of W[i][j] inside a head's K-major SW128 tile
  return (uint32_t)(i * 128 + ((((j >> 3) ^ i) & 7) << 4) + (j & 7) * 2);
}
__device__ __forceinline__ void bar_pool_team(int team) { asm volatile("bar.sync %0, 96;" ::"r"(team + 1) : "memory"); }
// bounded waits: a protocol bug traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait_guard(uint32_t bar, uint32_t parity, unsigned ns) {
  for (unsigned spins = 0;; ++spins) {
    uint32_t ok;
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
    if (spins > (1u << 26)) __trap();
    if (ns) __nanosleep(ns);
  }
}

// HL-DGN: z[graph][z_col + H*C] = pool over the graph's nodes of relu(conv1) * dm, dm = obs column 7.  G = 1: the
// epilogue pools all 64 columns of a tile into one graph.
__global__ void __launch_bounds__(kPoolThreads, 1) attn_table_pool_kernel(const AttnTableArgs a, const int G) {
  if (*a.n_used > kAttnUcap) return;            // uniform: the gather kernel handles this pass
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* meta = smem + 4 * kStage2;                                       // [4][kMeta]
  uint64_t* bars = reinterpret_cast<uint64_t*>(meta + 4 * kMeta);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  const uint32_t bar0 = smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (4 + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (8 + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (12 + b); };

  const int N = a.N, HC = 4 * kC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (a.n_graphs + G - 1) / G;
  const int my_tiles = blockIdx.x < n_tiles ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int n_items = 2 * my_tiles;              // item k: tile blockIdx.x + (k >> 1) * gridDim.x, head pair k & 1
  const int kb = G * N;                          // K index of the two bias rows (hi, lo); <= 62
  const int ksteps = (kb + 2 + 15) >> 4;

  for (int u = threadIdx.x; u < 4 * kStage2 / 16; u += kPoolThreads) reinterpret_cast<uint4*>(smem)[u] = make_uint4(0, 0, 0, 0);
  if (threadIdx.x == 0) {
    for (int s = 0; s < 4; ++s) {
      mbar_init(full_bar(s), kPoolTeam); mbar_init(empty_bar(s), 1);
      mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 8 * 32);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================================================================== MMA issuer
    if (lane == 0) {
      const uint32_t idesc = (make_idesc(128, 64) & ~((7u << 7) | (7u << 10))) | (1u << 15);   // fp16 x fp16, A MN-major
      for (int k = 0; k < n_items; ++k) {
        const int s = k & 3;                                                   // shared-memory stage == TMEM buffer
        const uint32_t sA = smem_u32(smem + s * kStage2), sB = sA + kStageA2;
        mbar_wait_guard(full_bar(s), (k >> 2) & 1, 0);
        mbar_wait_guard(tempty_bar(s), ((k >> 2) & 1) ^ 1, 0);
        tc_fence_after();
        for (int hl = 0; hl < 2; ++hl) {
          const uint64_t dv = make_smem_desc_ex(sB + hl * 2 * kBPanel, kBPanel >> 4, 1024 >> 4);
          const uint64_t dw = make_smem_desc(sA + hl * kAHead);
          for (int ks = 0; ks < ksteps; ++ks)
            umma_bf16(tmem_base + (uint32_t)(s * 128 + hl * 64), dv + (uint64_t)(ks * 128), dw + (uint64_t)(ks * 2), idesc, ks ? 1u : 0u);
        }
        umma_commit(tfull_bar(s));                                              // the epilogue frees the stage (empty_bar)
      }
    }
  } else if (warp >= 2 && warp < 10) {
    // ===================================================================== epilogue: lane = channel, registers = the graph's nodes
    // (rows of scripted nodes and rows beyond the graph are all-zero weight rows -> exactly 0)
    const int quarter = warp & 3, hl = (warp - 2) >> 2;
    for (int k = 0; k < n_items; ++k) {
      const int b = k & 3, hp = k & 1;
      const int tile = blockIdx.x + (k >> 1) * gridDim.x;
      const int g0 = tile * G;
      mbar_wait_guard(tfull_bar(b), (k >> 2) & 1, 20);
      tc_fence_after();
      const int h = hp * 2 + hl;
      float pool = 0.f;                          // relu(conv) * dm >= 0: 0 is the identity of max and add here
#pragma unroll 1
      for (int q = 0; q < 2; ++q) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(b * 128 + hl * 64 + q * 32), v);
        if (q == 1) { tc_fence_before(); mbar_arrive(tempty_bar(b)); }
        if (a.pool_mode == MLS_POOL_MAX) {
#pragma unroll
          for (int t = 0; t < 32; ++t) pool = fmaxf(pool, __uint_as_float(v[t]));
        } else {
#pragma unroll
          for (int t = 0; t < 32; ++t) pool += fmaxf(__uint_as_float(v[t]), 0.f);
        }
        if (q == 1) {
          if (a.pool_mode == MLS_POOL_MEAN) pool = pool / (float)N;
          a.z[(size_t)g0 * a.ldz + a.z_col + h * kC + quarter * 32 + lane] = __float2bfloat16_rn(pool);
        }
      }
      if (threadIdx.x == 64) mbar_arrive(empty_bar(b));                         // stage free for its producer team
    }
  } else if (warp >= 10) {
    // ===================================================================== producer teams
    const int team = (warp - 10) / 3, pt = ((warp - 10) % 3) * 32 + lane;      // 0..95
    const int hp = team & 1;
    const int self = a.transformer ? 0 : 1;
    const int cpg = csr_stride(N) / 16;                                         // 16-byte chunks of a graph's CSR lists
    unsigned char* sA = smem + team * kStage2;
    unsigned char* sBv = sA + kStageA2;
    const uint32_t sB32 = smem_u32(sBv);
    uint8_t* src_s = meta + team * kMeta;                                       // [gt][N*32]
    uint16_t* cid = reinterpret_cast<uint16_t*>(src_s + kMetaSrc);              // [64] compact key id of every tile row
    uint16_t* ptr_s = cid + 64;                                                 // [gt][N+1]
    float* dm_s = reinterpret_cast<float*>(ptr_s + 128);                        // [64] decision-maker flag
    const int gp = pt & 3;
    const unsigned char* gsrc = reinterpret_cast<const unsigned char*>(a.Vh) + hp * 512 + gp * 16;   // this pair's half of a value row
    uint32_t bias_hl[3];                                                        // channels pt, pt + 96, pt + 192 of the pair
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int chl = pt + r * kPoolTeam;
      const float bv = (a.bias && chl < 256) ? a.bias[hp * 256 + chl] : 0.f;
      const __half hi = __float2half_rn(bv), lo = __float2half_rn(bv - __half2float(hi));
      bias_hl[r] = (uint32_t)__half_as_ushort(hi) | ((uint32_t)__half_as_ushort(lo) << 16);
    }
    int use = 0;
    for (int k = team; k < n_items; k += 4, ++use) {
      const int tile = blockIdx.x + (k >> 1) * gridDim.x;
      const int g0 = tile * G, gt = min(G, a.n_graphs - g0), rt = gt * N;
      const size_t m0 = (size_t)g0 * N;
      // ---- phase A: tile metadata (global loads first) and the cleared weight matrices
      uint32_t pv = 0;
      uint16_t cv = 0;
      uint4 sv0 = make_uint4(0, 0, 0, 0), sv1 = make_uint4(0, 0, 0, 0);
      float dmv = 1.f;
      if (pt < rt) {
        cv = __ldg(a.row_cid + m0 + pt);
        dmv = __ldg(a.obs + (long long)(g0 + pt / N) * a.obs_stride + (pt % N) * 8 + 7);
      }
      if (pt < gt * (N + 1)) {                                                 // gt * (N + 1) <= 64
        const int gl = pt / (N + 1), il = pt - gl * (N + 1);
        const size_t cg = a.graph_id ? (size_t)__ldg(a.graph_id + (size_t)(g0 + gl) * a.gid_stride) : (size_t)(g0 + gl);
        pv = __ldg(a.csr_ptr + cg * (N + 1) + il);
      }
      {                                                                        // csr_stride(N) bytes (cpg chunks of 16 B) per graph: <= 128 chunks
        const int c0 = pt, c1 = pt + kPoolTeam;
        if (c0 < gt * cpg) {
          const int gl = c0 / cpg, cl = c0 - gl * cpg;
          const size_t cg = a.graph_id ? (size_t)__ldg(a.graph_id + (size_t)(g0 + gl) * a.gid_stride) : (size_t)(g0 + gl);
          sv0 = __ldg(reinterpret_cast<const uint4*>(a.csr_src + cg * csr_stride(N)) + cl);
        }
        if (c1 < gt * cpg) {
          const int gl = c1 / cpg, cl = c1 - gl * cpg;
          const size_t cg = a.graph_id ? (size_t)__ldg(a.graph_id + (size_t)(g0 + gl) * a.gid_stride) : (size_t)(g0 + gl);
          sv1 = __ldg(reinterpret_cast<const uint4*>(a.csr_src + cg * csr_stride(N)) + cl);
        }
      }
      mbar_wait_guard(empty_bar(team), (use & 1) ^ 1, 40);                     // the epilogue is done with this stage
      for (int u = pt; u < kStageA2 / 16; u += kPoolTeam) reinterpret_cast<uint4*>(sA)[u] = make_uint4(0, 0, 0, 0);
      if (use == 0) {
        // bias rows (kb, kb + 1) of the pair's 4 panels and the rows behind them, once: every tile has the same rows
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const int chl = pt + r * kPoolTeam;
          if (chl < 256) {
            unsigned char* panel = sBv + (chl >> 6) * kBPanel;
            const int e = chl & 63;
            *reinterpret_cast<uint16_t*>(panel + kb * 128 + ((((e >> 3) ^ kb) & 7) << 4) + (e & 7) * 2) = (uint16_t)(bias_hl[r] & 0xffffu);
            *reinterpret_cast<uint16_t*>(panel + (kb + 1) * 128 + ((((e >> 3) ^ (kb + 1)) & 7) << 4) + (e & 7) * 2) = (uint16_t)(bias_hl[r] >> 16);
          }
        }
        const int tail = 62 - rt;                                              // rows rt .. 63 of the 4 panels except kb, kb + 1
        for (int u = pt; u < tail * 32; u += kPoolTeam) {
          int row = rt + (u >> 5);
          if (row >= kb) row += 2;
          const int pc = u & 31;                                               // panel = pc >> 3, 16-byte chunk = pc & 7
          *reinterpret_cast<uint4*>(sBv + (pc >> 3) * kBPanel + row * 128 + ((pc & 7) << 4)) = make_uint4(0, 0, 0, 0);
        }
      }
      if (pt < rt) { cid[pt] = cv; dm_s[pt] = dmv; }
      if (pt < gt * (N + 1)) ptr_s[pt] = (uint16_t)pv;
      if (pt < gt * cpg) reinterpret_cast<uint4*>(src_s)[pt] = sv0;
      if (pt + kPoolTeam < gt * cpg) reinterpret_cast<uint4*>(src_s)[pt + kPoolTeam] = sv1;
      bar_pool_team(team);
      // ---- phase B: this pair's half (512 B) of the value rows of the tile's nodes, asynchronously ...
      for (int j = pt >> 2; j < rt; j += kPoolTeam / 4) {
        const unsigned char* src = gsrc + (size_t)cid[j] * (HC * 2);
        const uint32_t row = sB32 + j * 128;
        const uint32_t d0 = row + ((gp ^ (j & 7)) << 4), d1 = row + (((gp + 4) ^ (j & 7)) << 4);
#pragma unroll
        for (int i = 0; i < 8; ++i) cp_async16(((i & 1) ? d1 : d0) + (i >> 1) * kBPanel, src + i * 64);
      }
      // ---- ... and the normalised softmax weights of (target i, head hl of the pair): weight row i
      for (int tt = pt; tt < rt * 2; tt += kPoolTeam) {
        const int i = tt >> 1, hl = tt & 1, h = hp * 2 + hl;
        if (dm_s[i] == 0.f) continue;                                           // relu(conv) * 0: the row stays all zero
        const int gl = i / N, il = i - gl * N, rbase = gl * N;
        const uint16_t* ptr = ptr_s + gl * (N + 1);
        const int r0 = ptr[il], d = (int)ptr[il + 1] - r0;
        const uint8_t* src = src_s + gl * csr_stride(N) + r0;
        const float* Erow = a.E + (size_t)cid[i] * kAttnUcap * 4 + h;
        const int cnt = d + self;
        unsigned char* arow = sA + hl * kAHead;
        float ev[8];
        int jv[8];
        float mx = -INFINITY;
        for (int k0 = 0; k0 < cnt; k0 += 8) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const int kk = k0 + q;
            jv[q] = (kk < cnt && kk >= self) ? rbase + src[kk - self] : i;
            ev[q] = __ldg(Erow + (int)cid[jv[q]] * 4);
          }
#pragma unroll
          for (int q = 0; q < 8; ++q) if (k0 + q < cnt) mx = fmaxf(mx, ev[q]);
        }
        float sum = 0.f;
        if (cnt <= 8) {
#pragma unroll
          for (int q = 0; q < 8; ++q) { ev[q] = q < cnt ? f_ex2(ev[q] - mx) : 0.f; sum += ev[q]; }
        } else {
          for (int kk = 0; kk < cnt; ++kk) {
            const int j = kk >= self ? rbase + src[kk - self] : i;
            sum += f_ex2(__ldg(Erow + (int)cid[j] * 4) - mx);
          }
        }
        const float inv = f_rcp(sum + 1e-16f);
        if (cnt <= 8) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (q < cnt) *reinterpret_cast<__half*>(arow + a_off(i, jv[q])) = __float2half_rn(ev[q] * inv);
        } else {
          for (int kk = 0; kk < cnt; ++kk) {
            const int j = kk >= self ? rbase + src[kk - self] : i;
            *reinterpret_cast<__half*>(arow + a_off(i, j)) = __float2half_rn(f_ex2(__ldg(Erow + (int)cid[j] * 4) - mx) * inv);
          }
        }
        *reinterpret_cast<uint16_t*>(arow + a_off(i, kb)) = 0x3C00;          // 1.0 (fp16): + bias (hi)
        *reinterpret_cast<uint16_t*>(arow + a_off(i, kb + 1)) = 0x3C00;      // 1.0 (fp16): + bias (lo)
      }
      cp_async_wait_all();
      fence_proxy_async();
      mbar_arrive(full_bar(team));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------ per-tile records + row-major MMA kernel
// A producer team that builds a whole item itself spends its time in a per-item PROGRAM (metadata loads, ballots, need
// list, CSR walk, pair-logit reads, softmax: chains of dependent latencies run by 2-3 warps; profiles/
// r02_conv1_experiments.txt).  Here that program runs ONCE per tile in a full-occupancy pre-pass (one warp per tile, all
// four heads from one float4 table read) that leaves a record per tile:
//     hdr {nn, ne, 0, 0} | x_out row of every needed target [64] | compact key id of every tile row [64]
//     | entries: (target rank << 8 | source row) [ne] | normalised softmax weights fp16 [4 heads][ne]
// and the MMA kernel's producers only move data: three bulk copies (cp.async.bulk -> mbarrier) bring the record's fixed
// part and the head's entry list into the stage, the value rows are gathered with cp.async by the record's key ids, and the
// weights are scattered into the (cleared) K-major weight tile.
//   D[target][channel] = W[target][source] (A, K-major) x V[source][channel] (B, MN-major), M = 128, N = 128 per (tile, head)
// item; a TMEM lane is a target: an epilogue thread adds the conv bias, converts and writes 16-byte pieces of its target's
// x1 row through a transposition tile (whole 128-byte row segments per store).  Six 24 KiB stages / producer teams of 2
// warps; four independent pairs of DRAIN warps (pair g owns head g and TMEM buffer g; TMEM -> tile) each followed by its
// STORE warp (tile -> global); a stage returns to its team on tcgen05.commit.
constexpr int kRecFixed = 16 + 64 * 4 + 64 * 2;            // 400 bytes: header, x_out rows, key ids (a multiple of 16: bulk copies)
constexpr int kRecChunk = 512;                             // entries per in-kernel chunk
__host__ __device__ inline int rec_entry_cap(int rows) { return (rows * (kMaxList + 1) + 7) & ~7; }   // sources + self loop
__host__ __device__ inline int rec_stride(int rows) { return kRecFixed + 10 * rec_entry_cap(rows); }

// One warp per tile.  Lane l owns tile rows l and l + 32.
__global__ void __launch_bounds__(256, 4) attn_table_prep_kernel(const AttnTableArgs a, const int G) {
  if (*a.n_used > kAttnUcap) return;
  __shared__ uint16_t cid_sm[8][64], p0_sm[8][64], off_sm[8][64];
  __shared__ uint8_t need_sm[8][64], cnt_sm[8][64];
  __shared__ int cg_sm[8][64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N;
  const int n_tiles = (a.n_graphs + G - 1) / G;
  const int tile = blockIdx.x * 8 + warp;
  if (tile >= n_tiles) return;
  const int g0 = tile * G, gt = min(G, a.n_graphs - g0), rt = gt * N;
  const size_t m0 = (size_t)g0 * N;
  const int self = a.transformer ? 0 : 1;
  unsigned char* rec = a.rec + (size_t)tile * rec_stride(G * N);
  const int cap = rec_entry_cap(G * N);
  uint16_t* cid_s = cid_sm[warp];
  uint16_t* p0_s = p0_sm[warp];
  uint16_t* off_s = off_sm[warp];
  uint8_t* need_s = need_sm[warp];
  uint8_t* cnt_s = cnt_sm[warp];
  int* cg_s = cg_sm[warp];
  int xr[2], cnt[2], p0[2], gl[2];
  uint16_t cv[2];
  const uint8_t* srcp[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int r = lane + 32 * q;
    xr[q] = -1; cnt[q] = 0; cv[q] = 0; p0[q] = 0; gl[q] = 0; srcp[q] = nullptr;
    if (r < rt) {
      cv[q] = __ldg(a.row_cid + m0 + r);
      xr[q] = a.xrow ? __ldg(a.xrow + m0 + r) : (int)m0 + r;
      gl[q] = r / N;
      const int il = r - gl[q] * N;
      const size_t cg = a.graph_id ? (size_t)__ldg(a.graph_id + (size_t)(g0 + gl[q]) * a.gid_stride) : (size_t)(g0 + gl[q]);
      p0[q] = __ldg(a.csr_ptr + cg * (N + 1) + il);
      const int d = (int)__ldg(a.csr_ptr + cg * (N + 1) + il + 1) - p0[q];
      srcp[q] = a.csr_src + cg * csr_stride(N) + p0[q];
      if (xr[q] >= 0) cnt[q] = d + self;
      if (il == 0) cg_s[gl[q]] = (int)cg;
    }
    cid_s[r] = cv[q];
    p0_s[r] = (uint16_t)p0[q];
    cnt_s[r] = (uint8_t)cnt[q];
  }
  __syncwarp();
  const uint32_t lt = (1u << lane) - 1u;
  const uint32_t b0 = __ballot_sync(0xffffffffu, xr[0] >= 0), b1 = __ballot_sync(0xffffffffu, xr[1] >= 0);
  const int n0 = __popc(b0), nn = n0 + __popc(b1);
  const int rank[2] = {__popc(b0 & lt), n0 + __popc(b1 & lt)};
  // entry offsets in rank order: rows 0..31 first, then 32..63 (ranks are assigned the same way)
  int inc0 = cnt[0], inc1 = cnt[1];
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v0 = __shfl_up_sync(0xffffffffu, inc0, o), v1 = __shfl_up_sync(0xffffffffu, inc1, o);
    if (lane >= o) { inc0 += v0; inc1 += v1; }
  }
  const int tot0 = __shfl_sync(0xffffffffu, inc0, 31), ne = tot0 + __shfl_sync(0xffffffffu, inc1, 31);
  const int off[2] = {inc0 - cnt[0], tot0 + inc1 - cnt[1]};
  const int ne_pad = (ne + 7) & ~7;
  if (lane == 0) {
    *reinterpret_cast<int4*>(rec) = make_int4(nn, ne, 0, 0);
    a.tile_idx[tile] = make_int2(ne_pad, nn);
  }
  int* tab_x = reinterpret_cast<int*>(rec + 16);
  uint16_t* cid_g = reinterpret_cast<uint16_t*>(rec + 16 + 256);
  uint16_t* jr = reinterpret_cast<uint16_t*>(rec + kRecFixed);
  __half* wts = reinterpret_cast<__half*>(rec + kRecFixed + 2 * cap);          // [4][cap]
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int r = lane + 32 * q;
    cid_g[r] = cv[q];
    if (xr[q] >= 0) { tab_x[rank[q]] = xr[q]; need_s[rank[q]] = (uint8_t)r; off_s[rank[q]] = (uint16_t)off[q]; }
  }
  __syncwarp();
  // padding entries (read by the 16-byte granular copies, never scattered): keep them defined
  if (lane < ne_pad - ne) {
    jr[ne + lane] = 0;
    for (int h = 0; h < 4; ++h) wts[(size_t)h * cap + ne + lane] = __float2half_rn(0.f);
  }
  // one needed target per lane, in rank order (at most 32 of them in the typical tile: a single pass with every lane's
  // table reads in flight together, instead of one pass per half of the tile's rows)
#pragma unroll 1
  for (int rki = lane; rki < nn; rki += 32) {
    const int r = need_s[rki], c = cnt_s[r];
    if (c == 0) continue;
    const int glr = r / N, rbase = glr * N;
    const float4* Erow = reinterpret_cast<const float4*>(a.E) + (size_t)cid_s[r] * kAttnUcap;
    const uint8_t* src = a.csr_src + (size_t)cg_s[glr] * csr_stride(N) + p0_s[r];
    uint16_t* jo = jr + off_s[rki];
    __half* wo = wts + off_s[rki];
    const int rk = rki << 8;
    if (c <= 8) {
      float4 e[8];
      int jv[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        jv[k] = (k < c && k >= self) ? rbase + src[k - self] : r;
        e[k] = __ldg(Erow + cid_s[jv[k]]);
      }
      float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < c) { mx.x = fmaxf(mx.x, e[k].x); mx.y = fmaxf(mx.y, e[k].y); mx.z = fmaxf(mx.z, e[k].z); mx.w = fmaxf(mx.w, e[k].w); }
      float4 sm = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < c) {
          e[k].x = f_ex2(e[k].x - mx.x); e[k].y = f_ex2(e[k].y - mx.y); e[k].z = f_ex2(e[k].z - mx.z); e[k].w = f_ex2(e[k].w - mx.w);
          sm.x += e[k].x; sm.y += e[k].y; sm.z += e[k].z; sm.w += e[k].w;
        }
      const float4 inv = make_float4(f_rcp(sm.x + 1e-16f), f_rcp(sm.y + 1e-16f), f_rcp(sm.z + 1e-16f), f_rcp(sm.w + 1e-16f));
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < c) {
          jo[k] = (uint16_t)(rk | jv[k]);
          wo[k] = __float2half_rn(e[k].x * inv.x); wo[cap + k] = __float2half_rn(e[k].y * inv.y);
          wo[2 * cap + k] = __float2half_rn(e[k].z * inv.z); wo[3 * cap + k] = __float2half_rn(e[k].w * inv.w);
        }
    } else {
      float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      for (int k = 0; k < c; ++k) {
        const int j = k >= self ? rbase + src[k - self] : r;
        const float4 v = __ldg(Erow + cid_s[j]);
        mx.x = fmaxf(mx.x, v.x); mx.y = fmaxf(mx.y, v.y); mx.z = fmaxf(mx.z, v.z); mx.w = fmaxf(mx.w, v.w);
      }
      float4 sm = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int k = 0; k < c; ++k) {
        const int j = k >= self ? rbase + src[k - self] : r;
        const float4 v = __ldg(Erow + cid_s[j]);
        sm.x += f_ex2(v.x - mx.x); sm.y += f_ex2(v.y - mx.y); sm.z += f_ex2(v.z - mx.z); sm.w += f_ex2(v.w - mx.w);
      }
      const float4 inv = make_float4(f_rcp(sm.x + 1e-16f), f_rcp(sm.y + 1e-16f), f_rcp(sm.z + 1e-16f), f_rcp(sm.w + 1e-16f));
      for (int k = 0; k < c; ++k) {
        const int j = k >= self ? rbase + src[k - self] : r;
        const float4 v = __ldg(Erow + cid_s[j]);
        jo[k] = (uint16_t)(rk | j);
        wo[k] = __float2half_rn(f_ex2(v.x - mx.x) * inv.x); wo[cap + k] = __float2half_rn(f_ex2(v.y - mx.y) * inv.y);
        wo[2 * cap + k] = __float2half_rn(f_ex2(v.z - mx.z) * inv.z); wo[3 * cap + k] = __float2half_rn(f_ex2(v.w - mx.w) * inv.w);
      }
    }
  }
}

constexpr int kT6Threads = 960;
constexpr int kTeam6 = 64;
constexpr int kNumSt6 = 6;
constexpr int kStage1 = kAHead + 2 * kBPanel;  // 24 KiB
constexpr int kMetaFix = (kRecFixed + 127) & ~127;   // record fixed part rounded up
constexpr int kMeta8 = kMetaFix + 4 * kRecChunk;   // + one chunk of entries (2 B each) and of weights (2 B each)
constexpr int kEpiRow = 144;                   // epilogue staging row: 64 bf16 + 16 B pad (conflict-free 16-byte accesses)
constexpr int kEpiTile = 32 * kEpiRow;         // one warp's transposition tile
constexpr int kT6Smem = kNumSt6 * kStage1 + kNumSt6 * kMeta8 + 8 * kEpiTile + 512 * 4 /*bias*/ + 512 /*barriers*/ + 1024;

__device__ __forceinline__ void bar_team6(int team) { asm volatile("bar.sync %0, 64;" ::"r"(team + 1) : "memory"); }
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint4 relu_pack8(const uint32_t* v) {
  uint4 o;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.x) : "f"(__uint_as_float(v[1])), "f"(__uint_as_float(v[0])));
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.y) : "f"(__uint_as_float(v[3])), "f"(__uint_as_float(v[2])));
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.z) : "f"(__uint_as_float(v[5])), "f"(__uint_as_float(v[4])));
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.w) : "f"(__uint_as_float(v[7])), "f"(__uint_as_float(v[6])));
  return o;
}
// relu(v[0..7] + bias[0..7]) as 8 bf16
__device__ __forceinline__ uint4 bias_relu_pack8(const uint32_t* v, const float* bias) {
  const float4 b0 = *reinterpret_cast<const float4*>(bias), b1 = *reinterpret_cast<const float4*>(bias + 4);
  uint4 o;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.x) : "f"(__uint_as_float(v[1]) + b0.y), "f"(__uint_as_float(v[0]) + b0.x));
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.y) : "f"(__uint_as_float(v[3]) + b0.w), "f"(__uint_as_float(v[2]) + b0.z));
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.z) : "f"(__uint_as_float(v[5]) + b1.y), "f"(__uint_as_float(v[4]) + b1.x));
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(o.w) : "f"(__uint_as_float(v[7]) + b1.w), "f"(__uint_as_float(v[6]) + b1.z));
  return o;
}

__global__ void __launch_bounds__(kT6Threads, 1) attn_table_rows_kernel(const AttnTableArgs a, const int G) {
  if (*a.n_used > kAttnUcap) return;            // uniform: the gather kernel handles this pass
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* meta = smem + kNumSt6 * kStage1;                                 // [6][kMeta8]
  unsigned char* epi_tiles = meta + kNumSt6 * kMeta8;                             // [8][kEpiTile]
  float* bias_s = reinterpret_cast<float*>(epi_tiles + 8 * kEpiTile);             // [512]
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + 512);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 56);
  const uint32_t bar0 = smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (8 + s); };
  auto meta_bar = [&](int s) { return bar0 + 8u * (16 + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (24 + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (28 + b); };
  auto tile_full_bar = [&](int w) { return bar0 + 8u * (32 + w); };
  auto tile_free_bar = [&](int w) { return bar0 + 8u * (40 + w); };

  const int N = a.N, HC = 4 * kC;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (a.n_graphs + G - 1) / G;
  const int my_tiles = blockIdx.x < n_tiles ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int n_items = 4 * my_tiles;              // item k: tile blockIdx.x + (k >> 2) * gridDim.x, head k & 3, stage k % 6
  const int ksteps = (G * N + 8 <= 64) ? 4 : ((G * N + 15) >> 4);   // value rows behind the tile's nodes: bias rows or zero
  const int stride = rec_stride(G * N), cap = rec_entry_cap(G * N);

  for (int u = threadIdx.x; u < kNumSt6 * kStage1 / 16; u += kT6Threads) reinterpret_cast<uint4*>(smem)[u] = make_uint4(0, 0, 0, 0);
  // conv bias: as 8 extra value rows (fp16 hi + lo for each of the 4 heads, rows kb + 2h, kb + 2h + 1 of every stage; the
  // weight rows of head h carry ones in those two columns) when the tile leaves room for them, else added in the epilogue
  const int kb = G * N;
  const bool bias_mma = kb + 8 <= 64;
  for (int u = threadIdx.x; u < 512; u += kT6Threads) bias_s[u] = (a.bias && !bias_mma) ? a.bias[u] : 0.f;
  __syncthreads();
  if (bias_mma) {
    for (int u = threadIdx.x; u < kNumSt6 * 512; u += kT6Threads) {
      const int st = u >> 9, hh = (u >> 7) & 3, ch = u & 127;                 // head hh's bias for channel ch -> rows kb + 2 hh (+1)
      const float bv = a.bias ? a.bias[hh * kC + ch] : 0.f;
      const __half hi = __float2half_rn(bv), lo = __float2half_rn(bv - __half2float(hi));
      unsigned char* panel = smem + st * kStage1 + kAHead + (ch >> 6) * kBPanel;
      const int e = ch & 63, r0 = kb + 2 * hh;
      *reinterpret_cast<__half*>(panel + r0 * 128 + ((((e >> 3) ^ r0) & 7) << 4) + (e & 7) * 2) = hi;
      *reinterpret_cast<__half*>(panel + (r0 + 1) * 128 + ((((e >> 3) ^ (r0 + 1)) & 7) << 4) + (e & 7) * 2) = lo;
    }
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < kNumSt6; ++s) { mbar_init(full_bar(s), kTeam6); mbar_init(empty_bar(s), 1 + 2); mbar_init(meta_bar(s), 1); }
    for (int b = 0; b < 4; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 2 * 32); }
    for (int w = 0; w < 8; ++w) { mbar_init(tile_full_bar(w), 32); mbar_init(tile_free_bar(w), 32); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const bool is_epi = warp >= 4 && warp < 18 && (warp & 3) < 2;
  const bool is_store = warp >= 22;
  const bool is_prod = warp >= 2 && !is_epi && !is_store;
  if (warp == 0) {
    // ===================================================================== MMA issuer
    if (lane == 0) {
      // fp16 x fp16 (format fields cleared), B (values) MN-major (bit 16)
      const uint32_t idesc = (make_idesc(128, 128) & ~((7u << 7) | (7u << 10))) | (1u << 16);
      int s = 0;
      uint32_t sph = 0;
      for (int k = 0; k < n_items; ++k) {
        const int b = k & 3;
        const uint32_t sA = smem_u32(smem + s * kStage1), sB = sA + kAHead;
        mbar_wait_guard(full_bar(s), sph, 0);
        mbar_wait_guard(tempty_bar(b), ((k >> 2) & 1) ^ 1, 0);
        tc_fence_after();
        // A = weight rows [target][source]; the descriptor spans 128 rows, the tile holds 64: rows 64.. are whatever
        // follows in the stage (finite fp16) and only reach TMEM lanes 64.. , which nobody reads
        const uint64_t dw = make_smem_desc(sA);
        const uint64_t dv = make_smem_desc_ex(sB, kBPanel >> 4, 1024 >> 4);
        for (int ks = 0; ks < ksteps; ++ks)
          umma_bf16(tmem_base + (uint32_t)(b * 128), dw + (uint64_t)(ks * 2), dv + (uint64_t)(ks * 128), idesc, ks ? 1u : 0u);
        umma_commit(empty_bar(s));                                              // operands read: the stage goes back to its team
        umma_commit(tfull_bar(b));
        if (++s == kNumSt6) { s = 0; sph ^= 1u; }
      }
    }
  } else if (is_epi) {
    // ===================================================================== epilogue: lane = target, registers = channels
    // Tiles with at most 32 needed targets (the rule at N = 50) carry every weight row twice, at rows t and t + 32: the
    // lane quarters 0 and 1 hold the same targets and split the head's 128 channels; larger tiles: quarter = targets
    // 32 qq .., all 128 channels.  64 channels at a time go through the warp's private transposition tile so that a store
    // instruction writes whole 128-byte row segments (per-lane 16-byte pieces of 32 different rows are one L2 request
    // each: 0.39 ms of this kernel).
    const int qq = warp & 3, b = (warp >> 2) - 1;                              // b == head == accumulator buffer
    // Drain warps (this branch) move the accumulator into the pair's transposition tile; a STORE warp per drain warp
    // (below) writes the rows out, so that the address arithmetic / global stores of item k overlap the tcgen05.ld /
    // conversion of item k + 4 (the epilogue was the kernel's limiter: its warps were 75 % busy).  A tile row = 128 bytes of
    // channels + 16 bytes {x1 row, rows in the tile (-1: stop), byte offset inside a row, 0}.
    const int dw = b * 2 + qq;
    unsigned char* tile_s = epi_tiles + dw * kEpiTile;
    uint32_t msg = 0;
    int s = b % kNumSt6;
    for (int k = b; k < n_items; k += 4) {
      mbar_wait_guard(tfull_bar(b), (k >> 2) & 1, 20);
      tc_fence_after();
      const int4 hdr = *reinterpret_cast<const int4*>(meta + s * kMeta8);      // {nn, ne, 0, 0}
      const int* tab_x = reinterpret_cast<const int*>(meta + s * kMeta8 + 16);
      const int nn = hdr.x;
      const bool rep = nn <= 32;
      const int t0 = rep ? 0 : qq * 32;                                        // first target of this warp's TMEM lanes
      const int nv = max(0, min(32, nn - t0));                                 // targets among them
      int xr = 0;
      if (lane < nv) xr = tab_x[t0 + lane];
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar(s));                                // this warp is done with the stage's record
      s += 4; if (s >= kNumSt6) s -= kNumSt6;
      const int c0 = rep ? qq * 64 : 0, nhalf = rep ? 1 : 2;                   // this warp's channels of the head: [c0, c0 + 64 nhalf)
      const uint32_t tcol = tmem_base + ((uint32_t)(qq * 32) << 16) + (uint32_t)(b * 128 + c0);
      for (int hf = 0; hf < nhalf; ++hf) {
        mbar_wait_guard(tile_free_bar(dw), (msg & 1u) ^ 1u, 20);               // the store warp has read the previous tile
        if (nv > 0) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t v[32];
            tmem_ld32(tcol + (uint32_t)(hf * 64 + c * 32), v);
            const float* bp = bias_s + b * kC + c0 + hf * 64 + c * 32;
            if (bias_mma) {
#pragma unroll
              for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(tile_s + lane * kEpiRow + c * 64 + q * 16) = relu_pack8(v + 8 * q);
            } else {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(tile_s + lane * kEpiRow + c * 64 + q * 16) = bias_relu_pack8(v + 8 * q, bp + 8 * q);
            }
          }
        }
        *reinterpret_cast<int4*>(tile_s + lane * kEpiRow + 128) = make_int4(xr, nv, (b * kC + c0 + hf * 64) * 2, 0);
        if (hf == nhalf - 1) { tc_fence_before(); mbar_arrive(tempty_bar(b)); }   // accumulator drained
        mbar_arrive(tile_full_bar(dw));
        ++msg;
      }
    }
    mbar_wait_guard(tile_free_bar(dw), (msg & 1u) ^ 1u, 20);
    *reinterpret_cast<int4*>(tile_s + lane * kEpiRow + 128) = make_int4(0, -1, 0, 0);    // stop
    mbar_arrive(tile_full_bar(dw));
  } else if (is_store) {
    // ===================================================================== store warps: tile -> x1 rows
    const int sw = warp - 22;
    const unsigned char* tile_s = epi_tiles + sw * kEpiTile;
    const int srow = lane >> 3, schunk = lane & 7;                             // 4 rows x 8 chunks per instruction
    for (uint32_t msg = 0;; ++msg) {
      mbar_wait_guard(tile_full_bar(sw), msg & 1u, 20);
      const int nv = reinterpret_cast<const int*>(tile_s + 128)[1];
      if (nv < 0) break;
      for (int r0 = 0; r0 < nv; r0 += 4) {
        const int r = r0 + srow;
        if (r < nv) {
          const int4 pd = *reinterpret_cast<const int4*>(tile_s + r * kEpiRow + 128);
          const uint4 val = *reinterpret_cast<const uint4*>(tile_s + r * kEpiRow + schunk * 16);
          *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(a.x_out) + (size_t)pd.x * (HC * 2) + pd.z + schunk * 16) = val;
        }
      }
      __syncwarp();
      mbar_arrive(tile_free_bar(sw));
    }
  } else if (is_prod) {
    // ===================================================================== producer teams: data movement only
    const int p = warp >= 20 ? warp - 10 : ((warp - 2) >> 2) * 2 + ((warp - 2) & 1);   // 0..11
    const int team = p >> 1, pt = (p & 1) * 32 + lane;                         // 0..63
    unsigned char* sA = smem + team * kStage1;
    const uint32_t sB32 = smem_u32(sA + kAHead);
    unsigned char* mt = meta + team * kMeta8;
    const uint16_t* cid = reinterpret_cast<const uint16_t*>(mt + 16 + 256);     // [64] compact key id of every tile row
    const uint16_t* jr_s = reinterpret_cast<const uint16_t*>(mt + kMetaFix);    // [kRecChunk]
    const __half* w_s = reinterpret_cast<const __half*>(mt + kMetaFix + 2 * kRecChunk);
    const uint32_t mt32 = smem_u32(mt), mbar = meta_bar(team);
    const int gp = pt & 3;
    auto load_idx = [&](int k) -> int2 {
      if (k >= n_items) return make_int2(0, 0);
      return __ldg(a.tile_idx + blockIdx.x + (k >> 2) * gridDim.x);
    };
    int2 ix = load_idx(team);
    uint32_t mph = 0;
    int use = 0;
    for (int k = team; k < n_items; k += kNumSt6, ++use) {
      const int tile = blockIdx.x + (k >> 2) * gridDim.x, h = k & 3;
      const int g0 = tile * G, gt = min(G, a.n_graphs - g0), rt = gt * N;
      const int ne_pad = ix.x, nn = ix.y;
      ix = load_idx(k + kNumSt6);                                               // next item's sizes: in flight during this one
      const bool rep = nn <= 32;
      const unsigned char* rec = a.rec + (size_t)tile * stride;
      const unsigned char* gsrc = reinterpret_cast<const unsigned char*>(a.Vh) + h * (kC * 2) + gp * 16;   // this head's quarter of a value row
      mbar_wait_guard(empty_bar(team), (use & 1) ^ 1, 40);                     // MMAs and epilogue are done with this stage
      int c0 = 0, cn = ne_pad < kRecChunk ? ne_pad : kRecChunk;                 // first chunk of entries
      if (pt == 0) {
        mbar_expect_tx(mbar, (uint32_t)(kRecFixed + 4 * cn));
        bulk_g2s(mt32, rec, kRecFixed, mbar);
        if (cn > 0) {
          bulk_g2s(mt32 + kMetaFix, rec + kRecFixed, 2 * cn, mbar);
          bulk_g2s(mt32 + kMetaFix + 2 * kRecChunk, rec + kRecFixed + 2 * (size_t)cap * (1 + h), 2 * cn, mbar);
        }
      }
      // weight rows of the needed targets, cleared (rows behind them keep stale finite data: their TMEM lanes are not read)
      for (int u = pt; u < nn * 8; u += kTeam6) {
        reinterpret_cast<uint4*>(sA)[u] = make_uint4(0, 0, 0, 0);
        if (rep) reinterpret_cast<uint4*>(sA + 32 * 128)[u] = make_uint4(0, 0, 0, 0);
      }
      mbar_wait_guard(mbar, mph, 20);                                           // the record is here
      mph ^= 1u;
      // this head's quarter (256 B) of the value rows of the tile's nodes, asynchronously
      for (int j = pt >> 2; j < rt; j += kTeam6 / 4) {
        const unsigned char* src = gsrc + (size_t)cid[j] * (HC * 2);
        const uint32_t row = sB32 + j * 128;
        const uint32_t d0 = row + ((gp ^ (j & 7)) << 4), d1 = row + (((gp + 4) ^ (j & 7)) << 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) cp_async16(((i & 1) ? d1 : d0) + (i >> 1) * kBPanel, src + i * 64);
      }
      bar_team6(team);                                                         // weight rows cleared by everybody
      const int rep_off = rep ? 32 * 128 : 0;
      const int ne = reinterpret_cast<const int*>(mt)[1];                       // real entries (the copies are 16-byte granular)
      for (;;) {
        const int ce = min(cn, ne - c0);
        for (int e = pt; e < ce; e += kTeam6) {
          const uint32_t ent = jr_s[e];
          unsigned char* cell = sA + a_off((int)(ent >> 8), (int)(ent & 255u));
          const __half w = w_s[e];
          *reinterpret_cast<__half*>(cell) = w;
          *reinterpret_cast<__half*>(cell + rep_off) = w;
        }
        c0 += cn;
        if (c0 >= ne_pad) break;
        bar_team6(team);                                                       // everybody has read this chunk
        cn = ne_pad - c0 < kRecChunk ? ne_pad - c0 : kRecChunk;
        if (pt == 0) {
          mbar_expect_tx(mbar, (uint32_t)(4 * cn));
          bulk_g2s(mt32 + kMetaFix, rec + kRecFixed + 2 * (size_t)c0, 2 * cn, mbar);
          bulk_g2s(mt32 + kMetaFix + 2 * kRecChunk, rec + kRecFixed + 2 * (size_t)cap * (1 + h) + 2 * (size_t)c0, 2 * cn, mbar);
        }
        mbar_wait_guard(mbar, mph, 20);
        mph ^= 1u;
      }
      if (bias_mma) {                                                          // + bias (hi, lo) of this head
        for (int r = pt; r < nn; r += kTeam6) {
          unsigned char* c0p = sA + a_off(r, kb + 2 * h);
          unsigned char* c1p = sA + a_off(r, kb + 2 * h + 1);
          *reinterpret_cast<uint16_t*>(c0p) = 0x3C00; *reinterpret_cast<uint16_t*>(c1p) = 0x3C00;
          *reinterpret_cast<uint16_t*>(c0p + rep_off) = 0x3C00; *reinterpret_cast<uint16_t*>(c1p + rep_off) = 0x3C00;
        }
      }
      cp_async_wait_all();
      fence_proxy_async();
      mbar_arrive(full_bar(team));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace

size_t attn_table_record_bytes(int N, int n_graphs) {
  const int G = kAttnMaxRows / N;
  const size_t n_tiles = ((size_t)n_graphs + G - 1) / G;
  return n_tiles * (size_t)rec_stride(G * N);
}

int attn_table_conv_launch(const AttnTableArgs& a, int sm_count, cudaStream_t st) {
  if (!attn_table_supported(a.N, a.H)) {
    mls_set_error("table-mode attention: unsupported shape (N=%d, H=%d)", a.N, a.H);
    return MLS_ERR_UNSUPPORTED;
  }
  const bool pool = a.pool_mode >= 0;
  MLS_CHECK_ARG(pool ? a.z && a.obs : a.x_out && a.rec && a.tile_idx,
                "table-mode attention: pooling needs z and obs, the row output needs x_out, rec and tile_idx");
  static bool configured = false;
  if (!configured) {
    MLS_CUDA(cudaFuncSetAttribute(attn_table_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoolSmem));
    MLS_CUDA(cudaFuncSetAttribute(attn_table_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kT6Smem));
    configured = true;
  }
  compact_keys_kernel<<<1, 1024, 0, st>>>(a.used_bits, a.n_keys, a.cid_of_key, a.key_of_cid, a.n_used);
  const int rows = a.n_graphs * a.N;
  row_cid_kernel<<<(rows + 255) / 256, 256, 0, st>>>(a.key, a.cid_of_key, rows, a.row_cid);
  values_fp16_kernel<<<kAttnUcap * 64 / 256, 256, 0, st>>>(a);
  pair_logit_kernel<<<sm_count * 2, 256, 0, st>>>(a);
  const int G = pool ? 1 : kAttnMaxRows / a.N;                  // pooling: one graph per tile
  const int n_tiles = (a.n_graphs + G - 1) / G;
  const int grid = mls_cap_grid(n_tiles < sm_count ? n_tiles : sm_count);   // the persistent kernels take any grid
  if (grid > 0) {
    if (pool) {
      attn_table_pool_kernel<<<grid, kPoolThreads, kPoolSmem, st>>>(a, G);
    } else {
      attn_table_prep_kernel<<<(n_tiles + 7) / 8, 256, 0, st>>>(a, G);
      attn_table_rows_kernel<<<grid, kT6Threads, kT6Smem, st>>>(a, G);
      mls_count_launch();
    }
  }
  mls_count_launch(5);
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}

}  // namespace mls

// Standalone entry for tests/test_gemm_gpu.py: D[128 x 128] = A[rows_a x 64] (K-major) x B[64 x 128] (MN-major), K = kt.
extern "C" int mls_test_umma_mn(const void* A, const void* B, float* D, int rows_a, int kt, unsigned lbo16, unsigned sbo16,
                                unsigned kadv16, void* stream) {
  static bool configured = false;
  if (!configured) {
    MLS_CUDA(cudaFuncSetAttribute(mls::umma_mn_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 40 * 1024));
    configured = true;
  }
  mls::umma_mn_probe_kernel<<<1, 128, 40 * 1024, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const mls::bf16*>(A), reinterpret_cast<const mls::bf16*>(B), D, rows_a, kt, lbo16, sbo16, kadv16);
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}
