// conv2 attention (GATv2Conv / TransformerConv, second layer of L-DGN / DGN-R) on the compacted row sets (sm_100a).
//
// Only controlling nodes are conv2 targets (l_dgn.py:133-139, dgn_r.py:113-118: the network reads x[ctrl] only), and
// only their radius-graph sources are conv2 sources ("needed" rows, ctrl_need_list_kernel).  One work item =
// (graph, head); a persistent 128-thread CTA (head fixed per CTA) runs per item:
//   stage     cp.async of the head's 128-channel fp16 slices: the needed source rows into a [source][channel]
//             MN-major 128B-swizzled operand (GATv2: x_l, which is BOTH the logit operand and the value), the
//             target rows (x_r / q) and (Transformer) the key rows into padded rows; CSR block of the graph
//   logits    one LANE per edge (self loop first for GATv2), 128 channels in packed half2 math
//               GATv2:       e_ij = 0.6 (a_j + b_i) + 0.4 sum_c att_c |x_l[j,c] + x_r[i,c]|   (leaky_relu(s,.2) = .6 s + .4 |s|;
//                            the linear parts come from the projection GEMMs' epilogue dots, fp32)
//               Transformer: e_ij = <q_i, k_j> / sqrt(C)
//             all in base 2 (pre-scaled by log2 e)
//   softmax   4 lanes per target: 2^(e - max) / (sum + 1e-16) (PyG softmax), written as fp16 into the K-major
//             128B-swizzled weight matrix W[target][source]
//   aggregate ONE tcgen05.mma chain, transposed: out^T[channel][target] = X^T[channel][source] x W^T[source][target]
//             (M = 128 channels = the head, N = targets rounded to 16, K = 16 sources per step), fp32 in TMEM
//   epilogue  tcgen05.ld (lane = channel, registers = targets) + conv bias + ReLU -> bf16, 64 contiguous bytes per
//             warp store, straight into the controlling-node snapshot rows z[slot] (slots of a graph are consecutive)
// Reference math: PyG GATv2Conv / TransformerConv(root_weight=False) as called by l_dgn.py:133, dgn_r.py:113.
#include "conv2_attn.cuh"

#include "dgn_kernels.cuh"
#include "tcgen05_ptx.cuh"

namespace mls {

namespace {

constexpr int kThreads = 128;
constexpr int kPanel = 64 * 128;          // one 64-channel panel of the value operand: 64 source rows x 128 B
constexpr int kXBytes = 2 * kPanel;       // the head's 128 channels
constexpr int kRowPad = kC * 2 + 16;      // padded row of 128 fp16 (bank-conflict-free 16 B reads by row-owning lanes)

__device__ __forceinline__ void cp16(unsigned char* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float ex2f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcpf(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ uint16_t relu_bf16_bits(float x) {
  uint16_t d;
  asm("cvt.rn.relu.bf16.f32 %0, %1;" : "=h"(d) : "f"(x));
  return d;
}
// same descriptor helpers as attn_table.cu (SWIZZLE_128B; A operand MN-major)
__device__ __forceinline__ uint64_t desc_mn(uint32_t smem_addr, uint32_t lbo16, uint32_t sbo16) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo16 & 0x3FFFu) << 16;
  d |= (uint64_t)(sbo16 & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Targets are processed in blocks of at most kTB targets and kEdgeCap edge entries (one block for the typical graph:
// ~17 controlling nodes, ~106 entries; the worst case -- 64 targets x 34 entries -- takes several): the per-item shared
// memory is sized for a block, not for the worst case, so that seven CTAs fit an SM.
constexpr int kTB = 32;
constexpr int kEdgeCap = 256;
constexpr int kWRows = kTB;
constexpr int kWTile = kWRows * 128;      // 4 KB
constexpr int kTCols = 32;                // TMEM columns per CTA
constexpr int kCtasPerSm = 7;             // GATv2 form: 31.8 KB + 1 KB reserved per CTA, <= 72 registers (Transformer form: 4)

struct Conv2Layout {       // shared-memory offsets behind the 1024-byte aligned MMA operands
  size_t off_W, off_T, off_K, off_att, off_as, off_bt, off_e, off_eptr, off_ent, off_bar, total;
};
Conv2Layout conv2_layout(bool tr) {
  Conv2Layout L;
  size_t o = kXBytes;
  L.off_W = o; o += kWTile;
  L.off_T = o; o += (size_t)kTB * kRowPad;
  L.off_K = o; o += tr ? (size_t)64 * kRowPad : 0;
  L.off_att = o; o += 256;
  L.off_as = o; o += 256;
  L.off_bt = o; o += 256;
  L.off_e = o; o += (size_t)kEdgeCap * 4;
  L.off_eptr = o; o += 68 * 4;
  L.off_ent = o; o += (size_t)kEdgeCap * 2;
  L.off_bar = o; o += 16;
  L.total = o;                 // the dynamic window is declared 1024-byte aligned: no slack (7 GATv2 CTAs per SM need <= 32.1 KB each)
  return L;
}

// Prefetch groups of the pipeline (plain cp.async + a few scalar loads, all waited for at the top of the next item):
//   group A: the first block's target rows, the per-row logit scalars -- free to refill once the item's last logits are done
//   group B: source rows (MMA operand + logit operand), the first block's edge entries, per-target offsets -- free once
//            the item's last MMA has completed
template <bool TR, int LDZ>
__global__ void __launch_bounds__(kThreads, TR ? 4 : kCtasPerSm) conv2_attn_kernel(const Conv2Args a, const Conv2Layout L) {
  extern __shared__ __align__(1024) unsigned char sm_raw[];
  if (smem_u32(sm_raw) & 1023u) __trap();                   // SWIZZLE_128B operands need the 1024-byte alignment declared above
  unsigned char* sm = sm_raw;
  unsigned char* sX = sm;                                   // values [source k][channel], MN-major SW128 (GATv2: also logit operand)
  unsigned char* sW = sm + L.off_W;                         // weights [target of the block][source k], K-major SW128
  unsigned char* sT = sm + L.off_T;                         // targets of the block (x_r / q): [kTB][kRowPad]
  unsigned char* sK = sm + L.off_K;                         // Transformer keys: [k][kRowPad]
  __half* att_s = reinterpret_cast<__half*>(sm + L.off_att);
  float* s_as = reinterpret_cast<float*>(sm + L.off_as);    // [k]  <att, x_l[source k]> * 0.6 log2e
  float* s_bt = reinterpret_cast<float*>(sm + L.off_bt);    // [tk] <att, x_r[target]>  * 0.6 log2e
  float* s_e = reinterpret_cast<float*>(sm + L.off_e);      // [entry of the block] logit -> 2^(e - max)
  int* s_eptr = reinterpret_cast<int*>(sm + L.off_eptr);    // [cnt + 1] entry offsets per target (relative to the graph's block)
  uint16_t* s_ent = reinterpret_cast<uint16_t*>(sm + L.off_ent);   // entries of the block
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm + L.off_bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

  const int H = a.H, HC = H * kC;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int h = blockIdx.x % H;                             // gridDim.x is a multiple of H: the head is fixed per CTA
  const int gstep = gridDim.x / H;
  constexpr float kLog2e = 1.4426950408889634f;
  const float k06 = 0.6f * kLog2e;
  const float tr_scale = kLog2e / sqrtf((float)kC);
  const int ldz = LDZ > 0 ? LDZ : a.ldz;

  // stale value rows only ever meet zero weights, so they just have to stay finite: zero once
  for (int u = tid; u < kXBytes / 16; u += kThreads) reinterpret_cast<uint4*>(sX)[u] = make_uint4(0, 0, 0, 0);
  if (!TR) att_s[tid] = __float2half_rn(a.att[h * kC + tid] * (0.4f * kLog2e));
  const float bias_c = a.bias ? a.bias[h * kC + tid] : 0.f;  // this thread's output channel in the epilogue
  if (tid == 0) { mbar_init(smem_u32(bar), 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), kTCols);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  uint32_t parity = 0;

  auto load_meta = [&](int g, int4& m0, int2& m1) {
    if (g < a.n_graphs) {
      m0 = __ldg(reinterpret_cast<const int4*>(a.gmeta) + (size_t)g * 2);
      m1 = __ldg(reinterpret_cast<const int2*>(a.gmeta) + (size_t)g * 4 + 2);
    } else {
      m0 = make_int4(0, 0, 0, 0); m1 = make_int2(0, 0);
    }
  };
  // target rows [t0, t0 + n) of the graph whose first slot is `first` -> sT rows 0..n-1
  auto load_targets = [&](int first, int t0, int n) {
    for (int t = tid; t < n * 16; t += kThreads) {
      const int k = t >> 4, c = t & 15;
      cp16(sT + k * kRowPad + c * 16, a.Pt + (size_t)(first + t0 + k) * a.ldt + h * kC + c * 8);
    }
  };
  // edge entries [e0, e0 + n) of the graph's block at `ef` (e0 a multiple of 8 is not required: copied 2 bytes each when unaligned)
  auto load_entries = [&](int ef, int e0, int n) {
    if ((e0 & 7) == 0) {
      for (int t = tid; t * 8 < n; t += kThreads) cp16(reinterpret_cast<unsigned char*>(s_ent) + t * 16, a.eent + ef + e0 + t * 8);
    } else {
      for (int t = tid; t < n; t += kThreads) s_ent[t] = __ldg(a.eent + ef + e0 + t);
    }
  };
  // row of source k (compact index) in Ps / as
  auto src_row = [&](int first, int cnt, int nf, int k) { return k < cnt ? first + k : nf + k - cnt; };
  auto issue_A = [&](int first, int cnt, int nf, int nc) {
    load_targets(first, 0, cnt < kTB ? cnt : kTB);
    if (!TR) {
      if (tid < nc) cp4(s_as + tid, a.as + (size_t)src_row(first, cnt, nf, tid) * H + h);   // scaled by k06 where they are used
      if (tid < cnt) cp4(s_bt + tid, a.bt + (size_t)(first + tid) * H + h);
    }
  };
  auto issue_B = [&](int first, int cnt, int nf, int nc, int ef, int ne) {
#pragma unroll 2   // unrolled further, the GATv2 kernel spills more under its 72-register cap and runs slower
    for (int t = tid; t < nc * 16; t += kThreads) {
      const int k = t >> 4, c = t & 15;
      const __half* row = a.Ps + (size_t)src_row(first, cnt, nf, k) * a.lds + h * kC + c * 8;
      unsigned char* xd = sX + (c >> 3) * kPanel + k * 128 + (((c & 7) ^ (k & 7)) << 4);
      if (TR) {
        cp16(sK + k * kRowPad + c * 16, row);
        cp16(xd, row + HC);
      } else {
        cp16(xd, row);
      }
    }
    load_entries(ef, 0, ne < kEdgeCap ? ne : kEdgeCap);
    if (tid < cnt) cp4(s_eptr + tid, a.eabs + first + tid);      // absolute offsets: only differences are used below
    if (tid == 0) s_eptr[cnt] = ef + ne;
  };

  int g = blockIdx.x / H;
  int4 m0; int2 m1;
  load_meta(g, m0, m1);
  int4 n0; int2 n1;                                         // the item after: its meta is fetched a whole item before it is read
  load_meta(g + gstep, n0, n1);
  if (g < a.n_graphs) { issue_A(m0.x, m0.y, m0.z, m0.w); issue_B(m0.x, m0.y, m0.z, m0.w, m1.x, m1.y); }

  while (g < a.n_graphs) {
    const int first = m0.x, cnt = m0.y, nc = m0.w, ef = m1.x;
    // meta of the item after the next (two 16-byte loads, not read before the end of this item: no thread waits for them).
    // A graph without controlling nodes is an item with no blocks.
    const int gn = g + gstep;
    int4 p0; int2 p1;
    load_meta(gn + gstep, p0, p1);
    cp_wait_all();
    __syncthreads();
    if (cnt == 0 && gn < a.n_graphs) { issue_A(n0.x, n0.y, n0.z, n0.w); issue_B(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y); }
    for (int t0 = 0; t0 < cnt;) {
      // ---- block [t0, t1): at most kTB targets and kEdgeCap entries (a single target has at most kMaxList + 1 = 34)
      const int eb = s_eptr[t0];
      int t1;
      if (t0 == 0 && cnt <= kTB && s_eptr[cnt] - eb <= kEdgeCap) {
        t1 = cnt;                                                // the typical graph: one block (the scan below was 23 % of the kernel's instructions)
      } else {
        t1 = t0 + 1;
        while (t1 < cnt && t1 - t0 < kTB && s_eptr[t1 + 1] - eb <= kEdgeCap) ++t1;
      }
      const int nt = t1 - t0, E = s_eptr[t1] - eb;
      const bool last = t1 == cnt;
      const int nmma = nt <= 16 ? 16 : 32;
      if (t0 > 0) {                                            // later blocks (rare): their rows and entries, synchronously
        load_targets(first, t0, nt);
        load_entries(ef, eb - ef, E);
        cp_wait_all();
      }
      for (int u = tid; u < nmma * 8; u += kThreads) reinterpret_cast<uint4*>(sW)[u] = make_uint4(0, 0, 0, 0);
      if (t0 > 0) __syncthreads();
      // ---------------------------------------------------------------- logits: one lane per edge entry
      for (int e = tid; e < E; e += kThreads) {
        const uint32_t ent = s_ent[e];
        const int j = ent & 255u, tk = (int)(ent >> 8), tl = tk - t0;
        const unsigned char* tr = sT + tl * kRowPad;
        __half2 acc[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[q] = __float2half2_rn(0.f);
        if (!TR) {
          const unsigned char* xr = sX + j * 128;
          const int jx = j & 7;
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const uint4 xs = *reinterpret_cast<const uint4*>(xr + (c >> 3) * kPanel + (((c & 7) ^ jx) << 4));
            const uint4 xt = *reinterpret_cast<const uint4*>(tr + c * 16);
            const uint4 at = *reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(att_s) + c * 16);
            const __half2* x2 = reinterpret_cast<const __half2*>(&xs);
            const __half2* t2 = reinterpret_cast<const __half2*>(&xt);
            const __half2* a2 = reinterpret_cast<const __half2*>(&at);
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] = __hfma2(a2[q], __habs2(__hadd2(x2[q], t2[q])), acc[q]);
          }
        } else {
          const unsigned char* kr = sK + j * kRowPad;
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const uint4 xs = *reinterpret_cast<const uint4*>(kr + c * 16);
            const uint4 xt = *reinterpret_cast<const uint4*>(tr + c * 16);
            const __half2* x2 = reinterpret_cast<const __half2*>(&xs);
            const __half2* t2 = reinterpret_cast<const __half2*>(&xt);
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] = __hfma2(x2[q], t2[q], acc[q]);
          }
        }
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float2 f = __half22float2(acc[q]); s += f.x + f.y; }
        s_e[e] = TR ? s * tr_scale : fmaf(s_as[j] + s_bt[tk], k06, s);
      }
      __syncthreads();
      // the target rows and logit scalars are dead after the item's last block: refill them with the next item's
      // (overlaps softmax, MMA, epilogue)
      if (last && gn < a.n_graphs) issue_A(n0.x, n0.y, n0.z, n0.w);
      // ---------------------------------------------------------------- softmax -> W (4 lanes per target)
      {
        const int u = tid, tl = u >> 2, l = u & 3;             // kTB * 4 = kThreads: one pass
        int lo = 0, hi = 0;
        if (tl < nt) { lo = s_eptr[t0 + tl] - eb; hi = s_eptr[t0 + tl + 1] - eb; }
        float mx = -INFINITY;
        for (int x = lo + l; x < hi; x += 4) mx = fmaxf(mx, s_e[x]);
        __syncwarp();
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        float sum = 0.f;
        for (int x = lo + l; x < hi; x += 4) { const float pv = ex2f(s_e[x] - mx); s_e[x] = pv; sum += pv; }
        __syncwarp();
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        const float inv = rcpf(sum + 1e-16f);
        unsigned char* wrow = sW + tl * 128;
        for (int x = lo + l; x < hi; x += 4) {
          const int j = s_ent[x] & 255u;
          *reinterpret_cast<__half*>(wrow + ((((j >> 3) ^ tl) & 7) << 4) + (j & 7) * 2) = __float2half_rn(s_e[x] * inv);
        }
      }
      fence_proxy_async();
      __syncthreads();
      // ---------------------------------------------------------------- aggregate on the tensor core
      if (tid == 0) {
        tc_fence_after();
        // both operands fp16 (format 0), A (values) MN-major (bit 15), see attn_table.cu
        const uint32_t idesc = (make_idesc(128, nmma) & ~((7u << 7) | (7u << 10))) | (1u << 15);
        const uint64_t dv = desc_mn(smem_u32(sX), kPanel >> 4, 1024 >> 4);
        const uint64_t dw = make_smem_desc(smem_u32(sW));
        const int ksteps = (nc + 15) >> 4;
        for (int k = 0; k < ksteps; ++k) umma_bf16(tmem_base, dv + (uint64_t)(k * 128), dw + (uint64_t)(k * 2), idesc, k ? 1u : 0u);
        umma_commit(smem_u32(bar));
      }
      mbar_wait(smem_u32(bar), parity);
      parity ^= 1u;
      tc_fence_after();
      // the source rows, edge entries and offsets are dead after the item's last MMA: refill them (overlaps the epilogue)
      if (last && gn < a.n_graphs) issue_B(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y);
      // ---------------------------------------------------------------- epilogue: lane = channel, registers = targets
      {
        uint16_t* zc = reinterpret_cast<uint16_t*>(a.z) + (size_t)(first + t0) * ldz + a.z_col + h * kC + tid;
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16), v);
#pragma unroll
        for (int t8 = 0; t8 < 32; t8 += 8) {
          if (t8 < nt) {                                         // warp uniform: skip whole groups of 8 absent targets
#pragma unroll
            for (int t = t8; t < t8 + 8; ++t)
              if (t < nt) zc[t * ldz] = relu_bf16_bits(__uint_as_float(v[t]) + bias_c);
          }
        }
      }
      tc_fence_before();
      if (!last) __syncthreads();                              // the next block rewrites sT / s_ent / s_e / W
      t0 = t1;
    }
    g = gn; m0 = n0; m1 = n1; n0 = p0; n1 = p1;
  }
  cp_wait_all();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, kTCols);
}

template <bool TR>
int launch(const Conv2Args& a, int sm_count, cudaStream_t st) {
  const Conv2Layout L = conv2_layout(TR);
  static bool configured = false;
  if (!configured) {
    MLS_CUDA(cudaFuncSetAttribute(conv2_attn_kernel<TR, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    MLS_CUDA(cudaFuncSetAttribute(conv2_attn_kernel<TR, 0>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    MLS_CUDA(cudaFuncSetAttribute(conv2_attn_kernel<TR, 1152>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    MLS_CUDA(cudaFuncSetAttribute(conv2_attn_kernel<TR, 1152>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    configured = true;
  }
  const int per_sm = TR ? 4 : kCtasPerSm;
  long long items = (long long)a.n_graphs * a.H;
  long long grid = mls_cap_grid(sm_count * per_sm);         // graphs stride by gridDim.x / H: any multiple of H works
  grid -= grid % a.H;
  if (grid < a.H) grid = a.H;
  if (grid > items) grid = items;                           // items is a multiple of H
  if (grid <= 0) return MLS_OK;
  if (a.ldz == 1152) conv2_attn_kernel<TR, 1152><<<(unsigned)grid, kThreads, L.total, st>>>(a, L);   // immediate store offsets
  else conv2_attn_kernel<TR, 0><<<(unsigned)grid, kThreads, L.total, st>>>(a, L);
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}

}  // namespace

int conv2_attn_launch(const Conv2Args& a, int sm_count, cudaStream_t st) {
  if (!conv2_attn_supported(a.N, a.H)) {
    mls_set_error("conv2 attention: unsupported shape (N=%d, H=%d)", a.N, a.H);
    return MLS_ERR_UNSUPPORTED;
  }
  return a.transformer ? launch<true>(a, sm_count, st) : launch<false>(a, sm_count, st);
}

}  // namespace mls
