// Persistent warp-specialised bf16 GEMM on the 5th-gen tensor cores (sm_100a):
//     C[M, N] (bf16) = act( rowscale[m] * (A[M, K] @ B[N, K]^T) + bias[n] )
// A and B are K-major bf16 in global memory, moved by TMA (128B swizzle) into a 3/4-stage
// shared-memory ring; one thread issues tcgen05.mma (M=128, N=BN, K=16) into a double
// buffered fp32 accumulator in TMEM; four epilogue warps drain TMEM with tcgen05.ld, apply
// the fused epilogue and store bf16 rows.  One CTA per SM, static round-robin tile order
// with the N tiles of one M tile adjacent (A tile stays hot in L2).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "dgn_kernels.cuh"

namespace mls {

constexpr int kBM = 128, kBK = 64, kUmmaK = 16;
constexpr int kGemmEpiWarps = 16;       // 4 per TMEM lane quarter, each drains a quarter of the tile's columns
constexpr int kGemmThreads = 128 + kGemmEpiWarps * 32;      // 4 control warps (TMA, MMA, TMEM alloc, spare) + the epilogue warps

struct GemmEpilogue {
  __nv_bfloat16* C;      // [M, ldc]
  int ldc;
  const float* bias;     // [N] or NULL
  const float* obs;      // row scale = obs[(m / nodes) * obs_stride + (m % nodes) * 8 + 7], or NULL
  long long obs_stride;
  int nodes;
  int relu;
  // optional: dots[m][n / 128] = sum over the 128-column group of dotvec[n] * (value before bf16 rounding / ReLU).
  // Used for the per-node linear part of the GATv2 logits (<att_h, x_l[j,h,:]>, <att_h, x_r[i,h,:]>).
  const float* dotvec;   // [N] or NULL
  float* dots;           // [M, N / 128]
  // optional: output row m is node row row_index[m] for the row scale (compacted row sets)
  const int* row_index;
  // optional second dot vector (dots2 laid out like dots); dot_relu: the dots use max(value, 0).
  // C may be NULL when only the dots are wanted (last hidden layer of the dueling heads: the output
  // layer is three dot products per row, the hidden activations themselves are never needed).
  const float* dotvec2;
  float* dots2;
  int dot_relu;
  // C is written as IEEE fp16 (saturated to +-65504) instead of bf16: 11 significant bits for operands that feed
  // packed-half math (conv2 attention)
  int c_fp16;
  // optional fp32 output (beside or instead of C): Cf[m][n] = the epilogue value before narrowing.  Used by the
  // fp32-grade route, whose operands are 3-way bf16 splits concatenated along K (dgn_forward.cu).
  float* Cf;
  int ldcf;
  // target segment of a split launch (GemmShape::t_lo): C, dots and row_index above serve the source columns; the target
  // columns [t_lo, t_hi) go to Ct[m][n - t_lo] (row stride ldct), dots_t[m][(n - t_lo) / 128] and the row scale goes
  // through row_index_t.  bias and dotvec are indexed by the packed column n in both segments.
  __nv_bfloat16* Ct;
  int ldct;
  float* dots_t;
  const int* row_index_t;
  // split-K (GemmShape::k_split > 1): partial product s goes to Cf + s * cf_split_stride
  long long cf_split_stride;
};

struct GemmShape {
  int M, N, K;
  const int* m_dev;      // optional device-side row count (clamped to M)
  // optional second A matrix for the K range [k2_lo, k2_hi) (multiples of 64): those columns of the logical A come from
  // A2[m][k - k2_lo] (row stride lda2) instead of A[m][k] -- the dueling heads read their latent row from two matrices
  // (snapshot columns of relu(conv1) live in x1, the rest in z)
  const __nv_bfloat16* A2;
  int lda2, k2_lo, k2_hi;
  // optional split of the N columns (t_lo < t_hi, multiples of 256 or, without dots, of 128): the conv2 projections of
  // the source rows (columns outside [t_lo, t_hi)) and of the target rows (inside) in one launch over the packed weight
  // rows.  Target columns are computed for rows [0, min(M, *m_dev_t)) only, source columns for rows [0, min(M, *m_dev)),
  // and the second A matrix, if given, applies to the target columns only.
  const int* m_dev_t;
  int t_lo, t_hi;
  // optional split of K into k_split ranges of whole 64-wide blocks (0 / 1: none; fp32 output Cf only, no bias): every
  // (tile, range) pair is a work item and writes its partial product to its own Cf slice; the caller adds the slices up.
  // Gives weight-gradient products (M, N of a few tiles, K = the batch's rows) enough work items to fill the GPU.
  int k_split;
};

size_t gemm_smem_bytes(int BN);
// K-major bf16 matrix [rows, cols] with row stride ld_elems -> TMA descriptor with a 64 x box_rows box, 128B swizzle
int make_tmap_bf16(CUtensorMap* tm, const void* base, int rows, int cols, int ld_elems, int box_rows);
// host: build the two TMA descriptors + launch.  A: [M, K] row stride lda; B: [N, K] row stride ldb.
int gemm_bf16_launch(const __nv_bfloat16* A, int lda, const __nv_bfloat16* B, int ldb, GemmShape shape,
                     GemmEpilogue epi, int sm_count, cudaStream_t st);

// Dueling heads with 128-wide hidden layers in one persistent kernel: per row m < min(M, *m_dev),
//     hid = relu(A[m] @ W_h0^T + b_h0) (bf16),  h2 = relu(hid @ W_h1^T + b_h1),
//     head_final_row(m, <h2[0:128], hv1[0:128]>, <h2[128:256], hv1[128:256]>, <h2[0:128], hv2[0:128]>)
// with the rounding points and accumulation orders of the two-GEMM chain (MODE 2, then MODE 3).  shape: N = 256, K = latent,
// optional A2 K range.  W_h0 [256][K], W_h1 [256][256] (block diagonal [Q1 0; 0 V1]).
struct HeadVecs {
  const float *b_h0, *b_h1, *hv1, *hv2;     // [256] each
};
int head_dueling_launch(const __nv_bfloat16* A, int lda, GemmShape shape, const __nv_bfloat16* w_h0, const __nv_bfloat16* w_h1,
                        const HeadVecs& vec, const HeadOut& out, int sm_count, cudaStream_t st);

}  // namespace mls
