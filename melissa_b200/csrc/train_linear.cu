// bf16 training precision of the dense layers (DGNBase.set_train_precision("bf16")): forward and backward of
// y = x W^T + b as three products on the tcgen05 GEMM (gemm_tcgen05.cu, MODE 0 with the fp32 output Cf):
//     y  = fp32acc(bf16(x)  . bf16(W)^T) + b          A = x   [rows][in]  K-major,   B = W   [out][in]
//     dx = fp32acc(bf16(dy) . bf16(W))                A = dy  [rows][out] K-major,   B = W^T [in][out]
//     dW = fp32acc(bf16(dy)^T . bf16(x))              A = dy^T [out][rows],          B = x^T [in][rows], split along the rows
//     db = sum over rows of dy, fp32, from the unrounded dy
// This file holds the operand preparation: fp32 -> bf16 packs with K zero-padded to the GEMM's 64 and N (the B rows)
// zero-padded to 128, transposed packs for the two operands of dW (with the column sums of dy for db fused into the
// pass over dy), and the copy of a padded fp32 result into the caller's matrix.  No atomics: db is per-block partials
// summed in a fixed order, so the backward is bitwise reproducible.
#include <cuda_bf16.h>

#include "gemm_tcgen05.cuh"

namespace {

constexpr int kT = 64;                 // transpose tile (rows x columns)
constexpr int kPackThreads = 256;

inline long long pad_to(long long v, long long m) { return (v + m - 1) / m * m; }
inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// dst[r][k] = bf16(src[r][k]) for r < rows, k < cols; 0 elsewhere in [rows_out][kp] (kp a multiple of 8)
__global__ void __launch_bounds__(kPackThreads) pack_bf16_kernel(const float* __restrict__ src, long long ld, int rows, int cols,
                                                                 __nv_bfloat16* __restrict__ dst, int rows_out, int kp) {
  const int per_row = kp / 8;
  const long long n = (long long)rows_out * per_row;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / per_row), k0 = (int)(i % per_row) * 8;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = (r < rows && k0 + j < cols) ? __ldg(src + (long long)r * ld + k0 + j) : 0.f;
    uint4 o;
    uint32_t* w = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat162 p = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      w[j] = *reinterpret_cast<uint32_t*>(&p);
    }
    *reinterpret_cast<uint4*>(dst + (long long)r * kp + k0) = o;
  }
}

// dst[c][r] = bf16(src[r][c]) over a grid of 64 x 64 tiles: dst is [gridDim.y * 64][ldd] with ldd = gridDim.x * 64, and every
// element outside rows x cols is 0.  colsum_part (NULL: none) [gridDim.x][cols] receives the fp32 column sums of this block's
// 64 rows of src, added in row order.
__global__ void __launch_bounds__(kPackThreads) transpose_pack_bf16_kernel(const float* __restrict__ src, long long ld, int rows, int cols,
                                                                           __nv_bfloat16* __restrict__ dst, float* __restrict__ colsum_part) {
  __shared__ float t[kT][kT + 1];
  const int r0 = blockIdx.x * kT, c0 = blockIdx.y * kT;
  const long long ldd = (long long)gridDim.x * kT;
  for (int i = threadIdx.x; i < kT * kT; i += kPackThreads) {
    const int rr = i / kT, cc = i % kT;
    const int r = r0 + rr, c = c0 + cc;
    t[rr][cc] = (r < rows && c < cols) ? __ldg(src + (long long)r * ld + c) : 0.f;
  }
  __syncthreads();
  if (colsum_part && threadIdx.x < kT && c0 + threadIdx.x < cols) {
    float s = 0.f;
    for (int rr = 0; rr < kT; ++rr) s += t[rr][threadIdx.x];
    colsum_part[(long long)blockIdx.x * cols + c0 + threadIdx.x] = s;
  }
  for (int i = threadIdx.x; i < kT * kT / 2; i += kPackThreads) {
    const int cc = i / (kT / 2), rr = (i % (kT / 2)) * 2;
    const __nv_bfloat162 p = __floats2bfloat162_rn(t[rr][cc], t[rr + 1][cc]);
    *reinterpret_cast<__nv_bfloat162*>(dst + (long long)(c0 + cc) * ldd + r0 + rr) = p;
  }
}

// out[c] = sum over b < n_part of part[b][c], in order b = 0, 1, ...
__global__ void colsum_reduce_kernel(const float* __restrict__ part, int n_part, int cols, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float s = 0.f;
  for (int b = 0; b < n_part; ++b) s += part[(long long)b * cols + c];
  out[c] = s;
}

// dst[r][c] = sum over s < n_split of part[s][r][c] (part: [n_split][rows][ldp]), added in order s = 0, 1, ...
__global__ void split_sum_kernel(const float* __restrict__ part, int n_split, int rows, int cols, int ldp, float* __restrict__ dst) {
  const long long n = (long long)rows * cols, slice = (long long)rows * ldp;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    const float* p = part + (long long)r * ldp + c;
    float s = 0.f;
    for (int k = 0; k < n_split; ++k) s += p[k * slice];
    dst[i] = s;
  }
}

// dst[r][c] = src[r][c] for r < rows, c < cols (src row stride lds, dst row stride ldd)
__global__ void copy_cols_kernel(const float* __restrict__ src, long long lds, int rows, int cols, float* __restrict__ dst, long long ldd) {
  const long long n = (long long)rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    dst[(long long)r * ldd + c] = src[(long long)r * lds + c];
  }
}

// K ranges of the dW product (K = the rows, M x N = out x in: a few tiles): about two work items per SM of a B200, at least
// eight 64-wide K blocks per range so that the TMA ring fills
int dw_splits(int out, int nin, int rp) {
  const int tiles = ((out + 127) / 128) * (nin / (nin % 256 == 0 ? 256 : 128));
  const int s = (2 * 148 + tiles - 1) / tiles, by_k = rp / kT / 8;
  return s < by_k ? s : (by_k > 1 ? by_k : 1);
}

int grid_for(long long work) {
  const long long g = (work + kPackThreads - 1) / kPackThreads;
  return (int)(g < 148 * 16 ? (g > 0 ? g : 1) : 148 * 16);
}

// Scratch of one layer (rows, in, out): every piece starts on a 256-byte boundary.  The forward and the backward use
// separate pieces, so one workspace serves both.
struct Layout {
  int kin, nout, kout, nin, rp, rt, oc;     // K / N paddings; rp = rows padded to 64, rt = rp / 64 row tiles, oc = out padded to 64
  int ks;                                   // K ranges of dW
  size_t xb, wb, bpad, yf;                  // forward: bf16(x) [rows][kin], bf16(W) [nout][kin], bias [nout], y [rows][nout]
  size_t dyb, wtb, dxf;                     // dx: bf16(dy) [rows][kout], bf16(W^T) [nin][kout], dx [rows][nin]
  size_t dyt, xt, dwf, part;                // dW: bf16(dy^T) [oc][rp], bf16(x^T) [nin][rp], dW per K range [ks][out][nin], db partials [rt][out]
  size_t total;
  Layout(long long rows, int in, int out) {
    kin = (int)pad_to(in, mls::kBK); nout = (int)pad_to(out, 128); kout = (int)pad_to(out, mls::kBK); nin = (int)pad_to(in, 128);
    rp = (int)pad_to(rows, kT); rt = rp / kT; oc = (int)pad_to(out, kT);
    ks = dw_splits(out, nin, rp);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = align256(o + bytes); return at; };
    xb = take((size_t)rows * kin * 2); wb = take((size_t)nout * kin * 2); bpad = take((size_t)nout * 4); yf = take((size_t)rows * nout * 4);
    dyb = take((size_t)rows * kout * 2); wtb = take((size_t)nin * kout * 2); dxf = take((size_t)rows * nin * 4);
    dyt = take((size_t)oc * rp * 2); xt = take((size_t)nin * rp * 2); dwf = take((size_t)ks * out * nin * 4); part = take((size_t)rt * out * 4);
    total = o;
  }
};

int sm_count() {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  return sms;
}

// dst[M][n] (row stride ldd) = A[M][K] . B[n_pad][K]^T (+ bias[n_pad]): straight into dst when its rows are whole 128-column
// tiles and 16-byte aligned, else into the padded scratch [M][n_pad] and copied
int gemm_into(const __nv_bfloat16* A, int lda, const __nv_bfloat16* B, int M, int n, int n_pad, int K, const float* bias, float* dst,
              long long ldd, float* scratch, int sms, cudaStream_t st) {
  const bool direct = n == n_pad && ldd % 4 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0 && ldd < (1ll << 31);
  mls::GemmShape shape{M, n_pad, K, nullptr};
  mls::GemmEpilogue epi{};
  epi.bias = bias;
  epi.Cf = direct ? dst : scratch;
  epi.ldcf = direct ? (int)ldd : n_pad;
  int rc = mls::gemm_bf16_launch(A, lda, B, K, shape, epi, sms, st);
  if (rc || direct) return rc;
  copy_cols_kernel<<<grid_for((long long)M * n), kPackThreads, 0, st>>>(scratch, n_pad, M, n, dst, ldd);
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}

int check_shape(long long rows, int in, int out, const void* ws, size_t ws_bytes) {
  MLS_CHECK_ARG(rows >= 0 && rows < (1ll << 31) - kT && in >= 1 && out >= 1, "linear: bad shape (rows %lld, in %d, out %d)", rows, in, out);
  MLS_CHECK_ARG(rows == 0 || (ws && ws_bytes >= Layout(rows, in, out).total && (reinterpret_cast<uintptr_t>(ws) & 255) == 0),
                "linear: workspace must hold mls_linear_bf16_workspace_bytes() bytes on a 256-byte boundary");
  return MLS_OK;
}

}  // namespace

extern "C" size_t mls_linear_bf16_workspace_bytes(int64_t rows, int32_t in, int32_t out) {
  if (rows <= 0 || in < 1 || out < 1) return 0;
  return Layout(rows, in, out).total;
}

extern "C" int mls_linear_bf16_fwd(const float* x, int64_t ldx, const float* w, const float* b, int64_t rows, int32_t in, int32_t out,
                                   float* y, int64_t ldy, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = check_shape(rows, in, out, workspace, workspace_bytes)) return rc;
  if (rows == 0) return MLS_OK;
  MLS_CHECK_ARG(x && w && y && ldx >= in && ldy >= out, "linear forward: NULL argument or row stride below the width");
  const Layout L(rows, in, out);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  auto* xb = reinterpret_cast<__nv_bfloat16*>(ws + L.xb);
  auto* wb = reinterpret_cast<__nv_bfloat16*>(ws + L.wb);
  const cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int sms = sm_count();
  MLS_CHECK_ARG(sms > 0, "linear forward: no CUDA device");
  pack_bf16_kernel<<<grid_for(rows * (L.kin / 8)), kPackThreads, 0, st>>>(x, ldx, (int)rows, in, xb, (int)rows, L.kin);
  pack_bf16_kernel<<<grid_for((long long)L.nout * (L.kin / 8)), kPackThreads, 0, st>>>(w, in, out, in, wb, L.nout, L.kin);
  mls_count_launch(2);
  MLS_LAUNCH_CHECK();
  const float* bias = b;
  if (b && L.nout != out) {                                 // the epilogue reads one bias value per padded column
    float* bp = reinterpret_cast<float*>(ws + L.bpad);
    MLS_CUDA(cudaMemsetAsync(bp, 0, (size_t)L.nout * 4, st));
    MLS_CUDA(cudaMemcpyAsync(bp, b, (size_t)out * 4, cudaMemcpyDeviceToDevice, st));
    bias = bp;
  }
  return gemm_into(xb, L.kin, wb, (int)rows, out, L.nout, L.kin, bias, y, ldy, reinterpret_cast<float*>(ws + L.yf), sms, st);
}

extern "C" int mls_linear_bf16_bwd(const float* x, int64_t ldx, const float* w, const float* dy, int64_t lddy, int64_t rows, int32_t in,
                                   int32_t out, float* dx, int64_t lddx, float* dw, float* db, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  if (int rc = check_shape(rows, in, out, workspace, workspace_bytes)) return rc;
  MLS_CHECK_ARG(dw && (rows == 0 || (x && w && dy && ldx >= in && lddy >= out && (!dx || lddx >= in))),
                "linear backward: NULL argument or row stride below the width");
  const cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (rows == 0) {                                          // an empty batch contributes nothing
    MLS_CUDA(cudaMemsetAsync(dw, 0, (size_t)out * in * 4, st));
    if (db) MLS_CUDA(cudaMemsetAsync(db, 0, (size_t)out * 4, st));
    return MLS_OK;
  }
  const Layout L(rows, in, out);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  const int sms = sm_count();
  MLS_CHECK_ARG(sms > 0, "linear backward: no CUDA device");
  float* part = reinterpret_cast<float*>(ws + L.part);
  auto* dyt = reinterpret_cast<__nv_bfloat16*>(ws + L.dyt);
  auto* xt = reinterpret_cast<__nv_bfloat16*>(ws + L.xt);
  // dW = dy^T . x: both operands K-major along the rows, the column sums of dy (db) from the same pass
  transpose_pack_bf16_kernel<<<dim3(L.rt, L.oc / kT), kPackThreads, 0, st>>>(dy, lddy, (int)rows, out, dyt, db ? part : nullptr);
  transpose_pack_bf16_kernel<<<dim3(L.rt, L.nin / kT), kPackThreads, 0, st>>>(x, ldx, (int)rows, in, xt, nullptr);
  mls_count_launch(2);
  MLS_LAUNCH_CHECK();
  if (db) {
    colsum_reduce_kernel<<<(out + 127) / 128, 128, 0, st>>>(part, L.rt, out, db);
    mls_count_launch();
    MLS_LAUNCH_CHECK();
  }
  {
    float* dwf = reinterpret_cast<float*>(ws + L.dwf);
    mls::GemmShape shape{out, L.nin, L.rp, nullptr};
    shape.k_split = L.ks;
    mls::GemmEpilogue epi{};
    epi.Cf = dwf;
    epi.ldcf = L.nin;
    epi.cf_split_stride = (long long)out * L.nin;
    if (int rc = mls::gemm_bf16_launch(dyt, L.rp, xt, L.rp, shape, epi, sms, st)) return rc;
    split_sum_kernel<<<grid_for((long long)out * in), kPackThreads, 0, st>>>(dwf, L.ks, out, in, L.nin, dw);
    mls_count_launch();
    MLS_LAUNCH_CHECK();
  }
  if (!dx) return MLS_OK;
  // dx = dy . W: dy K-major along out, W^T [in][out] K-major along out
  auto* dyb = reinterpret_cast<__nv_bfloat16*>(ws + L.dyb);
  auto* wtb = reinterpret_cast<__nv_bfloat16*>(ws + L.wtb);
  pack_bf16_kernel<<<grid_for(rows * (L.kout / 8)), kPackThreads, 0, st>>>(dy, lddy, (int)rows, out, dyb, (int)rows, L.kout);
  // W^T through the transpose pack: [nin][kout] with kout = out padded to 64, i.e. W's rows padded to 64
  transpose_pack_bf16_kernel<<<dim3(L.kout / kT, L.nin / kT), kPackThreads, 0, st>>>(w, in, out, in, wtb, nullptr);
  mls_count_launch(2);
  MLS_LAUNCH_CHECK();
  return gemm_into(dyb, L.kout, wtb, (int)rows, in, L.nin, L.kout, nullptr, dx, lddx, reinterpret_cast<float*>(ws + L.dxf), sms, st);
}
