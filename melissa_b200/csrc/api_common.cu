// Error reporting + device probe for libmelissa_b200.
#include <stdarg.h>

#include "common.cuh"

#include <atomic>
static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};
void mls_count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
extern "C" unsigned long long mls_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

void mls_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" int mls_version(void) { return MLS_VERSION; }
extern "C" const char* mls_last_error(void) { return g_err; }

extern "C" int mls_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
  int dev = 0;
  MLS_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  MLS_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  return MLS_OK;
}

// ---- tuning options (process wide; A/B switches, defaults = fast paths).  Initial values come from the
// environment (MLS_ATTN_MMA, MLS_CONV2_MMA).
//   "attn_mma":  1 = in discrete-feature mode run conv1's attention through the pair-logit table and the tensor-core
//                aggregation kernel (attn_table.cu); 0 = gather kernel only
//   "conv2_mma": 1 = conv2 attention with half2 logits + tensor-core aggregation (conv2_attn.cu); 0 = gather kernel
//   "fp32_tc":   1 = precision fp32 runs its dense layers on the tensor cores through 3-way bf16 operand splits
//                (fp32-grade, dgn_forward.cu); 0 = SIMT sgemm
//   "max_ctas":  test only: n > 0 caps the grid of the persistent kernels (the tcgen05 GEMM and fused dueling heads, conv2
//                attention, the conv1 table kernels) at n CTAs, so that small inputs give every CTA many tiles; 0 = off
#include <stdlib.h>
#include <string.h>
static int g_attn_mma = -1, g_conv2_mma = -1, g_fp32_tc = -1, g_max_ctas = -1;
extern "C" int mls_get_option(const char* key) {
  if (key && !strcmp(key, "attn_mma")) {
    if (g_attn_mma < 0) { const char* e = getenv("MLS_ATTN_MMA"); g_attn_mma = e ? atoi(e) : 1; }
    return g_attn_mma;
  }
  if (key && !strcmp(key, "fp32_tc")) {
    if (g_fp32_tc < 0) { const char* e = getenv("MLS_FP32_TC"); g_fp32_tc = e ? atoi(e) : 1; }
    return g_fp32_tc;
  }
  if (key && !strcmp(key, "conv2_mma")) {
    if (g_conv2_mma < 0) { const char* e = getenv("MLS_CONV2_MMA"); g_conv2_mma = e ? atoi(e) : 1; }
    return g_conv2_mma;
  }
  if (key && !strcmp(key, "max_ctas")) {
    if (g_max_ctas < 0) { const char* e = getenv("MLS_MAX_CTAS"); g_max_ctas = e && atoi(e) > 0 ? atoi(e) : 0; }
    return g_max_ctas;
  }
  return -1;
}
int mls_cap_grid(int grid) {
  const int cap = mls_get_option("max_ctas");
  return cap > 0 && grid > cap ? cap : grid;
}
extern "C" int mls_set_option(const char* key, int value) {
  if (key && !strcmp(key, "conv2_mma")) { g_conv2_mma = value ? 1 : 0; return MLS_OK; }
  if (key && !strcmp(key, "fp32_tc")) { g_fp32_tc = value ? 1 : 0; return MLS_OK; }
  if (key && !strcmp(key, "attn_mma")) { g_attn_mma = value ? 1 : 0; return MLS_OK; }
  if (key && !strcmp(key, "max_ctas")) { g_max_ctas = value > 0 ? value : 0; return MLS_OK; }
  mls_set_error("unknown option %s", key ? key : "(null)");
  return MLS_ERR_INVALID;
}
