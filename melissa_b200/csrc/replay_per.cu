// Prioritized experience replay on the device (sm_100a): one fp64 sum tree per replay ring slot, built when a round is
// stored, sampled proportionally to priority, and refreshed after every update.
//
// Reference: tianshou 1.0 PrioritizedReplayBuffer (SegmentTree of float64 leaves p^alpha, sampling by prefix sum,
// update_weight with |td| + eps, max / min priority tracking) as the standard option of DQN-family training.
//
// Layout per slot: leaves are indexed by cell = episode * N + agent (B * N leaves), so a sampled leaf is the
// (episode, agent) pair directly.  Internal levels have fanout 32: node j of level k sums children 32j .. 32j+31 of
// level k-1, so one warp reads a node's children in one access.  Levels are stored leaves first, root last:
//   level 0 = leaves [L], level 1 [ceil(L/32)], ... , root [1];  slot s starts at trees + s * tree_size.
// Every sum is a fixed xor-butterfly warp reduction of the 32 children, so a node is a deterministic function of its
// children: the round build and the update's ancestor refresh give bit-identical nodes.
#include "common.cuh"

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxLevels = 16;                                 // 32^13 > 2^63 leaves
constexpr unsigned long long kMark = 0xFFF0000000000000ull;    // above the bits of every non-negative double

struct Levels {
  int n;                        // levels including the leaves (1 when L == 1: the leaf is the root)
  long long size[kMaxLevels];
  long long off[kMaxLevels];
  long long total;              // fp64 nodes per slot
};

Levels levels_of(long long L) {
  Levels lv{};
  long long s = L, off = 0;
  lv.n = 0;
  while (true) {
    lv.size[lv.n] = s;
    lv.off[lv.n] = off;
    off += s;
    ++lv.n;
    if (s == 1) break;
    s = (s + 31) / 32;
  }
  lv.total = off;
  return lv;
}

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(kFull, x, o);
  return x;
}

__device__ __forceinline__ double warp_incl_scan(double x, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double y = __shfl_up_sync(kFull, x, o);
    if (lane >= o) x += y;
  }
  return x;
}

__device__ __forceinline__ double prio_pow(double x, double alpha) { return alpha == 1.0 ? x : pow(x, alpha); }

// ---------------------------------------------------------------------------------------------- round build
// Block of 1024 threads = 1024 leaves -> 32 level-1 nodes -> 1 level-2 node.  Every leaf of the slot is written (acted:
// max_prio^alpha, else 0), so nothing of the slot's previous round survives.
__global__ void __launch_bounds__(1024) per_build_low_kernel(const uint8_t* __restrict__ flags, const double* __restrict__ max_prio,
                                                             double alpha, double* __restrict__ tree, Levels lv) {
  __shared__ double s_p, s_l1[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_p = prio_pow(*max_prio, alpha);
  __syncthreads();
  const long long i = (long long)blockIdx.x * 1024 + threadIdx.x;
  double x = 0.0;
  if (i < lv.size[0]) {
    x = (flags[i] & 1u) ? s_p : 0.0;
    tree[i] = x;
  }
  if (lv.n == 1) return;
  const double s = warp_sum(x);
  const long long j = i >> 5;
  if (lane == 0 && j < lv.size[1]) tree[lv.off[1] + j] = s;
  if (lv.n == 2) return;
  if (lane == 0) s_l1[warp] = s;                               // 0 for nodes past the level's end
  __syncthreads();
  if (warp == 0) {
    const double t = warp_sum(s_l1[lane]);
    if (lane == 0) tree[lv.off[2] + blockIdx.x] = t;           // gridDim.x == size[2]
  }
}

// Levels 3 .. root from level 2 (size L / 1024: 1600 nodes at B = 32768, N = 50), one block.
__global__ void __launch_bounds__(1024) per_build_high_kernel(double* __restrict__ tree, Levels lv) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = 3; k < lv.n; ++k) {
    for (long long node = warp; node < lv.size[k]; node += 32) {
      const long long c = node * 32 + lane;
      const double s = warp_sum(c < lv.size[k - 1] ? tree[lv.off[k - 1] + c] : 0.0);
      if (lane == 0) tree[lv.off[k] + node] = s;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------- sample
// One warp per sample.  The usable slots (first_slot + k) % R, k < n_slots, oldest first, are concatenated; with S_i the
// inclusive prefix sums of their leaves, T the total and v = u * T, the sample is the leaf
//   min{i : leaf_i > 0 and S_i >= v},  or the last positive leaf when there is none (v rounded past the last one).
// It is found hierarchically: the first slot whose root prefix reaches v, then per level the first positive child whose
// inclusive prefix reaches the remaining v.  A leaf of priority 0 is never returned; if the usable slots hold no
// positive leaf at all, the sample is (first_slot, cell 0) with leaf value 0.
__global__ void per_sample_kernel(const double* __restrict__ trees, int R, int N, int first_slot, int n_slots,
                                  const double* __restrict__ u, int M, int* __restrict__ rho, int* __restrict__ ep,
                                  int* __restrict__ agent, double* __restrict__ leaf_out, Levels lv) {
  const int lane = threadIdx.x & 31;
  const int m = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (m >= M) return;                                          // warp-uniform
  const long long root_off = lv.off[lv.n - 1];
  auto slot_of = [&](int k) { return (first_slot + k) % R; };

  double carry = 0.0;                                          // T, summed exactly as the selection pass sums it
  for (int c = 0; c < n_slots; c += 32) {
    const int k = c + lane;
    const double r = k < n_slots ? trees[(long long)slot_of(k) * lv.total + root_off] : 0.0;
    carry += __shfl_sync(kFull, warp_incl_scan(r, lane), 31);
  }
  double v = u[m] * carry;

  int sel = -1, last = -1;
  double sel_excl = 0.0, last_excl = 0.0;
  carry = 0.0;
  for (int c = 0; c < n_slots; c += 32) {
    const int k = c + lane;
    const double r = k < n_slots ? trees[(long long)slot_of(k) * lv.total + root_off] : 0.0;
    const double incl = warp_incl_scan(r, lane);
    const double pref = carry + incl;
    double prev = __shfl_up_sync(kFull, pref, 1);
    if (lane == 0) prev = carry;
    const unsigned pos = __ballot_sync(kFull, r > 0.0);
    const unsigned hit = __ballot_sync(kFull, r > 0.0 && pref >= v);
    if (hit) {
      const int j = __ffs(hit) - 1;
      sel = c + j;
      sel_excl = __shfl_sync(kFull, prev, j);
      break;
    }
    if (pos) {
      const int j = 31 - __clz(pos);
      last = c + j;
      last_excl = __shfl_sync(kFull, prev, j);
    }
    carry += __shfl_sync(kFull, incl, 31);
  }
  if (sel < 0) { sel = last; sel_excl = last_excl; }
  if (sel < 0) {                                               // no positive leaf in any usable slot
    if (lane == 0) {
      rho[m] = first_slot; ep[m] = 0; agent[m] = 0;
      if (leaf_out) leaf_out[m] = 0.0;
    }
    return;
  }
  const int slot = slot_of(sel);
  const double* tree = trees + (long long)slot * lv.total;
  v -= sel_excl;
  long long node = 0;
  double val = tree[root_off];
  for (int k = lv.n - 1; k >= 1; --k) {
    const long long c = node * 32 + lane;
    const double x = c < lv.size[k - 1] ? tree[lv.off[k - 1] + c] : 0.0;
    const double incl = warp_incl_scan(x, lane);
    double prev = __shfl_up_sync(kFull, incl, 1);
    if (lane == 0) prev = 0.0;
    const unsigned pos = __ballot_sync(kFull, x > 0.0);
    const unsigned hit = __ballot_sync(kFull, x > 0.0 && incl >= v);
    const int j = hit ? __ffs(hit) - 1 : (pos ? 31 - __clz(pos) : 0);
    v -= __shfl_sync(kFull, prev, j);
    val = __shfl_sync(kFull, x, j);
    node = node * 32 + j;
  }
  if (lane == 0) {
    rho[m] = slot;
    ep[m] = (int)(node / N);
    agent[m] = (int)(node % N);
    if (leaf_out) leaf_out[m] = val;
  }
}

// ---------------------------------------------------------------------------------------------- update
// Pass 1: every sample m marks its leaf with kMark | m by a 64-bit atomicMax on the leaf's bits, so the leaf ends up
// holding the mark of its LAST occurrence (numpy fancy assignment: the last write wins).  max_prio / min_prio take the
// raw |td| + eps (bits of non-negative doubles order like the doubles).  Entries out of the ring are ignored.
__device__ __forceinline__ bool valid_sample(int r, int e, int a, int R, long long B, int N) {
  return r >= 0 && r < R && e >= 0 && e < B && a >= 0 && a < N;
}

__global__ void per_mark_kernel(double* __restrict__ trees, long long tree_size, int R, long long B, int N, const int* __restrict__ rho,
                                const int* __restrict__ ep, const int* __restrict__ agent, const float* __restrict__ td, int M,
                                double eps, double* __restrict__ max_prio, double* __restrict__ min_prio) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = m < M && valid_sample(rho[m], ep[m], agent[m], R, B, N);
  double hi = 0.0, lo = __longlong_as_double(0x7FF0000000000000ll);   // +inf
  if (ok) {
    const long long leaf = (long long)rho[m] * tree_size + (long long)ep[m] * N + agent[m];
    atomicMax(reinterpret_cast<unsigned long long*>(trees + leaf), kMark | (unsigned long long)m);
    hi = lo = fabs((double)td[m]) + eps;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    hi = fmax(hi, __shfl_xor_sync(kFull, hi, o));
    lo = fmin(lo, __shfl_xor_sync(kFull, lo, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(reinterpret_cast<unsigned long long*>(max_prio), (unsigned long long)__double_as_longlong(hi));
    atomicMin(reinterpret_cast<unsigned long long*>(min_prio), (unsigned long long)__double_as_longlong(lo));
  }
}

// Pass 2: the sample whose mark survived writes (|td| + eps)^alpha.
__global__ void per_write_kernel(double* __restrict__ trees, long long tree_size, int R, long long B, int N, const int* __restrict__ rho,
                                 const int* __restrict__ ep, const int* __restrict__ agent, const float* __restrict__ td, int M,
                                 double alpha, double eps) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M || !valid_sample(rho[m], ep[m], agent[m], R, B, N)) return;
  double* leaf = trees + (long long)rho[m] * tree_size + (long long)ep[m] * N + agent[m];
  if ((unsigned long long)__double_as_longlong(*leaf) == (kMark | (unsigned long long)m))
    *leaf = prio_pow(fabs((double)td[m]) + eps, alpha);
}

// Pass 3, one launch per level k >= 1: one warp per sample recomputes the level-k ancestor of its leaf from its 32
// children (final after the previous launch).  Samples sharing an ancestor write the same value.
__global__ void per_refresh_kernel(double* __restrict__ trees, int R, long long B, int N, const int* __restrict__ rho,
                                   const int* __restrict__ ep, const int* __restrict__ agent, int M, int k, Levels lv) {
  const int lane = threadIdx.x & 31;
  const int m = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (m >= M) return;                                          // warp-uniform
  const int r = rho[m], e = ep[m], a = agent[m];
  if (!valid_sample(r, e, a, R, B, N)) return;                 // warp-uniform
  double* tree = trees + (long long)r * lv.total;
  const long long node = ((long long)e * N + a) >> (5 * k);
  const long long c = node * 32 + lane;
  const double s = warp_sum(c < lv.size[k - 1] ? tree[lv.off[k - 1] + c] : 0.0);
  if (lane == 0) tree[lv.off[k] + node] = s;
}

}  // namespace

extern "C" int64_t mls_per_tree_size(int64_t n_cells) {
  if (n_cells < 1) return -1;
  return levels_of(n_cells).total;
}

extern "C" int mls_per_build(const uint8_t* flags, int64_t n_episodes, int32_t n_nodes, const double* max_prio, double alpha,
                             double* tree, void* stream) {
  MLS_CHECK_ARG(flags && max_prio && tree, "NULL argument");
  MLS_CHECK_ARG(n_episodes > 0 && n_nodes > 0, "n_episodes and n_nodes must be positive");
  MLS_CHECK_ARG(alpha > 0.0, "alpha must be > 0");
  const Levels lv = levels_of(n_episodes * n_nodes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  per_build_low_kernel<<<(unsigned)((lv.size[0] + 1023) / 1024), 1024, 0, st>>>(flags, max_prio, alpha, tree, lv);
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  if (lv.n > 3) {
    per_build_high_kernel<<<1, 1024, 0, st>>>(tree, lv);
    mls_count_launch();
    MLS_LAUNCH_CHECK();
  }
  return MLS_OK;
}

extern "C" int mls_per_sample(const double* trees, int32_t ring_rounds, int64_t n_episodes, int32_t n_nodes, int32_t first_slot,
                              int32_t n_slots, const double* u, int32_t n_samples, int32_t* round_index, int32_t* episode,
                              int32_t* agent, double* leaf, void* stream) {
  MLS_CHECK_ARG(trees && u && round_index && episode && agent, "NULL argument");
  MLS_CHECK_ARG(ring_rounds > 0 && n_episodes > 0 && n_nodes > 0, "ring_rounds, n_episodes and n_nodes must be positive");
  MLS_CHECK_ARG(first_slot >= 0 && first_slot < ring_rounds && n_slots >= 1 && n_slots <= ring_rounds,
                "usable slots must be 1..ring_rounds slots starting inside the ring");
  if (n_samples <= 0) return MLS_OK;
  const Levels lv = levels_of(n_episodes * n_nodes);
  const long long threads = (long long)n_samples * 32;
  per_sample_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      trees, ring_rounds, n_nodes, first_slot, n_slots, u, n_samples, round_index, episode, agent, leaf, lv);
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}

extern "C" int mls_per_update(double* trees, int32_t ring_rounds, int64_t n_episodes, int32_t n_nodes, const int32_t* round_index,
                              const int32_t* episode, const int32_t* agent, const float* td, int32_t n_samples, double alpha,
                              double eps, double* max_prio, double* min_prio, void* stream) {
  MLS_CHECK_ARG(trees && round_index && episode && agent && td && max_prio && min_prio, "NULL argument");
  MLS_CHECK_ARG(ring_rounds > 0 && n_episodes > 0 && n_nodes > 0, "ring_rounds, n_episodes and n_nodes must be positive");
  MLS_CHECK_ARG(alpha > 0.0 && eps >= 0.0, "alpha must be > 0 and eps >= 0");
  if (n_samples <= 0) return MLS_OK;
  const Levels lv = levels_of(n_episodes * n_nodes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned blocks = (unsigned)((n_samples + 255) / 256);
  per_mark_kernel<<<blocks, 256, 0, st>>>(trees, lv.total, ring_rounds, n_episodes, n_nodes, round_index, episode, agent, td,
                                          n_samples, eps, max_prio, min_prio);
  per_write_kernel<<<blocks, 256, 0, st>>>(trees, lv.total, ring_rounds, n_episodes, n_nodes, round_index, episode, agent, td,
                                           n_samples, alpha, eps);
  const unsigned warp_blocks = (unsigned)(((long long)n_samples * 32 + 255) / 256);
  for (int k = 1; k < lv.n; ++k)
    per_refresh_kernel<<<warp_blocks, 256, 0, st>>>(trees, ring_rounds, n_episodes, n_nodes, round_index, episode, agent,
                                                    n_samples, k, lv);
  mls_count_launch(2 + (lv.n - 1));
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}
