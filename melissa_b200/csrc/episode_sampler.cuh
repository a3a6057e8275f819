// Device episode sampler: the reset tuple (graph, source, interested set, scripted set) of episode number `ep_no` of
// global episode slot `slot`, drawn from a counter-based Philox stream.  The round kernel (in-kernel restarts,
// env_round.cu) and the materialising kernel (mls_episode_sample) both draw through the functions below, so the
// tuples an environment plays and the tuples a caller materialises cannot diverge.
//
// Distribution (training-mode reset, reference core.py:371-395): graph uniform over [0, pool_size), source uniform
// over [0, N), k = int((0.1 + (1.0 - 0.1) * u) * N) with u a 53-bit uniform (numpy's uniform(0.1, 1.0) and the same
// fp64 expression), interested = a uniform k-subset of the nodes independent of the source, scripted = an independent
// uniform n_scripted-subset with the source removed when ratio < 1.
//
// Subsets: every node gets a 64-bit key per subset; the subset is the nodes of the k smallest keys (ties by index).
// The keys are i.i.d. uniform, so their order is an exchangeable random permutation of the nodes and its first k
// entries are a uniform k-subset; the index tie-break is the only departure, and two of N <= 256 keys tie with
// probability below N^2 / 2^65 < 2e-15.
//
// Counter domain: Philox4x32-10 counter words (c0, c1, c2, c3) = (slot, ep_no, j, 0x80000000 | stream).  The
// movement stream (env_round.cu) puts the slot's reset count, a non-negative int32, in c3, and the epsilon-greedy
// stream (dgn_kernels.cuh) the upper half of the 64-bit round counter, so neither ever sets bit 31 of c3: the three
// streams never share a counter, even under the same seed.
#pragma once
#include "common.cuh"

namespace episode_sampler {

constexpr uint32_t kDomain = 0x80000000u;
enum Stream : uint32_t { kScalars = 0, kGraph = 1, kSource = 2, kNodeKeys = 3 };

__device__ __forceinline__ Philox4 draw(const MlsEpisodeSampler& s, uint32_t slot, uint32_t ep_no, uint32_t stream,
                                        uint32_t j) {
  return philox4x32_10(s.seed, ((uint64_t)ep_no << 32) | slot, ((uint64_t)(kDomain | stream) << 32) | j);
}

// Lemire's multiply-shift bounded draw with rejection: exactly uniform over [0, n).  A rejected word is replaced by
// word 0 of draw j = 1, 2, ... of `stream`.
__device__ __forceinline__ int bounded(const MlsEpisodeSampler& s, uint32_t slot, uint32_t ep_no, uint32_t stream,
                                       uint32_t x, uint32_t n) {
  uint64_t m = (uint64_t)x * n;
  if ((uint32_t)m < n) {
    const uint32_t t = (0u - n) % n;    // 2^32 mod n
    for (uint32_t j = 1; (uint32_t)m < t; ++j) m = (uint64_t)draw(s, slot, ep_no, stream, j).v[0] * n;
  }
  return (int)(m >> 32);
}

struct Scalars {
  int graph, source, k;
};

// The per-episode draws; every thread of the episode may call it (it is a pure function of its arguments).
__device__ __forceinline__ Scalars scalars(const MlsEpisodeSampler& s, int n_nodes, uint32_t slot, uint32_t ep_no) {
  const Philox4 r = draw(s, slot, ep_no, kScalars, 0);
  Scalars o;
  o.graph = bounded(s, slot, ep_no, kGraph, r.v[0], (uint32_t)s.pool_size);
  o.source = bounded(s, slot, ep_no, kSource, r.v[1], (uint32_t)n_nodes);
  const double u = u01_from_u32x2(r.v[2], r.v[3]);
  const double density = __dadd_rn(0.1, __dmul_rn(1.0 - 0.1, u));    // numpy: low + (high - low) * u, no FMA
  o.k = (int)__dmul_rn(density, (double)n_nodes);
  return o;
}

// Node i's keys: .x orders the interest subset, .y the scripted subset.
__device__ __forceinline__ ulonglong2 node_keys(const MlsEpisodeSampler& s, uint32_t slot, uint32_t ep_no, int i) {
  const Philox4 r = draw(s, slot, ep_no, kNodeKeys, (uint32_t)i);
  return make_ulonglong2(((uint64_t)r.v[0] << 32) | r.v[1], ((uint64_t)r.v[2] << 32) | r.v[3]);
}

// Membership of node i, given the keys of all n_nodes nodes of its episode (keys[j] = node_keys(.., j)).
__device__ __forceinline__ void membership(const ulonglong2* keys, int n_nodes, int i, const Scalars& e,
                                           const MlsEpisodeSampler& s, bool& interested, bool& scripted) {
  const ulonglong2 mine = keys[i];
  int ri = 0, rs = 0;
#pragma unroll 1
  for (int j = 0; j < n_nodes; ++j) {
    const ulonglong2 o = keys[j];
    ri += (o.x < mine.x || (o.x == mine.x && j < i)) ? 1 : 0;
    rs += (o.y < mine.y || (o.y == mine.y && j < i)) ? 1 : 0;
  }
  interested = ri < e.k;
  scripted = rs < s.n_scripted && !(s.drop_source_from_scripted && i == e.source);
}

}  // namespace episode_sampler
