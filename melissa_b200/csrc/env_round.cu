// Batched environment round for Melissa's dissemination episodes (sm_100a).
//
// One thread per (episode, node); an episode occupies NP = 32*ceil(N/32) consecutive
// threads (1 warp for N<=32, 2 for N<=64, ...), a CTA carries G = 256/NP episodes.
// Episode-wide sets (who transmits, who holds the message, who is interested ...) are
// bitmasks built with one __ballot_sync per warp and exchanged through shared memory;
// every node keeps its own adjacency row (W words) in registers, the neighbour rows it
// needs for the 2-hop set / MPR live in shared memory.
//
// Semantics follow the reference line by line (see include/melissa_b200.h for the map):
//   World.step            graph_env/env/utils/core.py:225-266   -> world_step()
//   relay_message         core.py:268-279                       -> "relay pass"
//   move_graph            core.py:281-319                       -> "move"
//   heuristics            heuristics/core.py:12-62, mpr.py:7-72 -> scripted_action(), mpr_select()
//   GraphEnv.step / _execute_world_step / reward / obs rows
//                         graph_env/env/graph.py:303-389,402-463,254-271 -> finalize_round()
//   World.reset + GraphEnv.reset  core.py:388-437, graph.py:222-248 -> reset path
#include "common.cuh"
#include "episode_sampler.cuh"

namespace {

constexpr int kThreads = 256;
constexpr double kRadius = 0.20;          // constants.py:1
constexpr double kMoveStep = 0.06;        // constants.py:4
constexpr int kTTL = 4;                   // graph.py:332

struct EnvParams {
  MlsEnvDesc d;
  MlsEnvState s;
  MlsRoundInputs in;
  MlsRoundOutputs out;
  MlsResetTuples tup;      // reset tuples (mode 1) / recycle pool (mode 0, count==0 -> none)
  MlsEpisodeSampler smp;   // smp_on: resets / restarts draw from the device episode sampler instead of `tup`
  int smp_on;              // selects the SAMPLED kernels
  const int32_t* env_ids;  // mode 1
  int mode;                // 0 step, 1 reset, 2 info only
  int n_work;
};

enum { M_I = 0, M_A, M_B, M_C, M_COUNT };   // shared mask slots

template <int W>
struct Th {
  uint32_t adj[W];
  uint32_t rfrom[W];
  uint32_t node;
  uint32_t rc;
  double px, py;
};
struct Ep {
  int source, world_msgs, num_moves, graph, n_resets;
  double rsum;
};

template <int W>
struct Smem {
  uint32_t* adj;   // [G][NP][W]
  uint32_t* rf;    // [G][NP][W]
  uint32_t* mask;  // [M_COUNT][G][W]
  double* pos;     // [G][NP][2]
  double* rew;     // [G][NP]
  int* cnt;        // [G][4]
  int G, NP;
  __device__ uint32_t* adj_row(int le, int j) const { return adj + ((size_t)le * NP + j) * W; }
  __device__ uint32_t* rf_row(int le, int j) const { return rf + ((size_t)le * NP + j) * W; }
  __device__ uint32_t* m(int slot, int le) const { return mask + ((size_t)slot * G + le) * W; }
};

template <int W>
__device__ __forceinline__ bool any_w(const uint32_t (&a)[W]) {
  uint32_t o = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) o |= a[w];
  return o != 0;
}
template <int W>
__device__ __forceinline__ int popc_w(const uint32_t (&a)[W]) {
  int c = 0;
#pragma unroll
  for (int w = 0; w < W; ++w) c += __popc(a[w]);
  return c;
}

// publish one predicate per node as an episode bitmask (NP is a multiple of 32, so a warp
// never straddles two episodes or two mask words)
template <int W>
__device__ __forceinline__ void publish(const Smem<W>& sm, int slot, int le, int wq, bool pred) {
  uint32_t bal = __ballot_sync(0xffffffffu, pred);
  if ((threadIdx.x & 31) == 0) sm.m(slot, le)[wq] = bal;
}
template <int W>
__device__ __forceinline__ void read_mask(const Smem<W>& sm, int slot, int le, uint32_t (&o)[W]) {
#pragma unroll
  for (int w = 0; w < W; ++w) o[w] = sm.m(slot, le)[w];
}

// heuristics/mpr.py:7-72 on bitmask rows.  Adjacency is symmetric, so the providers of a
// strict 2-hop node t are adj[t] & N1(a).
template <int W>
__device__ void mpr_select(const Smem<W>& sm, int le, int self_i, const uint32_t (&n1)[W], uint32_t (&mpr)[W]) {
  uint32_t n2[W], unc[W];
#pragma unroll
  for (int w = 0; w < W; ++w) { n2[w] = n1[w]; mpr[w] = 0; }
#pragma unroll
  for (int w = 0; w < W; ++w) {
    uint32_t bits = n1[w];
    while (bits) {
      int j = w * 32 + __ffs(bits) - 1;
      bits &= bits - 1;
      const uint32_t* r = sm.adj_row(le, j);
#pragma unroll
      for (int v = 0; v < W; ++v) n2[v] |= r[v];
    }
  }
#pragma unroll
  for (int w = 0; w < W; ++w) if (w == (self_i >> 5)) n2[w] &= ~(1u << (self_i & 31));
#pragma unroll
  for (int w = 0; w < W; ++w) unc[w] = n2[w] & ~n1[w];      // strict 2-hop set
  // unique providers (mpr.py:44-48): covers ONLY that 2-hop node
#pragma unroll
  for (int w = 0; w < W; ++w) {
    uint32_t bits = unc[w];
    while (bits) {
      int t = w * 32 + __ffs(bits) - 1;
      uint32_t tb = bits & (0u - bits);
      bits &= bits - 1;
      const uint32_t* r = sm.adj_row(le, t);
      int c = 0;
#pragma unroll
      for (int v = 0; v < W; ++v) c += __popc(r[v] & n1[v]);
      if (c == 1) {
#pragma unroll
        for (int v = 0; v < W; ++v) mpr[v] |= r[v] & n1[v];
        unc[w] &= ~tb;
      }
    }
  }
  // greedy cover (mpr.py:53-70): max reach, ties -> largest id
  while (any_w<W>(unc)) {
    int best = -1, bestc = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      uint32_t bits = n1[w];
      while (bits) {
        int x = w * 32 + __ffs(bits) - 1;
        bits &= bits - 1;
        const uint32_t* r = sm.adj_row(le, x);
        int c = 0;
#pragma unroll
        for (int v = 0; v < W; ++v) c += __popc(r[v] & unc[v]);
        if (c > 0 && c >= bestc) { bestc = c; best = x; }
      }
    }
    if (best < 0) break;   // cannot happen: every strict 2-hop node has a provider
#pragma unroll
    for (int w = 0; w < W; ++w) if (w == (best >> 5)) mpr[w] |= 1u << (best & 31);
    const uint32_t* r = sm.adj_row(le, best);
#pragma unroll
    for (int v = 0; v < W; ++v) unc[v] &= ~r[v];
  }
}

// World.step (core.py:225-266).  `act` is agent.action on entry (-1 None) and on exit the
// value the reference leaves in agent.action (scripted agents: 0, core.py:264-266).
// `en` = this thread is a real node of an episode that takes part in this call.
template <int W>
__device__ __forceinline__ int world_step(const EnvParams& p, const Smem<W>& sm, Th<W>& th, Ep& ep,
                                          int act, bool en, bool reset_step, int le, int i, int wq,
                                          uint32_t mybit, int N, size_t in_row) {
  const int heur = p.d.heuristic;
  const bool cb = en && (th.node & MLS_F_SCRIPTED) && heur != MLS_HEUR_NONE;   // has action_callback
  bool hm = th.node & MLS_F_HAS_MESSAGE;
  const bool org = th.node & MLS_F_ORIGIN;
  bool hta = th.node & MLS_F_HAS_TAKEN_ACTION;
  int msgs = (th.node >> MLS_NODE_MSGS_SHIFT) & 0xff;

  // --- scripted heuristics, first loop (core.py:226-234)
  if (cb) {
    if (heur == MLS_HEUR_SILENT) act = 0;
    else if (heur == MLS_HEUR_SIMPLE_BROADCAST) act = hta ? 0 : 1;
    else if (heur == MLS_HEUR_BROADCAST_IF_ANY_INTERESTED) {
      // number_interested_neighbors is zeroed by Agent.reset and only refreshed by
      // move_graph (core.py:68,286-287,323-328): always 0 on static graphs / in the reset step
      int nin = 0;
      if (p.d.dynamic && !reset_step) {
        uint32_t I[W];
        read_mask<W>(sm, M_I, le, I);
#pragma unroll
        for (int w = 0; w < W; ++w) nin += __popc(th.adj[w] & I[w]);
      }
      act = nin > 0 ? 1 : 0;
    } else if (heur == MLS_HEUR_PROBABILISTIC_GOSSIP) {
      act = hta ? 0 : (p.in.gossip_bits ? (p.in.gossip_bits[in_row * N + i] ? 1 : 0) : 0);
    }
  }
  const bool relay_heur = (heur == MLS_HEUR_MPR || heur == MLS_HEUR_PROBABILISTIC_RELAY);
  if (relay_heur) {   // CTA-uniform
    uint32_t* myrf = sm.rf_row(le, i);
#pragma unroll
    for (int w = 0; w < W; ++w) myrf[w] = 0;
    __syncthreads();
    if (cb) {
      uint32_t sel[W];
      if (heur == MLS_HEUR_MPR) {
        mpr_select<W>(sm, le, i, th.adj, sel);
      } else {
#pragma unroll
        for (int w = 0; w < W; ++w)
          sel[w] = p.in.relay_bits ? (p.in.relay_bits[(in_row * N + i) * W + w] & th.adj[w]) : 0u;
      }
#pragma unroll
      for (int w = 0; w < W; ++w) {
        uint32_t bits = sel[w];
        while (bits) {
          int nbr = w * 32 + __ffs(bits) - 1;
          bits &= bits - 1;
          atomicOr(&sm.rf_row(le, nbr)[wq], mybit);     // agents[nbr].relays_for[self] = 1
        }
      }
    }
    __syncthreads();
    if (cb) {   // second loop (core.py:236-243)
      uint32_t rf[W];
      bool got = false;
#pragma unroll
      for (int w = 0; w < W; ++w) { rf[w] = myrf[w]; got |= (rf[w] & th.rfrom[w]) != 0; }
      if (any_w<W>(rf)) {
        act = 0;
        if (!hta && (hm || org) && (got || org)) act = 1;
      }
    }
  }
  // --- source override (core.py:246)
  if (en && i == ep.source && msgs == 0) act = 1;

  // --- relay pass in id order (core.py:249-254, 268-279)
  const bool want = en && act > 0;
  const bool cascade = (heur == MLS_HEUR_SIMPLE_BROADCAST || heur == MLS_HEUR_BROADCAST_IF_ANY_INTERESTED ||
                        heur == MLS_HEUR_PROBABILISTIC_GOSSIP);
  uint32_t T[W];
  if (!cascade) {
    publish<W>(sm, M_A, le, wq, want && hm);
    __syncthreads();
  } else {
    // a scripted node may want to transmit before it holds the message: a lower-id sender
    // can hand it the message within the same pass (ordered cascade)
    publish<W>(sm, M_B, le, wq, want);
    publish<W>(sm, M_C, le, wq, en && hm);
    __syncthreads();
    if (i == 0) {
      uint32_t wantm[W], hmm[W], t[W];
      read_mask<W>(sm, M_B, le, wantm);
      read_mask<W>(sm, M_C, le, hmm);
#pragma unroll
      for (int w = 0; w < W; ++w) t[w] = 0;
      for (int n = 0; n < N; ++n) {
        const int nw = n >> 5;
        const uint32_t nb = 1u << (n & 31);
        uint32_t wv = 0, hv = 0;
#pragma unroll
        for (int w = 0; w < W; ++w) if (w == nw) { wv = wantm[w]; hv = hmm[w]; }
        if ((wv & nb) && (hv & nb)) {
          const uint32_t* r = sm.adj_row(le, n);
#pragma unroll
          for (int w = 0; w < W; ++w) { hmm[w] |= r[w]; if (w == nw) t[w] |= nb; }
        }
      }
#pragma unroll
      for (int w = 0; w < W; ++w) sm.m(M_A, le)[w] = t[w];
    }
    __syncthreads();
  }
  read_mask<W>(sm, M_A, le, T);
  if (en) {
    int cnt = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) {
      uint32_t r = th.adj[w] & T[w];
      cnt += __popc(r);
      th.rfrom[w] |= r;
    }
    if (cnt) hm = true;
    th.rc += cnt;
    bool tx = false;
#pragma unroll
    for (int w = 0; w < W; ++w) if (w == wq) tx = (T[w] & mybit) != 0;
    if (tx) { msgs += 1; hta = true; }
    if (i == 0) ep.world_msgs += popc_w<W>(T);
  }
  // --- move (core.py:281-319): pos += 0.06*U(-1,1); edges = pairs with dist <= 0.2 (fp64)
  if (p.d.dynamic) {   // CTA-uniform
    if (en) {
      double ox, oy;
      if (p.in.move_offsets) {
        ox = p.in.move_offsets[(in_row * 2 + 0) * N + i];
        oy = p.in.move_offsets[(in_row * 2 + 1) * N + i];
      } else {
        // keyed by the batch-wide episode index (sub-batch views draw what the full-batch call draws)
        const uint32_t rng_row = (uint32_t)in_row + (uint32_t)((p.mode == 0 && p.d.batch_episodes > 0) ? p.d.episode_offset : 0);
        // the forced first step of a recycled episode runs before n_resets is bumped and with num_moves == 0, the counter of
        // the previous episode's first round: it draws under its own counter value instead
        Philox4 r = philox4x32_10(p.in.philox_seed, ((uint64_t)rng_row << 32) | (uint32_t)i,
                                  ((uint64_t)(uint32_t)ep.n_resets << 32) | (reset_step ? 0xFFFFFFFFu : (uint32_t)ep.num_moves));
        ox = kMoveStep * (-1.0 + 2.0 * u01_from_u32x2(r.v[0], r.v[1]));
        oy = kMoveStep * (-1.0 + 2.0 * u01_from_u32x2(r.v[2], r.v[3]));
      }
      th.px = th.px + ox;
      th.py = th.py + oy;
    }
    sm.pos[((size_t)le * sm.NP + i) * 2 + 0] = th.px;
    sm.pos[((size_t)le * sm.NP + i) * 2 + 1] = th.py;
    __syncthreads();
    if (en) {
      const double r2 = kRadius * kRadius;
      uint32_t row[W];
#pragma unroll
      for (int w = 0; w < W; ++w) row[w] = 0;
      for (int j = 0; j < N; ++j) {
        double dx = th.px - sm.pos[((size_t)le * sm.NP + j) * 2 + 0];
        double dy = th.py - sm.pos[((size_t)le * sm.NP + j) * 2 + 1];
        double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));    // no FMA contraction
        if (d2 <= r2 && j != i) {
#pragma unroll
          for (int w = 0; w < W; ++w) if (w == (j >> 5)) row[w] |= 1u << (j & 31);
        }
      }
      uint32_t* mine = sm.adj_row(le, i);
#pragma unroll
      for (int w = 0; w < W; ++w) { th.adj[w] = row[w]; mine[w] = row[w]; }
    }
    // the caller syncs before anybody reads the new rows
  }
  if (cb) act = 0;   // core.py:264-266
  if (en) {
    th.node = (th.node & ~(MLS_F_HAS_MESSAGE | MLS_F_HAS_TAKEN_ACTION | (0xffu << MLS_NODE_MSGS_SHIFT))) |
              (hm ? MLS_F_HAS_MESSAGE : 0u) | (hta ? MLS_F_HAS_TAKEN_ACTION : 0u) |
              ((uint32_t)(msgs & 0xff) << MLS_NODE_MSGS_SHIFT);
  }
  return act;
}

template <int W>
__device__ __forceinline__ void write_obs(const EnvParams& p, const Th<W>& th, int act_post, size_t row) {
  // graph.py:254-271
  if (!p.out.obs) return;
  const uint32_t f = th.node;
  float4 a, c;
  a.x = (float)th.px;
  a.y = (float)th.py;
  a.z = (float)popc_w<W>(th.adj);
  a.w = (float)((f >> MLS_NODE_MSGS_SHIFT) & 0xff);
  c.x = act_post > 0 ? 1.0f : 0.0f;
  c.y = (f & MLS_F_INTERESTED) ? 1.0f : 0.0f;
  c.z = (f & (MLS_F_HAS_MESSAGE | MLS_F_ORIGIN)) ? 1.0f : 0.0f;
  c.w = (f & MLS_F_SCRIPTED) ? 0.0f : 1.0f;
  float4* o = reinterpret_cast<float4*>(p.out.obs + row * 8);
  o[0] = a;
  o[1] = c;
}

// adjacency row + position of this node: from the episode's own copy (dynamic graphs, mid-episode) or
// from the topology pool (static graphs, and every reset)
template <int W>
__device__ __forceinline__ void load_topology(const EnvParams& p, const Smem<W>& sm, Th<W>& th, int graph, bool valid,
                                              bool do_reset, size_t row, int N, int le, int i) {
  if (!valid) return;
  if (p.d.dynamic && !do_reset) {
#pragma unroll
    for (int w = 0; w < W; ++w) th.adj[w] = p.s.adj[row * W + w];
    th.px = p.s.pos[row * 2 + 0];
    th.py = p.s.pos[row * 2 + 1];
  } else {
    const size_t gr = (size_t)graph * N + i;
#pragma unroll
    for (int w = 0; w < W; ++w) th.adj[w] = p.s.pool_adj[gr * W + w];
    th.px = p.s.pool_pos[gr * 2 + 0];
    th.py = p.s.pool_pos[gr * 2 + 1];
  }
  uint32_t* mine = sm.adj_row(le, i);
#pragma unroll
  for (int w = 0; w < W; ++w) mine[w] = th.adj[w];
}

// SAMPLED: the reset / recycle branch draws its tuples from the device episode sampler (p.smp) instead of p.tup.
// The sampled kernels of W <= 2 are held to the 64 registers of the pool kernels (16 CTAs of 64 threads per SM).
template <int W, bool SAMPLED>
__global__ void __launch_bounds__(kThreads, SAMPLED && W <= 2 ? 4 : 0) env_round_kernel(const EnvParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = p.d.n_nodes;
  const int NP = ((N + 31) >> 5) << 5;
  const int G = blockDim.x / NP;
  Smem<W> sm;
  sm.G = G; sm.NP = NP;
  {
    unsigned char* q = smem_raw;
    sm.pos = reinterpret_cast<double*>(q); q += sizeof(double) * G * NP * 2;
    sm.rew = reinterpret_cast<double*>(q); q += sizeof(double) * G * NP;
    sm.adj = reinterpret_cast<uint32_t*>(q); q += sizeof(uint32_t) * G * NP * W;
    sm.rf = reinterpret_cast<uint32_t*>(q); q += sizeof(uint32_t) * G * NP * W;
    sm.mask = reinterpret_cast<uint32_t*>(q); q += sizeof(uint32_t) * M_COUNT * G * W;
    sm.cnt = reinterpret_cast<int*>(q);
  }
  const int le = threadIdx.x / NP;
  const int i = threadIdx.x - le * NP;
  const int wq = i >> 5;
  const uint32_t mybit = 1u << (i & 31);
  const int k = blockIdx.x * G + le;
  const bool ep_valid = le < G && k < p.n_work;
  const int b = ep_valid ? ((p.mode == 1 && p.env_ids) ? p.env_ids[k] : k) : 0;
  const bool valid = ep_valid && i < N;
  const size_t row = (size_t)b * N + i;
  const int B = p.d.batch_episodes > 0 ? p.d.batch_episodes : p.d.n_episodes;   // batch-wide count (sub-batch views)
  const int b_off = p.d.batch_episodes > 0 ? p.d.episode_offset : 0;

  Th<W> th;
#pragma unroll
  for (int w = 0; w < W; ++w) { th.adj[w] = 0; th.rfrom[w] = 0; }
  th.node = 0; th.rc = 0; th.px = 0.0; th.py = 0.0;
  Ep ep;
  ep.source = -1; ep.world_msgs = 0; ep.num_moves = 0; ep.graph = 0; ep.n_resets = 0; ep.rsum = 0.0;

  bool do_reset = (p.mode == 1) && ep_valid;
  int act_post = 0;
  if (i < 4 && le < G) sm.cnt[le * 4 + i] = 0;
  if (threadIdx.x == 0) sm.cnt[G * 4] = 0;
  // mask words beyond the episode's warps (W is a power of two, NP / 32 need not be: N = 65..96, 129..224) are never
  // written by publish(): clear them once, or stale shared memory shows up as phantom nodes in every mask
  {
    const int wpn = NP >> 5;
    if (wpn < W)
      for (int t = threadIdx.x; t < M_COUNT * G * (W - wpn); t += blockDim.x)
        sm.mask[(t / (W - wpn)) * W + wpn + t % (W - wpn)] = 0u;
  }

  if (p.mode != 1) {
    // ------------------------------------------------------------ load state
    if (ep_valid) {
      const int32_t* e = p.s.episode + (size_t)b * MLS_EP_STRIDE;
      ep.source = e[MLS_EP_SOURCE]; ep.world_msgs = e[MLS_EP_WORLD_MSGS]; ep.num_moves = e[MLS_EP_NUM_MOVES];
      ep.graph = e[MLS_EP_GRAPH]; ep.n_resets = e[MLS_EP_N_RESETS];
      ep.rsum = p.s.rewards_sum[b];
    }
    if (valid) {
      th.node = p.s.node[row];
      th.rc = p.s.recv_count[row];
      if (p.s.recv_from) {
#pragma unroll
        for (int w = 0; w < W; ++w) th.rfrom[w] = p.s.recv_from[row * W + w];
      }
    }
    load_topology<W>(p, sm, th, ep.graph, valid, do_reset, row, N, le, i);
    publish<W>(sm, M_I, le, wq, valid && (th.node & MLS_F_INTERESTED));
    __syncthreads();
  }

  if (p.mode == 0) {
    // ------------------------------------------------------------ one round (graph.py:303-359)
    const bool acted = valid && (th.node & MLS_F_ACTIVE);
    int act = -1;
    if (acted) {
      int a = p.in.actions[row];
      act = a < 0 ? -1 : (a > 0 ? 1 : 0);
      th.node += 1u << MLS_NODE_STEPS_SHIFT;                    // steps_taken += 1 (graph.py:316-318)
    }
    act_post = world_step<W>(p, sm, th, ep, act, valid, false, le, i, wq, mybit, N, (size_t)b);
    // masks on the post-step state
    publish<W>(sm, M_B, le, wq, valid && (th.node & MLS_F_HAS_MESSAGE));
    publish<W>(sm, M_C, le, wq, acted);
    __syncthreads();
    uint32_t I[W], M[W], n2[W];
    read_mask<W>(sm, M_I, le, I);
    read_mask<W>(sm, M_B, le, M);
    double r = 0.0;
    if (acted) {
      // reward (graph.py:402-463) on the post-step (post-move) neighbourhood
#pragma unroll
      for (int w = 0; w < W; ++w) n2[w] = th.adj[w];
#pragma unroll
      for (int w = 0; w < W; ++w) {
        uint32_t bits = th.adj[w];
        while (bits) {
          int j = w * 32 + __ffs(bits) - 1;
          bits &= bits - 1;
          const uint32_t* rr = sm.adj_row(le, j);
#pragma unroll
          for (int v = 0; v < W; ++v) n2[v] |= rr[v];
        }
      }
#pragma unroll
      for (int w = 0; w < W; ++w) if (w == wq) n2[w] &= ~mybit;
      uint32_t MO[W];
#pragma unroll
      for (int w = 0; w < W; ++w) MO[w] = M[w];
#pragma unroll
      for (int w = 0; w < W; ++w) if (w == (ep.source >> 5)) MO[w] |= 1u << (ep.source & 31);
      int t = 0, c = 0, d = 0, nu = 0, nc = 0, u = 0, i1 = 0;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        t += __popc(n2[w] & I[w]);
        c += __popc(n2[w] & I[w] & MO[w]);
        d += __popc(th.adj[w]);
        nu += __popc(th.adj[w] & ~I[w]);
        nc += __popc(th.adj[w] & M[w]);
        u += __popc(th.adj[w] & I[w] & ~MO[w]);
        i1 += __popc(th.adj[w] & I[w]);
      }
      r = t > 0 ? __ddiv_rn((double)c, (double)t) : 0.0;
      if (act_post > 0) {
        double pu = d > 0 ? __ddiv_rn((double)nu, (double)d) : 0.0;
        double pc = d > 0 ? __ddiv_rn((double)nc, (double)d) : 0.0;
        r = __dsub_rn(r, __dadd_rn(pu, pc));
      } else if (u > 0) {
        r = __dsub_rn(r, __ddiv_rn((double)u, (double)i1));
      }
    }
    sm.rew[(size_t)le * NP + i] = r;
    // TTL (graph.py:330-334) and next active set (graph.py:336-345)
    bool trunc = th.node & MLS_F_TRUNCATED;
    if (acted && (int)((th.node >> MLS_NODE_STEPS_SHIFT) & 0xff) >= kTTL) trunc = true;
    const bool elig = p.d.is_testing || !(th.node & MLS_F_SCRIPTED);
    const bool active = valid && (th.node & MLS_F_HAS_MESSAGE) && !trunc && elig;
    if (valid)
      th.node = (th.node & ~(MLS_F_TRUNCATED | MLS_F_ACTIVE)) | (trunc ? MLS_F_TRUNCATED : 0u) |
                (active ? MLS_F_ACTIVE : 0u);
    publish<W>(sm, M_A, le, wq, active);
    if (p.out.info && valid) {
      atomicAdd(&sm.cnt[le * 4 + 0], (int)((th.node >> MLS_NODE_MSGS_SHIFT) & 0xff));
      atomicAdd(&sm.cnt[le * 4 + 1], (int)th.rc);
      atomicAdd(&sm.cnt[le * 4 + 2], popc_w<W>(th.adj));
    }
    __syncthreads();
    uint32_t A[W], ACT[W];
    read_mask<W>(sm, M_A, le, A);
    read_mask<W>(sm, M_C, le, ACT);
    const bool done = !any_w<W>(A);
    const int n_acted = popc_w<W>(ACT);
    if (ep_valid && i == 0) {
      // episode_rewards_sum += reward, agents in id order (graph.py:378-389): walk the acted bits only
      double s = ep.rsum;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        uint32_t bits = ACT[w];
        while (bits) {
          const int n = w * 32 + __ffs(bits) - 1;
          bits &= bits - 1;
          s = __dadd_rn(s, sm.rew[(size_t)le * NP + n]);
        }
      }
      ep.rsum = s;
      ep.num_moves += 1;
      if (p.out.done) p.out.done[b] = done ? 1 : 0;
      if (p.out.info) {
        int ni = 0, ci = 0, um = 0;
#pragma unroll
        for (int w = 0; w < W; ++w) { ni += __popc(I[w]); ci += __popc(M[w] & I[w]); um += __popc(M[w] & ~I[w]); }
        int4* o4 = reinterpret_cast<int4*>(p.out.info + b);          // MlsInfo = 12 x int32 + double (56 bytes, 8-aligned)
        int* o = reinterpret_cast<int*>(p.out.info + b);
        o[0] = ep.world_msgs; o[1] = popc_w<W>(M); o[2] = sm.cnt[le * 4 + 0]; o[3] = sm.cnt[le * 4 + 1];
        o[4] = sm.cnt[le * 4 + 2]; o[5] = ni; o[6] = ci; o[7] = um;
        o[8] = ep.num_moves; o[9] = n_acted; o[10] = ep.n_resets; o[11] = 0;
        p.out.info[b].episode_rewards_sum = ep.rsum;
        (void)o4;
      }
      if (p.out.transitions && n_acted) atomicAdd(&sm.cnt[G * 4], n_acted);
    }
    if (valid) {
      if (p.out.reward) p.out.reward[row] = r;
      if (p.out.terminated) p.out.terminated[row] = trunc ? 1 : 0;
    }
    do_reset = ep_valid && done && (SAMPLED || p.tup.count > 0);
  } else if (p.mode == 2) {
    // ------------------------------------------------------------ get_info only (graph.py:149-179)
    publish<W>(sm, M_B, le, wq, valid && (th.node & MLS_F_HAS_MESSAGE));
    if (valid) {
      atomicAdd(&sm.cnt[le * 4 + 0], (int)((th.node >> MLS_NODE_MSGS_SHIFT) & 0xff));
      atomicAdd(&sm.cnt[le * 4 + 1], (int)th.rc);
      atomicAdd(&sm.cnt[le * 4 + 2], popc_w<W>(th.adj));
    }
    __syncthreads();
    if (ep_valid && i == 0) {
      uint32_t I[W], M[W];
      read_mask<W>(sm, M_I, le, I);
      read_mask<W>(sm, M_B, le, M);
      MlsInfo inf;
      inf.total_messages_transmitted = ep.world_msgs;
      inf.covered = popc_w<W>(M);
      inf.messages_sent = sm.cnt[le * 4 + 0];
      inf.messages_received = sm.cnt[le * 4 + 1];
      inf.n_neighbours = sm.cnt[le * 4 + 2];
      int ni = 0, ci = 0, um = 0;
#pragma unroll
      for (int w = 0; w < W; ++w) { ni += __popc(I[w]); ci += __popc(M[w] & I[w]); um += __popc(M[w] & ~I[w]); }
      inf.interested_agents = ni;
      inf.coverage_interested_count = ci;
      inf.uninterested_with_message = um;
      inf.num_moves = ep.num_moves;
      inf.n_acted = 0;
      inf.episodes_started = ep.n_resets;
      inf.reserved = 0;
      inf.episode_rewards_sum = ep.rsum;
      p.out.info[b] = inf;
    }
    return;
  }

  // ---------------------------------------------------------------- reset / recycle
  const bool any_reset = (p.mode == 1) ? true : (__syncthreads_or(do_reset ? 1 : 0) != 0);
  if (p.mode == 0 && threadIdx.x == 0 && p.out.transitions && sm.cnt[G * 4])
    atomicAdd(p.out.transitions, (unsigned long long)sm.cnt[G * 4]);      // one atomic per CTA
  if (any_reset) {
    size_t trow = 0;
    bool s_int = false, s_scr = false;
    if constexpr (SAMPLED) {
      // episode number n_resets of global slot b + b_off + slot_offset.  The node keys go through sm.pos, which nobody
      // reads again before the forced step rewrites it (after the barrier in front of world_step)
      ulonglong2* keys = reinterpret_cast<ulonglong2*>(sm.pos) + (size_t)le * NP;
      episode_sampler::Scalars es{};
      uint32_t slot = 0;
      if (do_reset) {
        if (p.mode == 1) ep.n_resets = p.s.episode[(size_t)b * MLS_EP_STRIDE + MLS_EP_N_RESETS];
        slot = (uint32_t)(b + b_off) + (uint32_t)p.smp.slot_offset;
        es = episode_sampler::scalars(p.smp, N, slot, (uint32_t)ep.n_resets);
        if (valid) keys[i] = episode_sampler::node_keys(p.smp, slot, (uint32_t)ep.n_resets, i);
      }
      __syncthreads();
      if (do_reset) {
        ep.graph = es.graph;
        ep.source = es.source;
        if (valid) episode_sampler::membership(keys, N, i, es, p.smp, s_int, s_scr);
      }
    }
    if (do_reset) {
      // World.reset (core.py:388-437) + GraphEnv.reset (graph.py:227-248)
      if constexpr (!SAMPLED) {
        trow = (p.mode == 1) ? (size_t)k : (size_t)(((long long)b + b_off + (long long)ep.n_resets * B) % p.tup.count);
        ep.graph = p.tup.graph_index[trow];
        ep.source = p.tup.source[trow];
      }
      ep.world_msgs = 0; ep.num_moves = 0; ep.rsum = 0.0;
      if (!SAMPLED && p.mode == 1) ep.n_resets = p.s.episode[(size_t)b * MLS_EP_STRIDE + MLS_EP_N_RESETS];
      if (valid) {
        uint32_t f = 0;
        if (SAMPLED ? s_int : (p.tup.interested[trow * W + wq] & mybit) != 0) f |= MLS_F_INTERESTED;
        if (SAMPLED ? s_scr : (p.tup.scripted[trow * W + wq] & mybit) != 0) f |= MLS_F_SCRIPTED;
        if (i == ep.source) f |= MLS_F_ORIGIN | MLS_F_HAS_MESSAGE | (1u << MLS_NODE_STEPS_SHIFT);   // core.py:432-435
        th.node = f;
        th.rc = 0;
#pragma unroll
        for (int w = 0; w < W; ++w) th.rfrom[w] = 0;
      }
      load_topology<W>(p, sm, th, ep.graph, valid, do_reset, row, N, le, i);
    }
    // (threads of episodes that do not reset keep their interest mask slot untouched)
    if (do_reset) publish<W>(sm, M_I, le, wq, valid && (th.node & MLS_F_INTERESTED));
    __syncthreads();
    const bool en = valid && do_reset;
    // move/gossip/relay inputs of the forced step: per tuple in reset mode, per episode when recycling
    const size_t in_row = (p.mode == 1) ? (size_t)k : (size_t)b;
    int a_post = world_step<W>(p, sm, th, ep, -1, en, true, le, i, wq, mybit, N, in_row);
    if (en) {
      act_post = a_post;
      const bool elig = p.d.is_testing || !(th.node & MLS_F_SCRIPTED);
      const bool active = (th.node & MLS_F_HAS_MESSAGE) && elig;                // graph.py:242-246
      th.node = (th.node & ~(MLS_F_TRUNCATED | MLS_F_ACTIVE)) | (active ? MLS_F_ACTIVE : 0u);
    }
    if (do_reset && i == 0) ep.n_resets += 1;
  }

  // ---------------------------------------------------------------- write back
  if (valid) {
    p.s.node[row] = th.node;
    p.s.recv_count[row] = (uint16_t)th.rc;
    if (p.s.recv_from) {
#pragma unroll
      for (int w = 0; w < W; ++w) p.s.recv_from[row * W + w] = th.rfrom[w];
    }
    if (p.d.dynamic) {
#pragma unroll
      for (int w = 0; w < W; ++w) p.s.adj[row * W + w] = th.adj[w];
      p.s.pos[row * 2 + 0] = th.px;
      p.s.pos[row * 2 + 1] = th.py;
    }
    if (p.out.active) p.out.active[row] = (th.node & MLS_F_ACTIVE) ? 1 : 0;
    write_obs<W>(p, th, act_post, row);
  }
  if (ep_valid && i == 0) {
    int32_t* e = p.s.episode + (size_t)b * MLS_EP_STRIDE;
    e[MLS_EP_SOURCE] = ep.source; e[MLS_EP_WORLD_MSGS] = ep.world_msgs; e[MLS_EP_NUM_MOVES] = ep.num_moves;
    e[MLS_EP_GRAPH] = ep.graph; e[MLS_EP_N_RESETS] = ep.n_resets;
    p.s.rewards_sum[b] = ep.rsum;
  }
}

template <int W, bool SAMPLED>
int launch_env(const EnvParams& p, cudaStream_t stream) {
  const int N = p.d.n_nodes;
  const int NP = ((N + 31) / 32) * 32;
  // small CTAs (2 episodes of up to 64 nodes): more independent CTAs per SM overlap each other's load latency and barriers
  const int target = NP <= 64 ? 64 : kThreads;
  int G = target / NP;
  if (G < 1) G = 1;
  const int threads = G * NP;
  const int blocks = (p.n_work + G - 1) / G;
  size_t smem = sizeof(double) * G * NP * 3 + sizeof(uint32_t) * G * NP * W * 2 +
                sizeof(uint32_t) * M_COUNT * G * W + sizeof(int) * (G * 4 + 1);
  if (blocks == 0) return MLS_OK;
  env_round_kernel<W, SAMPLED><<<blocks, threads, smem, stream>>>(p);
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}

template <bool SAMPLED>
int dispatch_w(const EnvParams& p, cudaStream_t st) {
  const int W = (p.d.n_nodes + 31) / 32;
  if (W <= 1) return launch_env<1, SAMPLED>(p, st);
  if (W <= 2) return launch_env<2, SAMPLED>(p, st);
  if (W <= 4) return launch_env<4, SAMPLED>(p, st);
  return launch_env<8, SAMPLED>(p, st);
}

int dispatch_env(const EnvParams& p, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return p.smp_on ? dispatch_w<true>(p, st) : dispatch_w<false>(p, st);
}

int check_common(const MlsEnvDesc* d, const MlsEnvState* s) {
  MLS_CHECK_ARG(d && s, "desc/state is NULL");
  MLS_CHECK_ARG(d->n_nodes >= 1 && d->n_nodes <= MLS_MAX_NODES, "n_nodes must be in [1, %d], got %d", MLS_MAX_NODES, d->n_nodes);
  MLS_CHECK_ARG(d->n_episodes >= 0, "n_episodes < 0");
  MLS_CHECK_ARG(d->heuristic >= MLS_HEUR_NONE && d->heuristic <= MLS_HEUR_MPR, "Unknown heuristic policy: %d", d->heuristic);
  MLS_CHECK_ARG(s->node && s->recv_count && s->episode && s->rewards_sum, "state.node/recv_count/episode/rewards_sum must be set");
  MLS_CHECK_ARG(s->pool_adj && s->pool_pos && s->pool_size > 0, "topology pool must be set");
  MLS_CHECK_ARG(!d->dynamic || (s->adj && s->pos), "dynamic_graph needs state.adj and state.pos");
  const bool relay = d->heuristic == MLS_HEUR_MPR || d->heuristic == MLS_HEUR_PROBABILISTIC_RELAY;
  MLS_CHECK_ARG(!relay || s->recv_from, "heuristic %d needs state.recv_from", d->heuristic);
  return MLS_OK;
}

// mls_episode_sample: one thread per (tuple, node), NP = 32*ceil(N/32) threads per tuple as in the round kernel.
__global__ void __launch_bounds__(kThreads) episode_sample_kernel(const MlsEpisodeSampler smp, int N, int W,
                                                                  const int32_t* slot, const int32_t* episode_no, int n,
                                                                  int32_t* graph_index, int32_t* source, uint32_t* interested,
                                                                  uint32_t* scripted) {
  __shared__ ulonglong2 keys[kThreads];
  const int NP = ((N + 31) >> 5) << 5;
  const int G = blockDim.x / NP;
  const int le = threadIdx.x / NP;
  const int i = threadIdx.x - le * NP;
  const int m = blockIdx.x * G + le;
  const bool ok = m < n;          // uniform over the tuple's warps
  const bool valid = ok && i < N;
  episode_sampler::Scalars es{};
  if (ok) {
    const uint32_t s = (uint32_t)slot[m] + (uint32_t)smp.slot_offset, r = (uint32_t)episode_no[m];
    es = episode_sampler::scalars(smp, N, s, r);
    if (valid) keys[le * NP + i] = episode_sampler::node_keys(smp, s, r, i);
  }
  __syncthreads();
  bool in_i = false, in_s = false;
  if (valid) episode_sampler::membership(keys + le * NP, N, i, es, smp, in_i, in_s);
  const uint32_t bi = __ballot_sync(0xffffffffu, in_i), bs = __ballot_sync(0xffffffffu, in_s);
  if (!ok) return;
  const size_t row = (size_t)m * W;
  if ((i & 31) == 0) { interested[row + (i >> 5)] = bi; scripted[row + (i >> 5)] = bs; }
  if (i == 0) {
    graph_index[m] = es.graph;
    source[m] = es.source;
    for (int w = NP >> 5; w < W; ++w) { interested[row + w] = 0u; scripted[row + w] = 0u; }
  }
}

}  // namespace

// The word count W the kernels are instantiated with is the next of {1,2,4,8} >= ceil(N/32),
// but every [..][W] array in the ABI uses the exact W = ceil(N/32).  To keep the ABI simple
// the kernels index those arrays with the template W, so the host pads to that width.
extern "C" int mls_words_per_row(int n_nodes) {
  const int w = (n_nodes + 31) / 32;
  return w <= 1 ? 1 : (w <= 2 ? 2 : (w <= 4 ? 4 : 8));
}

extern "C" int mls_env_reset(const MlsEnvDesc* desc, const MlsEnvState* state, const int32_t* env_ids,
                             const MlsResetTuples* tuples, const MlsRoundInputs* in, const MlsRoundOutputs* out,
                             void* stream) {
  int rc = check_common(desc, state);
  if (rc) return rc;
  MLS_CHECK_ARG(tuples && tuples->count >= 0, "tuples missing");
  MLS_CHECK_ARG(tuples->count <= desc->n_episodes || env_ids, "more tuples than episodes");
  if (tuples->count == 0) return MLS_OK;
  MLS_CHECK_ARG(tuples->graph_index && tuples->source && tuples->interested && tuples->scripted, "tuple arrays missing");
  EnvParams p{};
  p.d = *desc; p.s = *state;
  if (in) p.in = *in;
  if (out) p.out = *out;
  p.tup = *tuples;
  p.env_ids = env_ids;
  p.mode = 1;
  p.n_work = tuples->count;
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_GOSSIP || p.in.gossip_bits, "probabilistic_gossip needs gossip_bits");
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_RELAY || p.in.relay_bits, "probabilistic_relay needs relay_bits");
  return dispatch_env(p, stream);
}

extern "C" int mls_env_step(const MlsEnvDesc* desc, const MlsEnvState* state, const MlsRoundInputs* in,
                            const MlsRoundOutputs* out, const MlsResetTuples* recycle, void* stream) {
  int rc = check_common(desc, state);
  if (rc) return rc;
  MLS_CHECK_ARG(in && in->actions, "actions missing");
  EnvParams p{};
  p.d = *desc; p.s = *state; p.in = *in;
  if (out) p.out = *out;
  if (recycle) {
    p.tup = *recycle;
    MLS_CHECK_ARG(recycle->count == 0 || (recycle->graph_index && recycle->source && recycle->interested && recycle->scripted),
                  "recycle tuple arrays missing");
  }
  p.mode = 0;
  p.n_work = desc->n_episodes;
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_GOSSIP || p.in.gossip_bits, "probabilistic_gossip needs gossip_bits");
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_RELAY || p.in.relay_bits, "probabilistic_relay needs relay_bits");
  return dispatch_env(p, stream);
}

static int check_sampler(const MlsEnvDesc* d, const MlsEnvState* s, const MlsEpisodeSampler* smp) {
  MLS_CHECK_ARG(smp, "sampler is NULL");
  MLS_CHECK_ARG(smp->pool_size >= 1 && smp->pool_size <= s->pool_size,
                "sampler pool_size must be in [1, %d] (the topology pool), got %d", s->pool_size, smp->pool_size);
  MLS_CHECK_ARG(smp->n_scripted >= 0 && smp->n_scripted <= d->n_nodes, "sampler n_scripted must be in [0, %d], got %d",
                d->n_nodes, smp->n_scripted);
  return MLS_OK;
}

extern "C" int mls_env_reset_sampled(const MlsEnvDesc* desc, const MlsEnvState* state, const int32_t* env_ids, int32_t n,
                                     const MlsEpisodeSampler* sampler, const MlsRoundInputs* in, const MlsRoundOutputs* out,
                                     void* stream) {
  int rc = check_common(desc, state);
  if (rc) return rc;
  rc = check_sampler(desc, state, sampler);
  if (rc) return rc;
  MLS_CHECK_ARG(n >= 0, "n < 0");
  MLS_CHECK_ARG(n <= desc->n_episodes || env_ids, "more resets than episodes");
  if (n == 0) return MLS_OK;
  EnvParams p{};
  p.d = *desc; p.s = *state;
  if (in) p.in = *in;
  if (out) p.out = *out;
  p.smp = *sampler;
  p.smp_on = 1;
  p.env_ids = env_ids;
  p.mode = 1;
  p.n_work = n;
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_GOSSIP || p.in.gossip_bits, "probabilistic_gossip needs gossip_bits");
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_RELAY || p.in.relay_bits, "probabilistic_relay needs relay_bits");
  return dispatch_env(p, stream);
}

extern "C" int mls_env_step_sampled(const MlsEnvDesc* desc, const MlsEnvState* state, const MlsRoundInputs* in,
                                    const MlsRoundOutputs* out, const MlsEpisodeSampler* sampler, void* stream) {
  int rc = check_common(desc, state);
  if (rc) return rc;
  rc = check_sampler(desc, state, sampler);
  if (rc) return rc;
  MLS_CHECK_ARG(in && in->actions, "actions missing");
  EnvParams p{};
  p.d = *desc; p.s = *state; p.in = *in;
  if (out) p.out = *out;
  p.smp = *sampler;
  p.smp_on = 1;
  p.mode = 0;
  p.n_work = desc->n_episodes;
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_GOSSIP || p.in.gossip_bits, "probabilistic_gossip needs gossip_bits");
  MLS_CHECK_ARG(desc->heuristic != MLS_HEUR_PROBABILISTIC_RELAY || p.in.relay_bits, "probabilistic_relay needs relay_bits");
  return dispatch_env(p, stream);
}

extern "C" int mls_env_info(const MlsEnvDesc* desc, const MlsEnvState* state, MlsInfo* info, void* stream) {
  int rc = check_common(desc, state);
  if (rc) return rc;
  MLS_CHECK_ARG(info, "info is NULL");
  EnvParams p{};
  p.d = *desc; p.s = *state;
  p.out.info = info;
  p.mode = 2;
  p.n_work = desc->n_episodes;
  return dispatch_env(p, stream);
}

extern "C" int mls_episode_sample(const MlsEpisodeSampler* sampler, int32_t n_nodes, const int32_t* slot,
                                  const int32_t* episode_no, int32_t n, int32_t* graph_index, int32_t* source,
                                  uint32_t* interested, uint32_t* scripted, void* stream) {
  MLS_CHECK_ARG(sampler, "sampler is NULL");
  MLS_CHECK_ARG(n_nodes >= 1 && n_nodes <= MLS_MAX_NODES, "n_nodes must be in [1, %d], got %d", MLS_MAX_NODES, n_nodes);
  MLS_CHECK_ARG(sampler->pool_size >= 1, "sampler pool_size must be >= 1, got %d", sampler->pool_size);
  MLS_CHECK_ARG(sampler->n_scripted >= 0 && sampler->n_scripted <= n_nodes, "sampler n_scripted must be in [0, %d], got %d",
                n_nodes, sampler->n_scripted);
  MLS_CHECK_ARG(n >= 0, "n < 0");
  MLS_CHECK_ARG(slot && episode_no && graph_index && source && interested && scripted, "episode_sample arrays missing");
  if (n == 0) return MLS_OK;
  const int NP = ((n_nodes + 31) / 32) * 32;
  const int G = kThreads / NP;
  episode_sample_kernel<<<(n + G - 1) / G, G * NP, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      *sampler, n_nodes, mls_words_per_row(n_nodes), slot, episode_no, n, graph_index, source, interested, scripted);
  mls_count_launch();
  MLS_LAUNCH_CHECK();
  return MLS_OK;
}
