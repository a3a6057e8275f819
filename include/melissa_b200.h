/* melissa_b200.h -- C ABI of libmelissa_b200.so (hand-written sm_100a CUDA).
 *
 * The reference (RaffaeleGalliera/melissa) is pure Python and has no FFI layer; its
 * boundary for the rollout hot path is Python duck typing.  Each entry point below names
 * the reference interface it replaces (file:line under the reference root).  Host code
 * (melissa_b200/*.py) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host; the caller (PyTorch)
 *    owns every buffer; the library allocates nothing;
 *  - every call enqueues on the given cudaStream_t (passed as void*) and never synchronises;
 *  - return 0 = OK, negative = error; mls_last_error() gives the message (thread local);
 *  - B episodes, N nodes per graph, W = mls_words_per_row(N) words per bitmask row
 *    (ceil(N/32) rounded up to 1, 2, 4 or 8); bit j of a row lives in word j/32, bit j%32.
 */
#ifndef MELISSA_B200_H
#define MELISSA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLS_VERSION 214
#define MLS_MAX_NODES 256

/* ---- errors ------------------------------------------------------------------------- */
#define MLS_OK 0
#define MLS_ERR_INVALID (-1) /* bad argument (the reference raises ValueError)            */
#define MLS_ERR_CUDA (-2)    /* a CUDA runtime call failed                                */
#define MLS_ERR_UNSUPPORTED (-3)

int mls_version(void);
const char* mls_last_error(void);
/* sm count / compute capability of the current device; -2 if no usable GPU. */
int mls_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
/* words per bitmask row for N nodes: 1 (N<=32), 2 (<=64), 4 (<=128), 8 (<=256). */
int mls_words_per_row(int n_nodes);
/* process-wide tuning options (A/B switches for benchmarking; defaults are the fast paths):
 *   "attn_mma"  1 = conv1 attention through the pair-logit table + tcgen05 aggregation (discrete-feature mode)
 *   "conv2_mma" 1 = conv2 attention with half2 logits + tcgen05 aggregation (graphs of <= 64 nodes)
 *   "max_ctas"  test only: n > 0 caps the grid of the persistent kernels at n CTAs (many tiles per CTA); 0 = off
 * set returns MLS_ERR_INVALID and get returns -1 for an unknown key (since version 213 also for the two removed
 * switches of the conv1 kernel choice and the needed-row layout). */
int mls_set_option(const char* key, int value);
int mls_get_option(const char* key);
/* kernels launched by this library since it was loaded (process wide; for bench accounting). */
unsigned long long mls_launch_count(void);

/* ===== environment round ===============================================================
 * Replaces graph_env/env/utils/core.py (World: reset :343-437, step :225-266,
 * relay_message :268-279, move_graph :281-319, neighbour masks :321-341),
 * graph_env/env/utils/heuristics/{core.py:12-62, mpr.py:7-72},
 * graph_env/env/utils/selector.py:1-52 and the round logic of graph_env/env/graph.py
 * (step :303-359, _execute_world_step :361-389, reward :402-463, obs rows :254-271,
 * get_info :149-179). */

enum MlsHeuristic { /* graph_env/env/utils/heuristics/__init__.py:4-11 */
  MLS_HEUR_NONE = 0,
  MLS_HEUR_SILENT = 1,
  MLS_HEUR_SIMPLE_BROADCAST = 2,
  MLS_HEUR_BROADCAST_IF_ANY_INTERESTED = 3,
  MLS_HEUR_PROBABILISTIC_GOSSIP = 4, /* random bits are host-fed (reference uses global np.random) */
  MLS_HEUR_PROBABILISTIC_RELAY = 5,  /* idem */
  MLS_HEUR_MPR = 6
};

typedef struct MlsEnvDesc {
  int32_t n_episodes; /* B */
  int32_t n_nodes;    /* N <= MLS_MAX_NODES */
  int32_t dynamic;    /* dynamic_graph (graph.py:39)                                     */
  int32_t is_testing; /* graph.py:37: scripted agents are policy-stepped too             */
  int32_t heuristic;  /* enum MlsHeuristic                                               */
  /* Sub-batch view (mls_env_step only): the state / output pointers address episodes
   * [episode_offset, episode_offset + n_episodes) of a batch of batch_episodes episodes, so that a caller can
   * pipeline a round in slices (H2D / compute / D2H overlap) with exactly the results of one full-batch call:
   * the recycle-pool row and the device movement stream are keyed by the batch-wide episode index.
   * batch_episodes == 0: not a view (offset 0, batch = n_episodes). */
  int32_t episode_offset;
  int32_t batch_episodes;
  int32_t reserved;
} MlsEnvDesc;

/* per-node packed state word (node[b][i]) */
#define MLS_F_HAS_MESSAGE 0x01u
#define MLS_F_INTERESTED 0x02u
#define MLS_F_SCRIPTED 0x04u
#define MLS_F_ORIGIN 0x08u
#define MLS_F_HAS_TAKEN_ACTION 0x10u
#define MLS_F_TRUNCATED 0x20u
#define MLS_F_ACTIVE 0x40u
#define MLS_NODE_STEPS_SHIFT 8 /* bits 8..15 steps_taken, bits 16..23 messages_transmitted */
#define MLS_NODE_MSGS_SHIFT 16

/* per-episode scalars (episode[b][MLS_EP_*]) */
#define MLS_EP_SOURCE 0
#define MLS_EP_WORLD_MSGS 1
#define MLS_EP_NUM_MOVES 2
#define MLS_EP_GRAPH 3     /* index into the topology pool                                */
#define MLS_EP_N_RESETS 4  /* how many episodes this slot has started (recycling cursor)  */
#define MLS_EP_STRIDE 8

typedef struct MlsEnvState {
  uint32_t* node;          /* [B][N]   packed flags | steps | msgs                        */
  uint16_t* recv_count;    /* [B][N]   sum_j received_from[i][j]                          */
  uint32_t* recv_from;     /* [B][N][W] (received_from[i][j] > 0); needed for MPR / prob. relay, else NULL */
  int32_t* episode;        /* [B][MLS_EP_STRIDE]                                          */
  double* rewards_sum;     /* [B]      episode_rewards_sum (graph.py:389)                 */
  uint32_t* adj;           /* [B][N][W] per-episode adjacency; dynamic mode only, else NULL */
  double* pos;             /* [B][N][2] per-episode positions;  dynamic mode only, else NULL */
  const uint32_t* pool_adj; /* [G][N][W] topology pool (static mode reads it every round)  */
  const double* pool_pos;   /* [G][N][2]                                                   */
  int32_t pool_size;        /* G */
  int32_t pad_;
} MlsEnvState;

/* What an episode starts from (reference reset chain, core.py:371-395; drawn on the host). */
typedef struct MlsResetTuples {
  const int32_t* graph_index;    /* [n] index into the pool                               */
  const int32_t* source;         /* [n]                                                   */
  const uint32_t* interested;    /* [n][W] bitmask                                        */
  const uint32_t* scripted;      /* [n][W] bitmask                                        */
  int32_t count;                 /* n                                                     */
  int32_t pad_;
} MlsResetTuples;

typedef struct MlsInfo { /* graph.py:149-179 as integer counts; fractions = count / N etc. */
  int32_t total_messages_transmitted;
  int32_t covered;                   /* sum has_message                                   */
  int32_t messages_sent;
  int32_t messages_received;
  int32_t n_neighbours;
  int32_t interested_agents;
  int32_t coverage_interested_count;
  int32_t uninterested_with_message;
  int32_t num_moves;
  int32_t n_acted;                   /* agent-transitions of the round just played        */
  int32_t episodes_started;
  int32_t reserved;
  double episode_rewards_sum;
} MlsInfo;

typedef struct MlsRoundInputs {
  const int8_t* actions;        /* [B][N] -1 = None, 0, 1; only entries of active agents are read (graph.py:312-318) */
  const double* move_offsets;   /* [B][2][N] dynamic mode: 0.06*U(-1,1), x then y (core.py:316-319); NULL -> Philox */
  const uint8_t* gossip_bits;   /* [B][N]    probabilistic_gossip draws, else NULL         */
  const uint32_t* relay_bits;   /* [B][N][W] probabilistic_relay draws, else NULL          */
  uint64_t philox_seed;         /* movement stream when move_offsets == NULL               */
} MlsRoundInputs;

typedef struct MlsRoundOutputs {
  float* obs;          /* [B][N][8] obs_matrix rows (graph.py:254-271); NULL = not wanted  */
  double* reward;      /* [B][N]   reward of each agent that acted, 0 elsewhere; NULL ok   */
  uint8_t* active;     /* [B][N]   agents that act next round (graph.py:336-345)           */
  uint8_t* terminated; /* [B][N]   TTL reached (graph.py:330-334); NULL ok                 */
  uint8_t* done;       /* [B]      no agent left to act; NULL ok                           */
  MlsInfo* info;       /* [B]      NULL ok                                                 */
  unsigned long long* transitions; /* [1] += agent-transitions of this round; NULL ok      */
} MlsRoundOutputs;

/* Reset the episodes env_ids[0..n) (NULL = episodes 0..n) from tuples[0..n), including the
 * forced first world step in which the source broadcasts (core.py:437, :246).
 * `in` may carry move_offsets / gossip_bits / relay_bits for that forced step, indexed by
 * tuple (not by episode).  Writes obs/active rows of the reset episodes. */
int mls_env_reset(const MlsEnvDesc* desc, const MlsEnvState* state, const int32_t* env_ids,
                  const MlsResetTuples* tuples, const MlsRoundInputs* in,
                  const MlsRoundOutputs* out, void* stream);

/* One round for all B episodes.  If `recycle` is non-NULL an episode that ends in this round
 * is restarted in the same launch from tuple (b + n_resets*B) % count: reward/terminated/
 * done/info describe the finished round, obs/active describe the fresh episode.
 * Host-fed draws and recycling: the forced first step of a restarted episode reads row b of move_offsets /
 * gossip_bits / relay_bits a second time in the same launch (the reference draws fresh values there); feed draws
 * from the host only without `recycle` (reset with mls_env_reset and its own rows) when that matters.  The device
 * Philox movement stream gives the forced step its own counter value. */
int mls_env_step(const MlsEnvDesc* desc, const MlsEnvState* state, const MlsRoundInputs* in,
                 const MlsRoundOutputs* out, const MlsResetTuples* recycle, void* stream);

/* get_info (graph.py:149-179) for all episodes without stepping. */
int mls_env_info(const MlsEnvDesc* desc, const MlsEnvState* state, MlsInfo* info, void* stream);

/* ---- device episode sampler (since version 214).  The second source of episode resets, next to MlsResetTuples:
 * instead of reading a row of a host-drawn pool, every restart draws a fresh training-mode tuple (core.py:371-395) from
 * a counter-based Philox stream keyed by (seed, global slot, episode number of that slot).  It matches the reference in
 * distribution, not draw for draw (the host pool is the draw-for-draw path):
 *   graph   uniform over [0, pool_size)            source  uniform over [0, N)
 *   k       int((0.1 + 0.9 u) * N), u a 53-bit uniform, in fp64 as numpy's uniform(0.1, 1.0) computes it
 *   interested  a uniform k-subset of the nodes, independent of source
 *   scripted    an independent uniform n_scripted-subset, minus source when drop_source_from_scripted
 * Episode number r of a slot is its episode[b][MLS_EP_N_RESETS] before the restart bumps it (r = 0: first reset).
 * The global slot is the batch-wide episode index (episode_offset + b for a sub-batch view) + slot_offset, so
 * sub-batch views draw what a full-batch call draws, and rank k of a job passing slot_offset = k * B draws
 * episodes no other rank draws.  The counters never meet those of the movement or epsilon-greedy streams. */
typedef struct MlsEpisodeSampler {
  uint64_t seed;
  int32_t pool_size;                 /* graphs drawn from [0, pool_size); 1 <= pool_size <= state.pool_size     */
  int32_t n_scripted;                /* round(ratio * N) with round half to even (Python's round); 0 <= . <= N */
  int32_t drop_source_from_scripted; /* ratio < 1 (core.py:213-215)                                           */
  int32_t slot_offset;               /* added to the batch-wide episode index                                 */
} MlsEpisodeSampler;

/* mls_env_reset with the tuple of episode k drawn by the sampler: slot env_ids[k] (NULL: k), episode number
 * episode[slot][MLS_EP_N_RESETS].  n episodes; `in` rows are indexed by k as in mls_env_reset. */
int mls_env_reset_sampled(const MlsEnvDesc* desc, const MlsEnvState* state, const int32_t* env_ids, int32_t n,
                          const MlsEpisodeSampler* sampler, const MlsRoundInputs* in, const MlsRoundOutputs* out,
                          void* stream);
/* mls_env_step whose finished episodes restart, in the same launch, from the sampler instead of a tuple pool. */
int mls_env_step_sampled(const MlsEnvDesc* desc, const MlsEnvState* state, const MlsRoundInputs* in,
                         const MlsRoundOutputs* out, const MlsEpisodeSampler* sampler, void* stream);
/* Materialise n sampled tuples: tuple m is episode number episode_no[m] of batch-wide slot slot[m] (slot_offset is
 * added as in the environment calls).  Output in the MlsResetTuples layout: graph_index [n], source [n],
 * interested / scripted [n][W] bitmasks with W = mls_words_per_row(n_nodes) (words past ceil(N/32) are zero). */
int mls_episode_sample(const MlsEpisodeSampler* sampler, int32_t n_nodes, const int32_t* slot, const int32_t* episode_no,
                       int32_t n, int32_t* graph_index, int32_t* source, uint32_t* interested, uint32_t* scripted,
                       void* stream);

/* ===== Q-network forward + action selection ============================================
 * Replaces graph_env/env/utils/networks/{common.py:6-64, dgn_r.py:82-129, l_dgn.py:92-151,
 * hl_dgn.py:82-119} (and the PyG / tianshou ops they call) and tianshou
 * DQNPolicy.forward / exploration_noise as driven by
 * graph_env/env/utils/policies/multi_agent_managers/shared_policy.py:81-183. */

enum MlsNetKind { MLS_NET_DGN_R = 0, MLS_NET_L_DGN = 1, MLS_NET_HL_DGN = 2 };
enum MlsPool { MLS_POOL_MEAN = 0, MLS_POOL_ADD = 1, MLS_POOL_MAX = 2 };
enum MlsPrecision { MLS_PREC_FP32 = 0, MLS_PREC_BF16 = 1 };

typedef struct MlsNetDesc {
  int32_t kind;       /* enum MlsNetKind                                                  */
  int32_t n_nodes;    /* agents_num                                                       */
  int32_t hidden;     /* hidden_dim (128)                                                 */
  int32_t heads;      /* num_heads (4)                                                    */
  int32_t input_dim;  /* 5                                                                */
  int32_t pool;       /* enum MlsPool (HL-DGN aggregator)                                 */
  int32_t precision;  /* enum MlsPrecision                                                */
  int32_t head_hidden;/* dueling hidden size (128), two hidden layers                     */
} MlsNetDesc;

/* fp32 parameters exactly as in the reference state_dict ([out, in] row major). */
typedef struct MlsNetWeights {
  const float *enc_w0, *enc_b0, *enc_w1, *enc_b1;      /* encoder.model.{0,2}             */
  /* GATv2 (L-DGN, HL-DGN): convK.{lin_l,lin_r}.{weight,bias}, convK.att [H*C], convK.bias [H*C]
   * Transformer (DGN-R):   convK.{lin_query,lin_key,lin_value}.{weight,bias}              */
  const float *c1_wa, *c1_ba, *c1_wb, *c1_bb, *c1_wc, *c1_bc, *c1_att, *c1_bias;
  const float *c2_wa, *c2_ba, *c2_wb, *c2_bb, *c2_wc, *c2_bc, *c2_att, *c2_bias;
  const float *q_w0, *q_b0, *q_w1, *q_b1, *q_w2, *q_b2; /* Q.model.{0,2,4}                 */
  const float *v_w0, *v_b0, *v_w1, *v_b1, *v_w2, *v_b2; /* V.model.{0,2,4}                 */
  /* network built without dueling_param (l_dgn.py:88-90,149; dgn_r.py, hl_dgn.py alike): q = out_linear(latent);
   * out_w [2][latent], out_b [2]; the Q / V pointers are then ignored (may be NULL).  NULL: dueling heads. */
  const float *out_w, *out_b;
} MlsNetWeights;

typedef struct MlsForwardArgs {
  const float* obs;          /* graph g starts at obs + g*obs_stride; N rows of 8 floats     */
  int64_t obs_stride;        /* floats: 8N for an obs matrix batch, 8N+1 for agent-obs rows  */
  int32_t n_graphs;
  int32_t ctrl_mode;         /* 0: ctrl_mask[g][N] (q/act are [g][N][..]); 1: one controlling
                                node per graph = clamp(obs[g][8N], 0, N-1) (common.py:63), q is [g][2] */
  const uint8_t* ctrl_mask;  /* mode 0 */
  float* q;                  /* out */
  int8_t* act;               /* out, NULL ok: greedy / epsilon-greedy action, -1 where not controlling */
  float eps;                 /* exploration rate (tianshou DQNPolicy.exploration_noise)      */
  int32_t flags;             /* MLS_FWD_* bits                                               */
  uint64_t philox_seed, philox_offset;
  const double* rand3;       /* optional host-fed uniforms [rows][3] = (u_eps, u_act0, u_act1) */
  void* workspace;           /* mls_dgn_workspace_bytes() bytes                              */
  size_t workspace_bytes;
  /* optional timing hook: cudaEvent_t pair recorded right before / after ONE launch of the
   * kernel class `prof_kernel` (enum MlsProfKernel) in the first chunk of this call */
  void* prof_start;
  void* prof_stop;
  int32_t prof_kernel;
  int32_t pad2_;
  /* optional device-side uint64 added to philox_offset (a round counter the caller bumps on
   * the stream; lets a captured CUDA graph draw fresh exploration noise on every replay) */
  const void* philox_offset_dev;
  /* with MLS_FWD_DISCRETE_FEATURES: device int32, set to the number of node rows whose features were not
   * small non-negative integers (those rows are evaluated with key 0); NULL ok */
  void* feature_errors;
  /* optional topology cache (static graph pools; bf16 precision): graph g of this call has the node positions of
   * pool graph graph_ids[g * graph_id_stride], whose radius_graph lists are in csr_cache (mls_dgn_csr_cache_build);
   * the per-call radius_graph pass is then skipped.  The caller guarantees that obs columns 0..1 of graph g equal
   * the positions the cache was built from.  NULL: lists are rebuilt from obs on every call (dynamic graphs). */
  const int32_t* graph_ids;
  int32_t graph_id_stride;   /* in int32 elements (MLS_EP_STRIDE when pointing at episode[b][MLS_EP_GRAPH]) */
  int32_t csr_cache_graphs;  /* pool size the cache was built for */
  const void* csr_cache;
  /* added to the output-row index that keys the exploration draw (Philox counter = row): a caller that processes a
   * batch in slices passes the slice's first row so that the draws equal those of one full-batch call */
  uint64_t philox_row0;
} MlsForwardArgs;

/* The caller guarantees that obs columns 2..6 (degree, messages transmitted, last action, interested,
 * has-message) hold small non-negative integers -- always true for observations produced by
 * mls_env_reset / mls_env_step (graph.py:263-269): degree < 2^ceil(log2 N), messages < 64, flags 0/1.
 * bf16 precision only: encoder + conv1 projections are then evaluated once per distinct feature key. */
#define MLS_FWD_DISCRETE_FEATURES 1
/* bf16 precision: the workspace already holds the packed bf16 weights (and, with MLS_FWD_DISCRETE_FEATURES, the
 * feature tables) of exactly these parameters, left there by mls_dgn_prepare with the same desc / flags on the same
 * workspace; the forward skips re-packing them (weights only change on an optimiser step). */
#define MLS_FWD_PREPARED 2

enum MlsProfKernel {
  MLS_PROF_NONE = 0,
  MLS_PROF_PROJ1 = 1, /* conv1 projection GEMM (first weight tensor)                         */
  MLS_PROF_PROJ2 = 2, /* conv2 projection GEMM (first weight tensor)                         */
  MLS_PROF_EDGE1 = 3, /* conv1 edge softmax/aggregate                                        */
  MLS_PROF_EDGE2 = 4, /* conv2 edge softmax/aggregate                                        */
  MLS_PROF_HEAD0 = 5  /* first dueling-head layer (Q)                                        */
};

size_t mls_dgn_workspace_bytes(const MlsNetDesc* desc, int32_t n_graphs);
/* graphs processed per internal pass (kernel launches cover this many graphs at a time). */
int mls_dgn_chunk_graphs(const MlsNetDesc* desc, int32_t n_graphs);
int mls_dgn_forward(const MlsNetDesc* desc, const MlsNetWeights* w, const MlsForwardArgs* args,
                    void* stream);
/* Pack the parameters into the workspace (bf16 weight matrices, stacked biases, feature tables when flags has
 * MLS_FWD_DISCRETE_FEATURES) for later mls_dgn_forward calls with MLS_FWD_PREPARED.  The packed region's layout does
 * not depend on the number of graphs.  fp32 precision: no-op. */
int mls_dgn_prepare(const MlsNetDesc* desc, const MlsNetWeights* w, int32_t flags, void* workspace,
                    size_t workspace_bytes, void* stream);
/* Topology cache of a static graph pool: radius_graph(pos, r=0.2, loop=False, max_num_neighbors=32)
 * (networks/common.py:47-48) of every pool graph, built once.  pos_obs: graph k's node i has its position at
 * pos_obs[k*obs_stride + i*8 + {0,1}] (fp32, the values the environment writes into obs columns 0..1). */
size_t mls_dgn_csr_cache_bytes(const MlsNetDesc* desc, int32_t n_pool_graphs);
int mls_dgn_csr_cache_build(const MlsNetDesc* desc, const float* pos_obs, int64_t obs_stride,
                            int32_t n_pool_graphs, void* cache, size_t cache_bytes, void* stream);

/* ===== training step (data-parallel DQN) ================================================
 * Replaces, for the batched path, the transition bookkeeping of
 * graph_env/env/utils/collectors/multi_agent_collector.py:240-308 (per-(env, agent) sub-buffers, a transition is
 * completed by the agent's next observation), tianshou's compute_nstep_return as called by DQNPolicy.process_fn
 * (estimation_step / discount_factor, l_dgn.py:69-76) and torch.optim.Adam (l_dgn.py:66).  The loss and the
 * backward pass are host-side torch autograd (melissa_b200/networks/autograd.py); the gradient all-reduce is NCCL
 * over one flat fp32 buffer (melissa_b200/data_parallel.py). */

/* Observation rows (8 fp32 per node, graph.py:254-271) <-> 12-byte packed nodes {float x, y; uint32 w}:
 * w bits 0..16 = feature key (has_message | interested << 1 | action << 2 | messages << 3 | degree << 9), bit 31 = dm.
 * Lossless for observations produced by mls_env_reset / mls_env_step; rows whose feature columns are not the small
 * integers the environment writes are counted in *errors (device int32, NULL ok) and packed with w = 0. */
#define MLS_PACKED_NODE_BYTES 12
int mls_obs_pack(const float* obs /*[rows][8]*/, int64_t n_node_rows, void* packed, int32_t* errors, void* stream);
/* out row m = frame src_frame[m] (NULL: m) of n_nodes packed nodes expanded to 8 floats each; with `agent`
 * (device int32 [n_frames]) column 8*n_nodes receives the controlling index (the reference's agent observation). */
int mls_obs_unpack(const void* packed, const int64_t* src_frame, const int32_t* agent, int32_t n_nodes,
                   int64_t n_frames, int64_t out_stride /*floats*/, float* out, void* stream);

/* n-step returns over the replay ring rew / flags [ring_rounds][n_episodes][n_nodes] (flags bit 0: the agent acted
 * in that round, bit 1: terminated after it).  Sample m = (round_index, episode, agent):
 *   returns[m]    = sum_{k<K} gamma^k rew[(round+k) % ring][episode][agent], K = min(n_step, steps to termination),
 *                   accumulated in fp64
 *   boot_round[m] = ring round of the bootstrap observation when the chain is alive after n_step steps, else -1
 *   boot_gamma[m] = gamma^n_step
 * The caller samples only transitions whose n-step window and bootstrap observation (round + n_step) are already
 * stored, so that round must not have been overwritten either: ring_rounds > n_step. */
int mls_nstep_returns(const double* rew, const uint8_t* flags, int32_t ring_rounds, int64_t n_episodes,
                      int32_t n_nodes, const int32_t* round_index, const int32_t* episode, const int32_t* agent,
                      int32_t n_samples, int32_t n_step, double gamma, float* returns, int32_t* boot_round,
                      float* boot_gamma, void* stream);

/* One torch.optim.Adam step (amsgrad = False) over flat fp32 buffers; grad is multiplied by grad_scale first
 * (1 / world size after the NCCL sum).  step counts from 1. */
int mls_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                  void* stream);

/* ---- training forward / backward of the GATv2 edge phase on per-sample edge lists (melissa_b200/csrc/train_gatv2.cu).
 * Replaces, for the gradient step, the edge phase of torch_geometric.nn.GATv2Conv as called by
 * graph_env/env/utils/networks/l_dgn.py:125,133 (gather, leaky_relu(x_l[j] + x_r[i]) . att, softmax over the
 * incoming edges, weighted sum) and its autograd.  Dense projections stay with the caller. */

/* Capacity of one edge list (self loop + 32 neighbours, rounded up). */
int mls_train_list_capacity(void);
/* Per sampled agent observation (rows of 8 * n_nodes + 1 floats, last column = controlling index): the nodes the
 * controlling node reads, S1 = {c} + radius neighbours (torch_cluster.radius_graph rule, networks/common.py:48), as
 * consecutive "slots" starting at slot_base[sample], and for every slot its source rows (self first).
 *   mode 0: s1_cnt[sample] = |S1|            (caller: slot_base = exclusive prefix sum)
 *   mode 1: tgt_row[slot] = sample * n_nodes + node, src_row[slot][capacity], src_cnt[slot]  (row = sample * n_nodes + node);
 *           used[row] = 1 (optional, caller-zeroed bytes [n_samples * n_nodes]) for every node row that is a source
 *   mode 2: the lists of EVERY node (HL-DGN pools over all of them): slot = sample * n_nodes + node, slot_base unused */
int mls_train_lists(const float* obs_rows, int64_t row_stride, int32_t n_samples, int32_t n_nodes, float r2, int32_t mode,
                    int32_t* s1_cnt, const int64_t* slot_base, int32_t* tgt_row, int32_t* src_row, int32_t* src_cnt,
                    uint8_t* used, void* stream);
/* out[t][heads * 128] = sum_e alpha[t][e][h] * xl[src_row[t][e]], alpha = softmax_e(<att_h, leaky_relu(xl[src] + xr[tgt_row[t]], 0.2)>)
 * (exp(e - max) / (sum + 1e-16)); tgt_row[t] < 0: zeros.  fp32. */
int mls_gatv2_edge_fwd(const float* xl, int64_t ldl, const float* xr, int64_t ldr, const float* att, const int32_t* tgt_row,
                       const int32_t* src_row, const int32_t* src_cnt, int32_t n_targets, int32_t heads, float* out,
                       float* alpha, void* stream);
/* Gradients of the above: d_xl [source rows][heads * 128] (accumulated atomically: zero it first), d_xr [target rows]
 * [heads * 128] (rows of real targets are overwritten), d_att_part [mls_gatv2_edge_bwd_blocks(n_targets)][heads * 128]
 * (per-block partial sums of d att: the caller adds them up). */
int mls_gatv2_edge_bwd_blocks(int32_t n_targets);
int mls_gatv2_edge_bwd(const float* xl, int64_t ldl, const float* xr, int64_t ldr, const float* att, const int32_t* tgt_row,
                       const int32_t* src_row, const int32_t* src_cnt, int32_t n_targets, int32_t heads, const float* alpha,
                       const float* dout, float* d_xl, float* d_xr, float* d_att_part, void* stream);

/* The same for torch_geometric.nn.TransformerConv(root_weight=False, beta=False) (dgn_r.py:105,113): logit = <q[tgt], k[src]> /
 * sqrt(128), out = sum_e alpha_e v[src]; no self loop (the first entry of every list -- the node itself -- is skipped).
 * k, v share the row stride lds.  Backward: d_k, d_v accumulated atomically (zero them first), d_q rows of real targets
 * overwritten. */
int mls_transformer_edge_fwd(const float* k, const float* v, int64_t lds, const float* q, int64_t ldq, const int32_t* tgt_row,
                             const int32_t* src_row, const int32_t* src_cnt, int32_t n_targets, int32_t heads, float* out,
                             float* alpha, void* stream);
int mls_transformer_edge_bwd(const float* k, const float* v, int64_t lds, const float* q, int64_t ldq, const int32_t* tgt_row,
                             const int32_t* src_row, const int32_t* src_cnt, int32_t n_targets, int32_t heads,
                             const float* alpha, const float* dout, float* d_k, float* d_v, float* d_q, void* stream);

/* ---- bf16 training precision of the dense layers (melissa_b200/csrc/train_linear.cu; DGNBase.set_train_precision("bf16")).
 * torch.nn.Linear forward and backward with bf16 operands, fp32 accumulation on the tcgen05 GEMM and fp32 everywhere else
 * (fp32 master weights, fp32 activations between layers).  x [rows][in] (row stride ldx), W [out][in] contiguous:
 *   y  = fp32acc(bf16(x) . bf16(W)^T) + b       (b added in fp32 in the GEMM epilogue; b NULL: none)
 *   dx = fp32acc(bf16(dy) . bf16(W))            (dx NULL: not computed)
 *   dW = fp32acc(bf16(dy)^T . bf16(x))
 *   db = sum over rows of dy in fp32, from the unrounded dy      (db NULL: not computed)
 * No atomics: the results are bitwise reproducible.  rows = 0 launches nothing; the backward then writes dW = 0, db = 0.
 * The caller provides scratch of mls_linear_bf16_workspace_bytes(rows, in, out) bytes on a 256-byte boundary (NULL ok
 * when rows = 0); the library allocates nothing. */
size_t mls_linear_bf16_workspace_bytes(int64_t rows, int32_t in, int32_t out);
int mls_linear_bf16_fwd(const float* x, int64_t ldx, const float* w, const float* b, int64_t rows, int32_t in, int32_t out,
                        float* y, int64_t ldy, void* workspace, size_t workspace_bytes, void* stream);
int mls_linear_bf16_bwd(const float* x, int64_t ldx, const float* w, const float* dy, int64_t lddy, int64_t rows, int32_t in,
                        int32_t out, float* dx, int64_t lddx, float* dw, float* db, void* workspace, size_t workspace_bytes,
                        void* stream);

/* ---- prioritized replay (melissa_b200/csrc/replay_per.cu).  Replaces tianshou PrioritizedReplayBuffer's numpy
 * SegmentTree (init_weight / sample_indices / get_weight / update_weight) for the device replay ring.
 * One fp64 sum tree per ring slot over its L = n_episodes * n_nodes cells (leaf = cell episode * N + agent, holding
 * p^alpha; 0 where the agent did not act), fanout 32, levels stored leaves first and root last; the trees of a ring
 * are [ring_rounds][mls_per_tree_size(L)] doubles.  max_prio / min_prio are device doubles (tianshou starts both at 1). */

/* fp64 nodes of one slot's tree over n_cells leaves (leaves + internal levels + root); -1 if n_cells < 1. */
int64_t mls_per_tree_size(int64_t n_cells);
/* Round build: every leaf of `tree` (one slot) = (*max_prio)^alpha where flags bit 0 (acted) is set, else 0; then every
 * internal level.  The slot's root is the round's total priority. */
int mls_per_build(const uint8_t* flags /*[L]*/, int64_t n_episodes, int32_t n_nodes, const double* max_prio, double alpha,
                  double* tree, void* stream);
/* Proportional sampling, one sample per u[m] in [0, 1).  The usable slots are (first_slot + k) % ring_rounds for
 * k < n_slots, oldest first, their leaves concatenated in that order; with S_i the inclusive prefix sums, T their total and
 * v = u * T the sample is the leaf min{i : leaf_i > 0 and S_i >= v}, or the last positive leaf if v passes it.  A leaf of
 * priority 0 is never returned (if the usable slots hold none that is positive: slot first_slot, cell 0, leaf 0).
 * -> round_index (ring slot), episode, agent; leaf (NULL ok) = the leaf's value. */
int mls_per_sample(const double* trees, int32_t ring_rounds, int64_t n_episodes, int32_t n_nodes, int32_t first_slot,
                   int32_t n_slots, const double* u, int32_t n_samples, int32_t* round_index, int32_t* episode,
                   int32_t* agent, double* leaf, void* stream);
/* Priority update after a learning step: leaf (round_index[m], episode[m], agent[m]) = (|td[m]| + eps)^alpha, the last
 * occurrence of a leaf in the batch wins; its ancestors are recomputed from their children level by level (no atomics:
 * the tree stays a deterministic function of its leaves); *max_prio / *min_prio take the max / min of |td| + eps.
 * Samples outside the ring are ignored. */
int mls_per_update(double* trees, int32_t ring_rounds, int64_t n_episodes, int32_t n_nodes, const int32_t* round_index,
                   const int32_t* episode, const int32_t* agent, const float* td, int32_t n_samples, double alpha,
                   double eps, double* max_prio, double* min_prio, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MELISSA_B200_H */
