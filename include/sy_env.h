/*
 * sy_env.h -- C ABI of the B200-native batched Scotland Yard environment (libsy_env.so).
 *
 * This is the drop-in boundary for the reference's environment hot path.  The reference has
 * no FFI of its own (it is pure Python); the entry points below are what a binding for
 *   /root/reference/src/environment/yard.py        CustomEnvironment.reset / step / observations
 *   /root/reference/src/environment/action_mask.py compute_action_mask
 *   /root/reference/src/environment/reward_calculator.py RewardCalculator
 *   /root/reference/src/environment/pathfinding.py Pathfinder.get_distance
 * would call (see INTEGRATION.md for the ctypes stub a reference maintainer would add).
 *
 * Conventions
 *   - plain C, no torch / CUDA types in signatures; `sy_stream_t` is a `cudaStream_t` passed as void*.
 *   - every function returns SY_OK (0) or an error code; `sy_last_error()` gives the text
 *     (thread-local).  Nothing throws across the ABI.  Invalid *actions* are data, not errors:
 *     they mean "stay" exactly as in yard.py:171-178,223-229.
 *   - ownership: the CALLER owns every state / observation / output buffer (device memory, e.g.
 *     torch tensors) and passes raw pointers; the library owns only its opaque handle and the
 *     per-graph tables it builds in `sy_load_graphs` (dense weights, all-pairs distances, CSR).
 *   - all launches are asynchronous on the given stream; no host synchronisation inside
 *     `sy_step` / `sy_reset` / `sy_sample_actions`.
 *   - shapes: B envs on this device, N nodes, P police, A = P + 1 agents (agent 0 = MrX,
 *     agent 1+k = Police k, as yard.py:54-56), G graphs in the pool.
 */
#ifndef SY_ENV_H
#define SY_ENV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SY_ABI_VERSION 4
#define SY_NUM_REWARD_WEIGHTS 11 /* order = REWARD_WEIGHT_NAMES, src/reward_net.py:5-17 */
#define SY_MAX_AGENTS 16
#define SY_NUM_STATS 16
#define SY_MAX_COPY_SEGMENTS 8
#define SY_DEFAULT_ACTION (-1) /* yard.py:16 ; for police identical to `None` (yard.py:210-215) */

enum {
  SY_OK = 0,
  SY_ERR_INVALID_ARGUMENT = 1,
  SY_ERR_CUDA = 2,
  SY_ERR_STATE = 3 /* call order violated, e.g. step before load_graphs */
};

enum { SY_REWARD_FP64 = 0, SY_REWARD_FP32 = 1 };
enum { SY_STATUS_TERMINATED = 1, SY_STATUS_TRUNCATED = 2, SY_STATUS_FROZEN = 4 }; /* done = any bit */
enum { SY_WINNER_NONE = 0, SY_WINNER_MRX = 1, SY_WINNER_POLICE = 2 };

/* indices into the int64 statistics vector (see sy_stats); summed over ranks by the host */
enum {
  SY_STAT_ENV_STEPS = 0,
  SY_STAT_EPISODES = 1,
  SY_STAT_MRX_WINS = 2,
  SY_STAT_POLICE_WINS = 3, /* captures, reward_calculator.py:63-67 */
  SY_STAT_TRUNCATIONS = 4, /* timestep > max_timestep, reward_calculator.py:68-74 */
  SY_STAT_OUT_OF_MONEY = 5, /* reward_calculator.py:75-79 */
  SY_STAT_SUM_EPISODE_LENGTH = 6,
  SY_STAT_SUM_BUDGET_SPENT = 7, /* over all steps (edge weight + toll of every police move) */
  /* the aggregates of src/eval/metrics.py:AggregatedMetrics (MetricsTracker.get_aggregated_metrics, :168-232) */
  SY_STAT_SUM_SQ_EPISODE_LENGTH = 8,
  SY_STAT_SUM_LENGTH_POLICE_WINS = 9, /* -> mean_time_to_catch */
  SY_STAT_SUM_LENGTH_MRX_WINS = 10,   /* -> mean_survival_time */
  SY_STAT_SUM_EPISODE_BUDGET_SPENT = 11, /* budget spent inside FINISHED episodes -> mean_budget_spent / efficiency */
  SY_STAT_POLICE_MOVES = 12,             /* over all steps; x toll = tolls paid */
  /* belief quality at reveal steps (src/eval/belief_quality.py:8-11 via metrics.py:127-147): cross-entropy of the
   * predicted belief at MrX's true node, scored before the reveal collapses the map; Q24 fixed point (value * 2^24,
   * integer sums are order-independent).  Counted while config.belief == SY_BELIEF_SCORED and statistics are on
   * (scoring costs the observe kernel ~4 us per step at 65 536 envs, hence opt-in). */
  SY_STAT_REVEALS = 13,
  SY_STAT_SUM_BELIEF_CE_Q24 = 14,   /* -> mean_belief_ce */
  SY_STAT_SUM_SQ_BELIEF_CE_Q24 = 15 /* -> belief_ce_std */
};

#define SY_BELIEF_SCORED 2

typedef void* sy_stream_t;
typedef struct SyEnv SyEnv;

/* Replaces the constructor arguments of CustomEnvironment (yard.py:18-28) plus the knobs the
 * reference only has as ablation YAML (src/configs/ablation/mechanism.yaml:1-26). */
typedef struct SyConfig {
  int32_t struct_bytes;    /* = sizeof(SyConfig); ABI guard */
  int32_t device;          /* CUDA ordinal */
  int32_t num_envs;        /* B: envs held by THIS handle (one shard of the global batch) */
  int32_t num_nodes;       /* N  (graph_nodes) */
  int32_t num_police;      /* P  (number_of_agents, yard.py:33) */
  int32_t agent_money;     /* yard.py:42,117-119 */
  int32_t mrx_money;       /* MAX_MONEY_LIMIT = 1000, yard.py:11 */
  int32_t max_timestep;    /* 250, reward_calculator.py:68; in [0, SY_MAX_TIMESTEP] */
  int32_t reveal_interval; /* 0 = MrX always visible (reference behaviour) */
  int32_t toll;            /* 0 = reference behaviour; else legality and police charge use w + toll; in [0, SY_MAX_TOLL] */
  int32_t belief;          /* 0 off | 1 maintain belief_map | SY_BELIEF_SCORED (2): also score it at reveal steps */
  int32_t reward_mode;     /* SY_REWARD_FP64 (python-float weights) | SY_REWARD_FP32 (0-dim fp32 tensors) */
  int32_t auto_reset;      /* 0/1: same-step auto-reset of finished envs (Philox start nodes) */
  int32_t resample_graph;  /* 0/1: on (auto-)reset draw graph_id uniformly from the pool */
  int64_t env_offset;      /* global index of env 0: keeps Philox streams shard-invariant */
  uint64_t seed;
  double reward_weights[SY_NUM_REWARD_WEIGHTS];
  /* Robustness hook of src/eval/ood_eval.py:191-234 (RobustnessWrapper.reveal_skip_prob, and `reveal_probability`
   * of src/configs/ablation/belief.yaml as 1 - p): every scheduled reveal is skipped with this probability, one
   * Philox(seed; env, episode, timestep) Bernoulli draw per env and reveal step.  0 = every scheduled reveal happens
   * (bit-identical to a library without the hook). */
  float reveal_skip_prob;
  int32_t reserved0;
} SyConfig;
/* Bounds sy_create enforces (sy_set_group_tolls / sy_set_group_rules hold groups to the same ones).
 * SY_MAX_TIMESTEP: an episode lasts at most max_timestep + 2 steps (the visit counters are incremented before the
 * timeout test), so a police that never moves counts at most 65 535 visits, exactly what the u16 counters hold.
 * SY_MAX_TOLL (below): with edge weights <= 255, w + toll and a step's police charges stay far inside int32.
 * The episode statistics sum the squared lengths and the budget spent per episode (up to 15 x (2^31 - 1)) in 64 bits. */
#define SY_MAX_TIMESTEP 65533

/* Every pointer struct below starts with `struct_bytes` = sizeof(the struct): the library rejects a struct of another
 * size with SY_ERR_INVALID_ARGUMENT instead of reading past the caller's memory (a binding written against an older
 * header would otherwise hand the kernels garbage pointers). */

/* Per-env state, device pointers, caller-owned (yard.py:111-127 state, batched).
 * Absent agents: an env whose mechanism group plays with fewer police than the config (sy_set_group_rules, P_g <
 * num_police) keeps the [B, A, ...] layout; its agents P_g + 1 .. A - 1 are absent and carry exactly these values:
 * pos -1, money 0, agent_budget 0.0f, reward (and reward64) 0.0, terminated / truncated / done equal to the env's own
 * flags, an all-zero action_mask row and node_features column (both dtypes); sy_sample_actions and the in-kernel
 * action draws give them -1, their actions are ignored whatever they hold, and their init_pos entries (sy_reset) are
 * ignored and come back as -1. */
typedef struct SyState {
  uint64_t struct_bytes; /* = sizeof(SyState) */
  int32_t* pos;      /* [B, A]  MrX_pos + police_positions (-1: absent agent, see above) */
  int32_t* money;    /* [B, A]  agents_money (0: absent agent) */
  int32_t* timestep; /* [B] */
  int32_t* graph_id; /* [B] index into the graph pool */
  int32_t* episode;  /* [B] episodes started (Philox counter) */
  uint8_t* done;     /* [B] 1 = finished and frozen until reset (only without auto_reset) */
  uint16_t* visits;  /* [B, N] node_visit_counts (yard.py:59,244-245) */
  float* belief;     /* [B, N] belief_map, may be NULL when config.belief == 0 */
  const uint8_t* belief_hint; /* [B, N] or NULL: observation hint of ParticleBeliefTracker.update (belief_module.py:
                                 102-106), non-zero = candidate node: after the propagation the belief of node j is
                                 multiplied by 0.1 + 0.9 * (hint[j] != 0) before it is normalised.  Read by sy_step only;
                                 envs whose row is all zero are not re-weighted (`if observation_hint:` is False) */
} SyState;

/* Dynamic observation tensors written every reset/step (yard.py:271-335).  Static graph
 * tensors (adjacency_matrix, edge_index, edge_features) are per-graph and are built once by
 * the host from the same CSR; belief_map is SyState.belief; agent_position is SyState.pos.
 * Absent agents (see SyState) have all-zero action_mask rows and node_features columns and agent_budget 0.0f. */
typedef struct SyObs {
  uint64_t struct_bytes; /* = sizeof(SyObs) */
  uint8_t* action_mask;  /* [B, A, N] bool */
  float* node_features;  /* [B, N, A] one-hot of positions, column 0 = MrX (blank while hidden) */
  float* agent_budget;   /* [B, A]  yard.py:329-331 */
  int32_t* mrx_revealed; /* [B] MrX node if visible this step else -1 */
  uint8_t* node_features_u8; /* [B, N, A] or NULL.  Non-NULL: the one-hot is written here as bytes INSTEAD of the float32
                                array (node_features may then be NULL): exact, and 3 N A fewer bytes per env-step */
} SyObs;

/* Step results (reward_calculator.py:26-92). */
typedef struct SyOut {
  uint64_t struct_bytes; /* = sizeof(SyOut) */
  float* reward;       /* [B, A] */
  double* reward64;    /* [B, A] or NULL: the float64 value before the float32 cast (fp64 mode) */
  uint8_t* terminated; /* [B, A] */
  uint8_t* truncated;  /* [B, A] */
  uint8_t* done;       /* [B, A] terminated | truncated */
  int8_t* winner;      /* [B]   SY_WINNER_* (env.current_winner, yard.py:250) */
  int64_t* stats;      /* non-NULL: collect episode statistics (accumulated inside the library; read with sy_stats) */
  uint8_t* status;     /* [B] or NULL: the three flag arrays in one byte per env -- SY_STATUS_* bits (every agent of an env
                          carries the same flags, reward_calculator.py:63-79) */
} SyOut;

int sy_abi_version(void);
const char* sy_last_error(void);
/* number of CUDA kernels this library has launched in this process (for bench `gpu_launches`) */
int64_t sy_launch_count(void);

/* replaces CustomEnvironment.__init__ (yard.py:18-78) */
int sy_create(const SyConfig* config, SyEnv** out_env);
void sy_destroy(SyEnv* env);
/* Tuning knobs of a handle (results are identical for every setting -- tests/test_gpu_fullsize.py runs the BASELINE
 * configs through each of them; bench.py records what it used; measurements in DESIGN.md section 4c).
 *   SY_OPT_STEP_KERNEL  SY_STEP_AUTO (default): batches whose 32-env tiles fit one wave of the fused kernel's grid
 *                       (<= ~9 500 envs) take SY_STEP_FUSED, larger ones SY_STEP_TWO_KERNELS.
 *                       SY_STEP_FUSED: sy_step is ONE persistent kernel -- dynamics, belief propagation and a bulk-store
 *                       (cp.async.bulk / TMA) observation stream as three warp-specialised roles, software-pipelined
 *                       over the tiles of a CTA; in sy_rollout_random* its dynamics warps also draw the next step's
 *                       actions.  Needs 16-byte aligned observation buffers and a belief map of <= ~400 nodes (else the
 *                       call falls back to two kernels).  SY_STEP_TWO_KERNELS: dynamics kernel, then observation kernel.
 *                       (With the default SY_OPT_LAGGED_KERNEL the random rollouts of such batches take the lagged
 *                       kernels instead; an explicit SY_STEP_FUSED keeps the fused kernel there too.)
 *   SY_OPT_WRITER_PATH  writers of the two-kernel path's observation kernel: SY_WRITER_LSU (default) = 16-byte
 *                       streaming stores; SY_WRITER_BULK = zero-page bulk fill + chunk images + bulk stores.
 *   SY_OPT_NF_FILL      0 (default).  1: split step for batches of >= 8192 envs with float32 node_features: the zero
 *                       fill of node_features (63 % of a step's bytes, independent of the state) is handed to the TMA
 *                       engine by its own small kernel NEXT TO the dynamics kernel (second stream), then the belief
 *                       propagation and the writers of the ones run as two concurrent kernels; all joined on the
 *                       caller's stream before sy_step returns (events; capturable).  Measured slower (DESIGN.md 4c).
 *   SY_OPT_LAGGED_KERNEL SY_LAGGED_AUTO (default): a deferred step with pending observations is ONE launch
 *                       (sy_step_lagged_kernel: the pending observation roles + the dynamics warps of the next step in
 *                       the same CTA) and sy_rollout_random* step deferred WHEN the batch's 32-env tiles fit one wave of
 *                       that kernel (<= ~9 500 envs): a step then costs max(dynamics, observations) instead of their
 *                       sum (c2: 11.8 -> 8.8 us per step).  SY_LAGGED_ON: at every batch size (measured slower beyond one
 *                       wave, DESIGN.md 4c).  SY_LAGGED_OFF: pending observations and dynamics as two launches, rollouts
 *                       step plainly.
 *   SY_OPT_TAIL_SPLIT   1 (default): when the observation kernel's grid ends in a partly filled wave, the tiles of that
 *                       wave are cut into 2 or 4 parts (one CTA each) so the wave is full and short; applies to the
 *                       warp-per-env belief path (large N).  0: always one CTA per 32-env tile.
 *   SY_OPT_ROLLOUT_KERNEL 1 (default): where the lagged kernel is in use and the batch is at most one CTA per SM
 *                       (<= ~4 700 envs), sy_rollout_random* run the whole rollout as ONE launch
 *                       (sy_rollout_lagged_kernel: a CTA owns its tile for all steps; envs are independent, so nothing is
 *                       synchronised across CTAs).  0: one launch per step.
 *   SY_OPT_PDL          0 (default).  1: the dynamics and observation kernels of the two-launch path are launched with
 *                       programmatic stream serialisation (griddepcontrol): a kernel's CTAs may be scheduled, and run their
 *                       state-independent prologue, while the previous kernel of the stream drains.  Measured: c3 sy_step
 *                       0.1341 -> 0.1321 ms, replayed graph 0.1292 -> 0.1287; c4 and 16 384-env batches slower. */
enum { SY_OPT_WRITER_PATH = 0, SY_OPT_STEP_KERNEL = 1, SY_OPT_NF_FILL = 2, SY_OPT_LAGGED_KERNEL = 3, SY_OPT_TAIL_SPLIT = 4,
       SY_OPT_ROLLOUT_KERNEL = 5, SY_OPT_PDL = 6 };
enum { SY_WRITER_BULK = 0, SY_WRITER_LSU = 1 };
enum { SY_STEP_FUSED = 0, SY_STEP_TWO_KERNELS = 1, SY_STEP_AUTO = 2 };
enum { SY_LAGGED_OFF = 0, SY_LAGGED_ON = 1, SY_LAGGED_AUTO = 2 };
int sy_set_option(SyEnv* env, int32_t option, int32_t value);
/* new Philox key for subsequent (auto-)resets and action sampling (torchrl `set_seed`) */
int sy_set_seed(SyEnv* env, uint64_t seed);

/* Host-built float64 tables so that rewards are bit-identical to NumPy's:
 * exp_neg[d] = np.exp(-d) (reward_calculator.py:186,199,214), coverage[c] = np.exp(-np.log1p(c))
 * (reward_calculator.py:204-205).  HOST pointers; indices past the end read as exp(-inf) = 0
 * (exp_neg) or clamp (coverage). */
int sy_set_reward_tables(SyEnv* env, const double* exp_neg, int32_t n_exp, const double* coverage,
                         int32_t n_cov, sy_stream_t stream);

/* Upload the graph pool as CSR (HOST pointers; every undirected edge appears in both rows,
 * neighbours ascending, weights 1..255) and build on device: the dense weight table
 * (yard.py:404-418), the all-pairs shortest-path table that replaces Pathfinder.get_distance
 * (pathfinding.py:34-137), the move-count table (yard.py:420-472) and 1/deg for the belief.
 * row_ptr [G, N+1] (offsets local to each graph), col / w [G, nnz_stride]. */
int sy_load_graphs(SyEnv* env, int32_t num_graphs, const int32_t* row_ptr, const int32_t* col,
                   const int32_t* w, int32_t nnz_stride, sy_stream_t stream);
/* Sample the whole pool ON THE DEVICE: replaces ConnectedGraph.sample (graph_layout.py:9-80: random recursive tree
 * over a uniform insertion order, extra edges first-fit over a uniform shuffle under the degree cap, weights
 * U{1..max_weight-1}) and the resample-until-the-edge-count-matches loop of CustomEnvironment.__init__/reset
 * (yard.py:67-101: the first sample fixes the count, later ones are redrawn up to 100 times) -- same distribution,
 * Philox streams keyed by (seed; graph_offset + slot, generation, attempt), one warp per pool slot; then the tables of
 * sy_load_graphs are built from the result.  A new `generation` refreshes the pool ("new graph on reset" at scale);
 * with an unchanged shape the tables keep their addresses.  Envs must be reset afterwards.  attempts_host (HOST,
 * [num_graphs], may be NULL) receives the 0-based attempt that produced each slot.  Fails with SY_ERR_STATE and the
 * reference's message when a slot cannot reach the edge count.  num_nodes <= 8192.  Synchronises the stream. */
int sy_generate_graphs(SyEnv* env, int32_t num_graphs, int32_t num_edges, int32_t max_edges_per_node, int32_t max_weight,
                       uint64_t seed, uint32_t generation, uint32_t graph_offset, int32_t* attempts_host,
                       sy_stream_t stream);
/* Edge lists of a device-sampled pool in the reference's order (tree edges, then the extras) = GraphInstance
 * .edge_links / .edges (graph_layout.py:53).  HOST buffers: edge_links int32 [G, max_edges, 2], weights int32
 * [G, max_edges], counts int32 [G]; rows valid up to counts[g].  Synchronises the stream. */
int sy_read_graph_edges(SyEnv* env, int32_t* edge_links, int32_t* weights, int32_t* counts, int32_t max_edges,
                        sy_stream_t stream);
/* copy graph g's tables to HOST buffers (any may be NULL): weights u8 [N, N], apsp u16 [N, N]
 * (0xFFFF = unreachable).  Synchronises the stream.  For tests / get_distance parity. */
int sy_read_graph_tables(SyEnv* env, int32_t g, uint8_t* weights, uint16_t* apsp, sy_stream_t stream);

/* replaces CustomEnvironment.reset (yard.py:80-142) for the envs whose reset_mask byte is
 * non-zero (NULL = all).  init_pos [B, A] / init_graph_id [B] (device, may be NULL) let a caller
 * hand over the reference's own start nodes and graphs; otherwise Philox(seed; env, episode).
 * restart != 0 sets the episode counter of the reset envs to 0, else it is incremented.
 * Observations of every env in the batch are rewritten. */
int sy_reset(SyEnv* env, const uint8_t* reset_mask, const int32_t* init_pos, const int32_t* init_graph_id,
             int32_t restart, const SyState* state, const SyObs* obs, sy_stream_t stream);

/* replaces CustomEnvironment.step (yard.py:144-269) for the whole batch.
 * actions int64 [B, A] (device): target node per agent; -1 = DEFAULT_ACTION / None. */
int sy_step(SyEnv* env, const int64_t* actions, const SyState* state, const SyObs* obs, const SyOut* out,
            sy_stream_t stream);

/* Software-pipelined stepping for policies that read only the compact state (SyState.pos / money, SyObs.agent_budget /
 * mrx_revealed: the random policy, both reference agents' action selection -- gnn_agent.py:45-82 builds its features from
 * positions, mappo_agent.py:87-142 from the budget / position vector).  sy_step_deferred = the dynamics of yard.py:144-269
 * exactly as sy_step (state, rewards, flags, statistics are those of the new state when it completes), but the three
 * dense observation tensors -- action_mask, node_features, belief_map -- of the NEW state are left pending.  The next
 * sy_step_deferred writes them while it runs the following step's dynamics (one launch: the latency-bound dynamics hide
 * under the HBM-bound observation stream of the same 32-env tile), so after every deferred call the dense tensors
 * describe the state BEFORE that call.  sy_flush_observations writes whatever is pending (no-op otherwise); sy_step,
 * sy_step_host*, sy_reset flush implicitly, so mixing the calls is always correct.  Pending observations are written
 * into the SyObs of the call that carries them.  Where the lagged kernel is in use (SY_OPT_LAGGED_KERNEL), sy_rollout_random /
 * sy_rollout_random_dev step deferred and flush once at the end.  sy_observations_pending: 1 while a flush is owed. */
int sy_step_deferred(SyEnv* env, const int64_t* actions, const SyState* state, const SyObs* obs, const SyOut* out,
                     sy_stream_t stream);
int sy_flush_observations(SyEnv* env, const SyState* state, const SyObs* obs, sy_stream_t stream);
int sy_observations_pending(SyEnv* env);

/* HOST pointers (pinned memory recommended) that `sy_step_host` fills; any member may be NULL. */
typedef struct SyHostOut {
  uint64_t struct_bytes; /* = sizeof(SyHostOut) */
  float* reward;       /* [B, A] */
  uint8_t* terminated; /* [B, A] */
  uint8_t* truncated;  /* [B, A] */
  uint8_t* done;       /* [B, A] */
  int8_t* winner;      /* [B] */
  uint8_t* status;     /* [B] compact flags (SyOut.status).  Any member may be NULL = not copied: a host loop that reads
                          `status` instead of the three [B, A] arrays moves 3A - 1 fewer bytes per env over PCIe */
} SyHostOut;

/* Host-buffer form of sy_step, the shape of the reference's own call (yard.py:144: python ints in,
 * python dicts out): copies actions_host [B, A] to the caller's device staging buffer actions_dev,
 * runs the step, copies rewards / flags / winner back into host_out and SYNCHRONISES the stream.
 * Observations stay in the caller's device buffers (SyObs) for a device-side policy. */
int sy_step_host(SyEnv* env, const int64_t* actions_host, int64_t* actions_dev, const SyState* state,
                 const SyObs* obs, const SyOut* out, const SyHostOut* host_out, sy_stream_t stream);

/* int32 wire format of the same three calls: a host-side caller moves half the bytes over PCIe (node ids fit 16 bits).
 * Semantics are identical: -1 = DEFAULT_ACTION / None, anything that is not an affordable neighbour means `stay`. */
int sy_step_i32(SyEnv* env, const int32_t* actions, const SyState* state, const SyObs* obs, const SyOut* out,
                sy_stream_t stream);
/* int16 wire format (num_nodes <= 32767): a quarter of the int64 bytes */
int sy_step_i16(SyEnv* env, const int16_t* actions, const SyState* state, const SyObs* obs, const SyOut* out,
                sy_stream_t stream);
int sy_step_host_i16(SyEnv* env, const int16_t* actions_host, int16_t* actions_dev, const SyState* state,
                     const SyObs* obs, const SyOut* out, const SyHostOut* host_out, sy_stream_t stream);
int sy_sample_actions_i16(SyEnv* env, const SyState* state, uint32_t step_counter, int16_t* actions,
                          sy_stream_t stream);
/* Host loops with overlap (off by default): sy_step_host* then return as soon as the step's RESULTS are in host_out --
 * the observation kernel may still be running on `stream` (everything issued to that stream later is ordered after it)
 * -- and sy_sample_actions_host runs on a library stream right behind the step's dynamics, next to the observation
 * kernel.  A host-side policy that only needs rewards / flags / state therefore works while the observations of the
 * same step are still being written (they never leave the device on this path). */
int sy_set_host_overlap(SyEnv* env, int32_t on);
/* sy_sample_actions + device->host copy + synchronise in one call (a host-side policy stand-in for host loops):
 * bytes_per_action = 8 | 4 | 2 selects the wire format of actions_dev / actions_host. */
int sy_sample_actions_host(SyEnv* env, const SyState* state, uint32_t step_counter, void* actions_dev, void* actions_host,
                           int32_t bytes_per_action, sy_stream_t stream);
/* `num_steps` iterations of { sy_sample_actions_host(step_counter0 + k); sy_step_host*(those HOST actions) } issued from C:
 * the host-buffer loop of a host-side policy (gnn_trainer.py:201-250 with RandomAgent) with every per-step copy and
 * synchronisation of the two calls, and no interpreter between them.  Buffers as in the two calls. */
int sy_host_rollout_random(SyEnv* env, int32_t num_steps, uint32_t step_counter0, void* actions_dev, void* actions_host,
                           int32_t bytes_per_action, const SyState* state, const SyObs* obs, const SyOut* out,
                           const SyHostOut* host_out, sy_stream_t stream);
int sy_step_host_i32(SyEnv* env, const int32_t* actions_host, int32_t* actions_dev, const SyState* state,
                     const SyObs* obs, const SyOut* out, const SyHostOut* host_out, sy_stream_t stream);
int sy_sample_actions_i32(SyEnv* env, const SyState* state, uint32_t step_counter, int32_t* actions,
                          sy_stream_t stream);

/* uniform random valid action per agent (Philox(seed; env, step_counter, agent)); -1 when the
 * agent has no affordable move (gnn_trainer.py:227-229).  The `random policy` of the benchmarks. */
int sy_sample_actions(SyEnv* env, const SyState* state, uint32_t step_counter, int64_t* actions,
                      sy_stream_t stream);

/* Heuristic opponents for the whole batch: an evading MrX and chasing police, the counterpart of the heuristics of
 * src/eval/exploitability.py:122,188 (parity unpinned: that source is not available, the rules below are this library's).
 * One launch; reads the state, SyObs.mrx_revealed, the all-pairs distance table D and the mechanism group rows (toll,
 * police count), and writes actions int64 [B, A].  Notation for env b: toll_b = its group's toll (else config.toll), P_b =
 * its police count (agents past P_b are absent); neighbour j of node u is affordable for money m iff w(u, j) + toll_b <= m
 * (the rule of the step, the mask and the sampler); D[x][y] of 0xFFFF counts as 65 535; police positions are those of
 * the state read (before the step).
 *   random draw   = exactly sy_sample_actions(step_counter) for that (env, agent) (-1 without an affordable neighbour).
 *   exploration   an agent takes the random draw when Philox(env_offset + b, step_counter, 4, agent).x < explore_<side>,
 *                 with explore_<side> = floor(epsilon * 2^32) in [0, 2^32] (2^32: always, 0: never).
 *   SY_HEUR_EVADE (MrX) candidates: its own node and every affordable neighbour no present police occupies; score of c:
 *                 min over present police i of D[c][pos_i]; highest score wins, ties to the own node, then to the lowest
 *                 id.  The own node means "stay".
 *   SY_HEUR_CHASE (police) target = mrx_revealed[b] when >= 0, else the env's last_seen entry; unknown (-1): the random
 *                 draw.  Otherwise: no affordable neighbour -> -1; every affordable neighbour occupied by another present
 *                 police -> the agent's own node (it stays, but acts: "every police skipped" is not triggered); else the
 *                 affordable unoccupied neighbour with the smallest D[j][target], ties to the lowest id.
 *   SY_HEUR_CHASE_BELIEF  as CHASE, but a hidden MrX's target is the first argmax of belief[b, :] (never unknown).  Needs
 *                 config.belief != 0 and SyState.belief, and is refused with SY_ERR_STATE while observations are pending
 *                 (the belief map lags the state after sy_step_deferred).
 *   SY_HEUR_RANDOM  the random draw.  SY_HEUR_NONE  that side's columns of `actions` are left untouched (e.g. written by
 *                 a learned policy before the call: score it against heuristic opponents).
 * Absent agents get -1 from every kind but NONE.  Frozen envs get actions by the same rules (the step ignores them).
 * last_seen: caller-owned DEVICE int32 [B] or NULL.  Per env the call computes ls = rev >= 0 ? rev : (timestep == 0 ? -1 :
 * last_seen[b]) with rev = mrx_revealed[b] and writes it back (whatever the kinds).  It is MrX's last revealed node of the
 * current episode when the call has been made at every step of that episode (a plain step loop, RolloutCollector); fill
 * it with -1 when starting.  NULL: a hidden MrX is never remembered.
 * Preconditions of sy_sample_actions (graphs and reward tables loaded); SY_ERR_STATE while mechanism groups wait for their
 * reset, as the step entry points.  SY_ERR_INVALID_ARGUMENT for a wrong struct_bytes, a kind out of range, a threshold
 * above 2^32, a NULL SyObs.mrx_revealed, or CHASE_BELIEF without a belief map. */
enum { SY_HEUR_NONE = 0, SY_HEUR_RANDOM = 1, SY_HEUR_EVADE = 2, SY_HEUR_CHASE = 3, SY_HEUR_CHASE_BELIEF = 4 };
typedef struct SyHeuristic {
  uint64_t struct_bytes;   /* = sizeof(SyHeuristic) */
  int32_t mrx_kind;        /* SY_HEUR_NONE | SY_HEUR_RANDOM | SY_HEUR_EVADE */
  int32_t police_kind;     /* SY_HEUR_NONE | SY_HEUR_RANDOM | SY_HEUR_CHASE | SY_HEUR_CHASE_BELIEF */
  uint64_t explore_mrx;    /* floor(epsilon_mrx * 2^32), in [0, 2^32] */
  uint64_t explore_police; /* floor(epsilon_police * 2^32), in [0, 2^32] */
  int32_t* last_seen;      /* [B] device or NULL */
} SyHeuristic;
int sy_heuristic_actions(SyEnv* env, const SyHeuristic* h, const SyState* state, const SyObs* obs,
                         uint32_t step_counter, int64_t* actions, sy_stream_t stream);

/* Add the statistics accumulated since the last call to `stats` (device, int64 [SY_NUM_STATS], caller-owned and
 * cumulative) and clear the library's internal accumulators.  Asynchronous on `stream`.  Statistics are collected by
 * sy_step only while SyOut.stats is non-NULL (they are kept in per-tile-group lines inside the library so that the
 * step kernel's atomics do not serialise on one cache line). */
int sy_stats(SyEnv* env, int64_t* stats, sy_stream_t stream);

/* Mechanism groups: one handle evaluates up to SY_MAX_GROUPS mechanisms side by side.  Every env belongs to one group,
 * and a group replaces, for its envs, the config's reward weights (fp32 reward mode uses (float)w), police start budget
 * (agent_money), reveal schedule (reveal_interval, reveal_skip_prob), through sy_set_group_tolls the toll, and through
 * sy_set_group_rules the number of police and the episode horizon (max_timestep), each bounded by the config's.
 * Group membership enters no random stream, so a group equal to the config reproduces a handle without groups bit for
 * bit.  Every step path runs with groups (its GROUPS instantiation) except the split step of SY_OPT_NF_FILL, which acts
 * as off while groups are set (results are the same).  The statistics are also summed per group (sy_group_stats).
 * The library's group buffers are allocated once and updated in place, but a CUDA graph captured before a
 * sy_set_groups call carries the groups of its capture: recapture it after changing the groups. */
#define SY_MAX_GROUPS 1024
typedef struct SyGroup {
  uint64_t struct_bytes; /* = sizeof(SyGroup) */
  double reward_weights[SY_NUM_REWARD_WEIGHTS];
  int32_t agent_money, reveal_interval;
  float reveal_skip_prob;
  int32_t reserved0;
} SyGroup;
/* groups: HOST table [num_groups]; group_id: DEVICE int32 [B], or NULL = (env_offset + b) % num_groups (every group then
 * sees the same graph mix, and a sharded batch is assigned as the unsharded one); num_groups = 0 clears the groups.
 * Validates (the table on the host, the ids with one small kernel + one synchronise of `stream`) and copies both into
 * library-owned memory; a rejected call keeps the previous groups.  The new groups take effect at the next sy_reset of
 * every env (NULL reset_mask, or one with every byte set): until then the step and rollout entry points fail with
 * SY_ERR_STATE (so a state saved under groups cannot be resumed mid-episode: the reset starts new episodes).  Fails with
 * SY_ERR_STATE while observations are pending.  Clears the per-group statistics.  Every group gets the config's toll,
 * num_police and max_timestep. */
int sy_set_groups(SyEnv* env, int32_t num_groups, const SyGroup* groups, const int32_t* group_id, sy_stream_t stream);
/* Per-group tolls: an env pays its group's toll instead of SyConfig.toll -- a move is legal iff w + toll <= budget (MrX and
 * police; action_mask, the random sampler and the mobility term of the rewards follow the same rule), and a police move
 * costs w + toll.  tolls: HOST int32 [num_groups], each in [0, SY_MAX_TOLL] (the bound of SyConfig.toll: with edge
 * weights <= 255, w + toll and the per-step sums of the police charges cannot overflow an int32); num_groups must be the
 * number set by sy_set_groups.
 * A rejected call keeps the previous tolls.  Like sy_set_groups: fails with SY_ERR_STATE while observations are pending
 * (or when no groups are set), and the new tolls take effect at the next sy_reset of every env, which the step and
 * rollout entry points require until then.  A CUDA graph captured before the call must be captured again.  Synchronises
 * `stream`. */
#define SY_MAX_TOLL 1048576
int sy_set_group_tolls(SyEnv* env, int32_t num_groups, const int32_t* tolls, sy_stream_t stream);
/* Per-group police count and episode horizon.  num_police / max_timestep: HOST int32 [num_groups], either may be NULL
 * (= the config's value for every group); num_police[g] in [1, config.num_police], max_timestep[g] in
 * [0, config.max_timestep] (the bounds keep the coverage table, the u16 visit counters and every buffer sized by the
 * handle valid).  Agents 0 .. num_police[g] of an env of group g play exactly as in a handle built with
 * num_police = num_police[g], max_timestep = max_timestep[g] and the group's other fields (start nodes, moves, capture,
 * "every police skipped", rewards in both modes, visits, belief, reveals and statistics, bit for bit; budget spent and
 * police moves count its police only); the timeout is timestep > max_timestep[g].  The other agents are absent (see
 * SyState).  num_groups must be the number set by sy_set_groups; a rejected call keeps the previous values.  Like
 * sy_set_group_tolls: fails with SY_ERR_STATE while observations are pending (or when no groups are set), the new
 * values take effect at the next sy_reset of every env, which the step and rollout entry points require until then,
 * and a CUDA graph captured before the call must be captured again.  Clears nothing else.  Synchronises `stream`. */
int sy_set_group_rules(SyEnv* env, int32_t num_groups, const int32_t* num_police, const int32_t* max_timestep,
                       sy_stream_t stream);
/* Add the per-group statistics accumulated since the last call to `stats` (DEVICE int64 [num_groups, SY_NUM_STATS],
 * caller-owned, cumulative) and clear the accumulators; num_groups must be the number set.  They are collected by the
 * same steps as sy_stats, with the same integer sums, so the sum over groups equals the handle-wide vector. */
int sy_group_stats(SyEnv* env, int32_t num_groups, int64_t* stats, sy_stream_t stream);

/* The path's one collective (SURVEY.md 8(e)): fold the accumulated statistics into `stats_local` (device, int64
 * [SY_NUM_STATS], this rank's cumulative vector, as sy_stats does) and write their sum over all ranks of `nccl_comm`
 * (an `ncclComm_t`, passed as void*) to `stats_global` (device, int64 [SY_NUM_STATS]) with one ncclAllReduce on `stream`
 * (NVLink / NVSwitch on a B200 box).  NCCL is resolved at run time from the host process (libnccl.so.2; SY_NCCL_LIB
 * overrides the name), so the library does not link against it.  Replaces the Python-side aggregation of
 * src/eval/metrics.py:168-232 across workers; student_mechanism_design_b200.sharding.allreduce_stats is the
 * torch.distributed form of the same reduction. */
int sy_allreduce_stats(SyEnv* env, void* nccl_comm, int64_t* stats_local, int64_t* stats_global, sy_stream_t stream);

/* Trajectory recording for rollout loops (gnn_trainer.py:234-250 stores every transition): up to
 * SY_MAX_COPY_SEGMENTS device-to-device copies dst[i] <- src[i] of bytes[i] bytes in ONE kernel launch on `stream`
 * (HOST tables of DEVICE pointers), instead of one copy per stored tensor and step. */
int sy_copy_segments(int32_t num_segments, void* const* dst, const void* const* src, const uint64_t* bytes, sy_stream_t stream);

/* `num_steps` steps of the random-valid policy rollout the reference's trainers start from (gnn_trainer.py:201-250 with
 * RandomAgent, src/agent/random_agent.py:7): per step sy_sample_actions(step_counter0 + k) into `actions` (device,
 * int64 [B, A]) followed by sy_step, issued back to back from C on `stream` (no host work per step beyond the launches;
 * capturable in a CUDA graph).  Buffers hold the state / observation / result of the last step afterwards. */
int sy_rollout_random(SyEnv* env, int32_t num_steps, uint32_t step_counter0, int64_t* actions, const SyState* state,
                      const SyObs* obs, const SyOut* out, sy_stream_t stream);

/* The same with the step counter in DEVICE memory: step k samples with *step_counter_dev + k and the call ends by
 * adding num_steps to it on the stream, so a CUDA graph captured around this call draws fresh actions on every replay
 * (small batches are launch-latency bound: BASELINE config 2 runs ~1.8x faster from a replayed graph). */
int sy_rollout_random_dev(SyEnv* env, int32_t num_steps, uint32_t* step_counter_dev, int64_t* actions,
                          const SyState* state, const SyObs* obs, const SyOut* out, sy_stream_t stream);

/* replaces compute_action_mask (action_mask.py:30-83) for Q queries on dense float64 inputs
 * (device pointers): adj [N,N]; weights [N,N] or NULL (adjacency as unit costs, :99-113);
 * toll_matrix [N,N] or NULL (then toll_scalar is used everywhere, :86-96); cur [Q]; budget [Q];
 * out [Q, N] bool. */
int sy_action_mask_dense(int32_t num_queries, int32_t num_nodes, const double* adjacency,
                         const double* weights, const double* toll_matrix, double toll_scalar,
                         const int32_t* current_node, const double* budget, uint8_t* out_mask,
                         sy_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SY_ENV_H */
