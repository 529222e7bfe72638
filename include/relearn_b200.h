/*
 * relearn_b200.h -- C ABI of the B200-native rollout/update hot path of relearn.
 *
 * This is the drop-in boundary: a Rust `relearn-b200-sys` crate binds exactly these symbols and
 * implements relearn's traits over the opaque handles (see INTEGRATION.md).  Each entry point
 * cites the reference interface it replaces (file:line in edlanglois/relearn).
 *
 * Conventions
 *  - every function returns rl_status; no exception crosses the boundary; rl_last_error() gives
 *    the message of the last failure on that context (thread-local for ctx-less calls).
 *  - handles are opaque, owned by the library, freed by *_destroy.  A handle is not thread safe;
 *    different handles may be used from different threads (mirrors Rust `&mut` exclusivity).
 *  - bulk data lives in device memory owned by the library.  Host pointers are used only for
 *    configs, weights, statistics and explicit read-backs.  `*_dev` arguments are device pointers.
 *  - all work is enqueued on the context's stream; functions that return host scalars synchronise.
 *  - there is no CPU fallback: every compute entry point fails with RL_ERR_CUDA without a GPU.
 *
 * Device layouts (E = lanes/envs on this device, F = features, T = step capacity):
 *   obs      f32 [T][F][E]   feature planes, lane index fastest (coalesced across lanes)
 *   action   u8  [T][E]
 *   reward   f32 [T][E]
 *   succ     u8  [T][E]      RL_CONTINUE / RL_TERMINATE / RL_INTERRUPT / RL_PAD (unused slot)
 *   next_obs f32 [T][F][E]   successor observation, valid only where succ == RL_INTERRUPT
 */
#ifndef RELEARN_B200_H
#define RELEARN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RL_VERSION_MAJOR 0
#define RL_VERSION_MINOR 1

typedef int32_t rl_status;
enum {
    RL_OK = 0,
    RL_ERR_INVALID_ARG = 1,
    RL_ERR_CUDA = 2,
    RL_ERR_UNSUPPORTED = 3,
    RL_ERR_OOM = 4,
    RL_ERR_NCCL = 5,
    /* WriteExperienceError::Full (src/agents/buffers/mod.rs:225-228) */
    RL_ERR_BUFFER_FULL = 6,
    /* OptimizerStepError (src/torch/optimizers/mod.rs:80-94); parameters are restored */
    RL_STEP_NAN_LOSS = 16,
    RL_STEP_NAN_CONSTRAINT = 17,
    RL_STEP_LOSS_NOT_IMPROVING = 18,
    RL_STEP_CONSTRAINT_VIOLATED = 19
};

/* Successor tags (src/envs/mod.rs:257-269) */
enum { RL_CONTINUE = 0, RL_TERMINATE = 1, RL_INTERRUPT = 2, RL_PAD = 255 };

typedef struct rl_ctx rl_ctx;
typedef struct rl_env rl_env;
typedef struct rl_mlp rl_mlp;
typedef struct rl_adam rl_adam;
typedef struct rl_traj rl_traj;
typedef struct rl_tabq rl_tabq;
typedef struct rl_ucb1 rl_ucb1;
typedef struct rl_bts rl_bts;
typedef struct rl_replay rl_replay;
typedef struct rl_grunet rl_grunet;

/* ------------------------------------------------------------------------------------------ */
/* Context                                                                                     */
/* ------------------------------------------------------------------------------------------ */
/* `stream` is a cudaStream_t to enqueue on (e.g. torch's current stream) or NULL to create one. */
rl_status rl_ctx_create(int32_t device, void *stream, rl_ctx **out);
rl_status rl_ctx_destroy(rl_ctx *ctx);
rl_status rl_ctx_synchronize(rl_ctx *ctx);
const char *rl_last_error(rl_ctx *ctx);
const char *rl_status_str(rl_status status);
uint32_t rl_version(void);
int32_t rl_device_count(void);
/* Number of kernels this library has launched on the context since creation. */
uint64_t rl_ctx_launch_count(rl_ctx *ctx);
/* Device properties the host needs for roofline reporting. */
rl_status rl_ctx_device_info(rl_ctx *ctx, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor,
                             uint64_t *total_mem_bytes);

/* Device timers on the context stream (cudaEvent) and a peak-FMA probe, for roofline reporting. */
typedef struct rl_event rl_event;
rl_status rl_event_create(rl_ctx *ctx, rl_event **out);
rl_status rl_event_destroy(rl_event *ev);
rl_status rl_event_record(rl_event *ev);
/* waits for `stop`; ms = device time between the two records */
rl_status rl_event_elapsed_ms(rl_event *start, rl_event *stop, float *ms);
rl_status rl_probe_fp32_tflops(rl_ctx *ctx, double *tflops);

/* Raw device memory for caller-supplied streams of actions / noise and for read-backs. */
rl_status rl_malloc(rl_ctx *ctx, size_t bytes, void **out_dev);
rl_status rl_free(rl_ctx *ctx, void *dev);
rl_status rl_memcpy_h2d(rl_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
rl_status rl_memcpy_d2h(rl_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
rl_status rl_memset(rl_ctx *ctx, void *dst_dev, int32_t value, size_t bytes);
/* Page-locked host memory for weights / statistics that cross the boundary every period. */
rl_status rl_malloc_host(rl_ctx *ctx, size_t bytes, void **out_host);
rl_status rl_free_host(rl_ctx *ctx, void *host);

/* Data-parallel group over NCCL (no reference counterpart: relearn has no collectives;
 * replaces the crossbeam thread fan-out of src/simulation/train.rs:124-158 across GPUs).
 * `unique_id` is the 128-byte ncclUniqueId made by rank 0 and shared by the host. */
#define RL_NCCL_UNIQUE_ID_BYTES 128
rl_status rl_nccl_unique_id(void *out_id128);
rl_status rl_ctx_comm_init(rl_ctx *ctx, const void *unique_id128, int32_t rank, int32_t world_size);
rl_status rl_ctx_comm_info(rl_ctx *ctx, int32_t *rank, int32_t *world_size);
/* Whether the update's reductions run as ONE kernel per pass that sums the partial rows and exchanges the sums
 * with every peer through CUDA-IPC-mapped mailboxes over NVLink (peer_mailboxes = 1; set up by rl_ctx_comm_init
 * on a single node, RL_XREDUCE=nccl disables it) or as reduce + ncclAllReduce (0), and whether any wait for a peer
 * timed out (then the results of that update are invalid).  Synchronises the context stream. */
rl_status rl_ctx_comm_peer_info(rl_ctx *ctx, int32_t *peer_mailboxes, int32_t *timed_out);
/* In-place sum all-reduce of `n` f64 on the context stream (used by the update kernels; exposed
 * for tests). */
rl_status rl_ctx_allreduce_f64(rl_ctx *ctx, double *buf_dev, size_t n);

/* ------------------------------------------------------------------------------------------ */
/* Environments   (BuildEnv::build_env src/envs/builders.rs:17; Environment src/envs/mod.rs:76) */
/* ------------------------------------------------------------------------------------------ */
typedef enum {
    RL_ENV_CARTPOLE = 0,    /* CartPole (+ Visible / LatentStepLimit)  src/envs/cartpole.rs, wrappers/step_limit.rs */
    RL_ENV_CHAIN = 1,       /* Chain                          src/envs/chain.rs */
    RL_ENV_MEMORY_GAME = 2, /* MemoryGame                     src/envs/memory.rs */
    RL_ENV_BANDIT_META = 3, /* MetaEnv<UniformBernoulliBandits> + TrialEpisodeLimit  src/envs/meta.rs, bandits.rs */
    RL_ENV_PARTITION_GAME = 4 /* PartitionGame (no configuration: cfg may be NULL)  src/envs/partition.rs */
} rl_env_kind;

/* CartPoleConfig {PhysicalConstants, EnvironmentParams} (cartpole.rs:157-216) wrapped by
 * VisibleStepLimit (step_limit.rs:97-123).  max_steps_per_episode == 0 means unwrapped. */
typedef struct rl_cartpole_cfg {
    double gravity, mass_cart, mass_pole, length_half_pole, friction_cart, friction_pole, time_step;
    double action_force, max_pos, max_angle, discount_factor;
    uint64_t max_steps_per_episode;
    /* 1 = VisibleStepLimit (the observation gains the `remaining` feature, step_limit.rs:97-223);
     * 0 = LatentStepLimit (same interruption, observation unchanged, step_limit.rs:13-90) */
    uint64_t step_limit_visible;
} rl_cartpole_cfg;
/* Chain (chain.rs:21-45) */
typedef struct rl_chain_cfg { uint64_t size; double discount_factor; } rl_chain_cfg;
/* MemoryGame (memory.rs:24-55) */
typedef struct rl_memory_cfg { uint64_t num_actions, history_len; } rl_memory_cfg;
/* MetaEnv<UniformBernoulliBandits{num_arms}>.wrap(TrialEpisodeLimit{episodes_per_trial})
 * (bandits.rs:128-181, meta.rs:49-203,541-617) */
/* distribution: 0 = UniformBernoulliBandits (means ~ U[0,1], Bernoulli rewards), 1 = OneHotBandits (one arm chosen
 * uniformly pays 1, DeterministicBandit rewards; bandits.rs:187-243) */
typedef struct rl_bandit_meta_cfg { uint64_t num_arms, episodes_per_trial, distribution; } rl_bandit_meta_cfg;

void rl_cartpole_cfg_default(rl_cartpole_cfg *cfg, uint64_t max_steps_per_episode);
void rl_chain_cfg_default(rl_chain_cfg *cfg);

/* EnvStructure (src/envs/mod.rs:165-193) flattened to what the feature encoders need. */
typedef struct rl_env_structure {
    int32_t num_features;     /* FeatureSpace::num_features of the observation space */
    int32_t num_actions;      /* FiniteSpace::size of the action space */
    int32_t num_observations; /* FiniteSpace::size of the observation space, 0 if not finite */
    double reward_lo, reward_hi, discount_factor;
} rl_env_structure;

/* `num_envs` lanes on this device, global lane ids [lane_offset, lane_offset + num_envs): the
 * Philox counter uses the global id so results do not depend on how lanes are sharded. */
rl_status rl_env_create(rl_ctx *ctx, rl_env_kind kind, const void *cfg, uint64_t num_envs,
                        uint64_t lane_offset, uint64_t seed, rl_env **out);
rl_status rl_env_destroy(rl_env *env);
rl_status rl_env_structure_of(rl_env *env, rl_env_structure *out);

/* Noise source = the `&mut Prng` arguments of Environment/Actor.  PHILOX (default): counter-based
 * Philox4x32-10 keyed by (seed; lane, step, stream, draw).  REPLAY: per-lane streams of u32 words
 * consumed sequentially the way rand_core::BlockRng hands out ChaCha words (parity mode).
 * env_words_dev / actor_words_dev: u32 [num_envs][words_per_lane] (lane-major). */
typedef enum { RL_NOISE_PHILOX = 0, RL_NOISE_REPLAY = 1 } rl_noise_mode;
rl_status rl_env_set_noise_replay(rl_env *env, const uint32_t *env_words_dev, const uint32_t *actor_words_dev,
                                  uint64_t words_per_lane);
rl_status rl_env_set_noise_philox(rl_env *env, uint64_t seed, uint32_t step_counter);
/* 64-bit noise slot of the Philox source (host-side; lets a CPU checker replay production noise) */
uint64_t rl_philox_slot(uint64_t seed, uint64_t lane, uint32_t step, int32_t stream, uint32_t draw);

/* Unfused path: Environment::initial_state + observe for every lane (mod.rs:76-100). */
rl_status rl_env_reset_all(rl_env *env);
/* Environment::step + observe for every lane with auto-reset on episode end, the way
 * Steps::step starts a new episode on the next call (src/simulation/steps.rs:113-168).
 * Device pointers into library-owned buffers, valid until the env is destroyed. */
typedef struct rl_step_out {
    const float *obs;      /* f32 [F][E]: observation the NEXT action must be taken on */
    const float *reward;   /* f32 [E] */
    const uint8_t *succ;   /* u8 [E] */
    const float *next_obs; /* f32 [F][E], valid where succ == RL_INTERRUPT */
} rl_step_out;
rl_status rl_env_step(rl_env *env, const uint8_t *actions_dev, rl_step_out *out);
rl_status rl_env_observation(rl_env *env, const float **obs_dev);
/* Debug/parity access to the raw state.  CartPole: f64 [4][E] (x, x', theta, theta') + u32 [E]
 * (steps_remaining | flag<<31).  Other kinds: u32 [E] packed state only (f64 part unused). */
rl_status rl_env_get_state(rl_env *env, double *f64_host, uint32_t *u32_host);
rl_status rl_env_set_state(rl_env *env, const double *f64_host, const uint32_t *u32_host);

/* ------------------------------------------------------------------------------------------ */
/* Feature encoding (FeatureSpace::batch_features src/spaces/mod.rs:329-412)                    */
/* ------------------------------------------------------------------------------------------ */
typedef enum {
    RL_SPACE_INTERVAL = 0,   /* [x as f32]                 src/spaces/interval.rs:101-117 */
    RL_SPACE_INDEX = 1,      /* one-hot(size)              src/spaces/index.rs:97-138 */
    RL_SPACE_BOOLEAN = 2,    /* [0|1]                      src/spaces/boolean.rs:125-139 */
    RL_SPACE_OPTION_INDEX = 3/* [is_none, one-hot(size)]   src/spaces/option.rs:88-116 */
} rl_space_kind;
/* elems: f64 for INTERVAL, i64 otherwise (OPTION_INDEX: -1 = None).  out: f32 [n][num_features]
 * row-major (the reference layout), both device pointers. */
rl_status rl_encode_features(rl_ctx *ctx, rl_space_kind kind, uint64_t size, const void *elems_dev, uint64_t n,
                             float *out_dev);

/* LazyHistoryFeatures (src/torch/agents/features.rs:70-215) over the stored episodes of `traj`, in the packed order of
 * PackedStructure / PackedSeqIter (src/torch/packed.rs:346-420): episodes sorted by length descending (ties in buffer
 * order: lane, then time; the reference's sort_unstable leaves ties unordered), interleaved time-major.  The update
 * kernels of this library read the [T][F][E] planes directly and never need this; it materialises the reference's own
 * layout for callers that do (a libtorch module on the other side of the boundary, checks against the reference).
 * Device outputs, any may be NULL; N = num_steps, M = num_episodes, L = max_len:
 *   obs f32 [N][F] (observation_features), ext_obs f32 [N + M][F] and ext_invalid u8 [N + M]
 *   (extended_observation_features: per episode one more row -- the successor observation on Interrupt, zeros and
 *   invalid = 1 on Terminate), action i64 [N] (actions), reward f32 [N] (rewards), batch_sizes i64 [L],
 *   ext_batch_sizes i64 [L + 1].  Sizing by the trajectory's capacity (T E rows, 2 T E for ext) is always enough. */
typedef struct rl_packed_info {
    uint64_t num_steps, num_episodes, max_len;
} rl_packed_info;
rl_status rl_pack_history(rl_traj *traj, float *obs_dev, float *ext_obs_dev, uint8_t *ext_invalid_dev, int64_t *action_dev,
                          float *reward_dev, int64_t *batch_sizes_dev, int64_t *ext_batch_sizes_dev, rl_packed_info *info);

/* ------------------------------------------------------------------------------------------ */
/* MLP module (BuildModule / Module::variables src/torch/modules/mod.rs:21-235, ff/mlp.rs)      */
/* ------------------------------------------------------------------------------------------ */
typedef enum { RL_ACT_IDENTITY = 0, RL_ACT_RELU = 1, RL_ACT_SIGMOID = 2, RL_ACT_TANH = 3 } rl_activation;
/* MlpConfig{hidden_sizes, activation, output_activation = Identity} (mlp.rs:25-34).  Parameters are
 * flat f32 in Module::variables() order: per Linear kernel[out,in] row-major then bias[out]
 * (linear.rs:108-110, mlp.rs:126-128).  n_hidden = 1 (<= 1024 units; the default [128] takes the tensor-core /
 * warp-specialised kernels), 2 or 3 (<= 256 units per layer, <= 48 K parameters: layer-generic kernels);
 * anything else returns RL_ERR_UNSUPPORTED. */
rl_status rl_mlp_create(rl_ctx *ctx, int32_t in_dim, const int32_t *hidden_sizes, int32_t n_hidden, int32_t out_dim,
                        rl_activation activation, rl_mlp **out);
rl_status rl_mlp_destroy(rl_mlp *mlp);
rl_status rl_mlp_num_params(rl_mlp *mlp, uint64_t *n);
rl_status rl_mlp_set_weights(rl_mlp *mlp, const float *host, uint64_t n);
/* The same copy enqueued on the context stream without waiting for it (the per-period weight refresh of an actor,
 * train.rs:124-158: no host round trip between the update and the next rollout).  `pinned_host` must be page-locked
 * (rl_malloc_host; RL_ERR_INVALID_ARG otherwise) and must not change until the next call that synchronises the context
 * (rl_ctx_synchronize, rl_rollout with a summary, any read-back). */
rl_status rl_mlp_set_weights_async(rl_mlp *mlp, const float *pinned_host, uint64_t n);
rl_status rl_mlp_get_weights(rl_mlp *mlp, float *host, uint64_t n);
/* Forward on feature planes: x f32 [F][n] -> out f32 [out_dim][n] (Mlp::forward mlp.rs:139-151). */
rl_status rl_mlp_forward(rl_mlp *mlp, const float *x_dev, uint64_t n, float *out_dev);

/* ------------------------------------------------------------------------------------------ */
/* Recurrent module Chain<Gru, Linear> (src/torch/modules/chain.rs:12-186, seq/rnn/gru.rs,      */
/* seq/rnn/mod.rs:166-280, ff/linear.rs): one GRU layer in_dim -> hidden, activation, Linear     */
/* hidden -> out_dim.  Parameters are flat f32 in Module::variables() order: w_ih[3H,in],         */
/* w_hh[3H,H], b_ih[3H], b_hh[3H] (gate order r, z, n as libtorch), then kernel[out,H], bias.     */
/* ------------------------------------------------------------------------------------------ */
rl_status rl_grunet_create(rl_ctx *ctx, int32_t in_dim, int32_t hidden, int32_t out_dim, rl_activation activation,
                           rl_grunet **out);
/* Chain<Lstm, Linear> (seq/rnn/lstm.rs) behind the same handle type, the cell fixed at creation: one LSTM layer in_dim ->
 * hidden (num_layers 1, biases present), activation, Linear hidden -> out_dim.  Flat parameters w_ih[4H,in], w_hh[4H,H],
 * b_ih[4H], b_hh[4H] (gate order i, f, g, o as libtorch's lstm_cell), then kernel[out,H], bias[out]: 4H(in+H) + 8H +
 * out*H + out values.  (h, c) start at zero in every episode.  Same ranges as rl_grunet_create; every function below that
 * takes an rl_grunet* accepts it, and rl_grunet_destroy frees it. */
rl_status rl_lstmnet_create(rl_ctx *ctx, int32_t in_dim, int32_t hidden, int32_t out_dim, rl_activation activation,
                            rl_grunet **out);
rl_status rl_grunet_destroy(rl_grunet *net);
rl_status rl_grunet_num_params(rl_grunet *net, uint64_t *n);
rl_status rl_grunet_set_weights(rl_grunet *net, const float *host, uint64_t n);
rl_status rl_grunet_get_weights(rl_grunet *net, float *host, uint64_t n);
/* SeqPacked::seq_packed over the stored episodes of a trajectory (hidden state zero at the first step of
 * every episode, gru.rs:23-28,72-102).  out_dev: f32 [T][out_dim][E], zeros in unused slots. */
rl_status rl_grunet_seq_forward(rl_grunet *net, rl_traj *traj, float *out_dev);

/* ------------------------------------------------------------------------------------------ */
/* Rollout = Agent::actor + Steps + TakeAlignedSteps + write_experience + OnlineStepsSummary     */
/* (src/simulation/steps.rs:113-168, take_steps.rs:18-89, agents/buffers/vec.rs:113-141,        */
/*  buffers/mod.rs:237-261, simulation/summary.rs:198-216, train.rs:98-158)                     */
/* Each lane is one reference "worker": it starts fresh episodes, takes min_steps (+ up to       */
/* slack_steps to finish the episode), and its dangling last step is dropped with the previous   */
/* step becoming Interrupt(dropped observation).                                                 */
/* ------------------------------------------------------------------------------------------ */
typedef enum {
    RL_ACTOR_REPLAY_ACTIONS = 0,     /* scripted actions u8 [T][E] (parity mode) */
    RL_ACTOR_RANDOM = 1,             /* RandomAgent: action_space.sample (src/agents/random.rs) */
    RL_ACTOR_CATEGORICAL_POLICY = 2, /* PolicyActor::act (src/torch/agents/policies/actor.rs:42-55) */
    RL_ACTOR_EPS_GREEDY_Q = 3,       /* DqnActor::act (src/torch/agents/dqn.rs:360-379) */
    RL_ACTOR_TABULAR_EPS_GREEDY = 4, /* BaseTabularQLearningActor::act (src/agents/tabular.rs:222-232) */
    RL_ACTOR_UCB1 = 5,               /* BaseUCB1Actor::act (src/agents/bandits/ucb.rs:214-243) */
    /* ResettingMetaAgent (src/agents/meta.rs:16-227) over the inner agent rl_actor_cfg.inner_kind, on RL_ENV_BANDIT_META
     * only (RL_ERR_UNSUPPORTED elsewhere).  Every lane carries its own inner agent, rebuilt at every trial start from the
     * inner env structure (one observation, num_arms actions, the env's reward range) and updated online from the meta
     * observation's previous step; it lives one trial inside one launch and never reaches device memory.  The inner actor
     * always acts in training mode (meta.rs:103-106), so rl_actor_cfg.training is ignored.  lanes_per_env must be 0. */
    RL_ACTOR_RESETTING_META = 6,
    /* BaseBetaThompsonSamplingActor::act (src/agents/bandits/thompson_sampling.rs:192-212) over rl_actor_cfg.bts: training
     * draws num_samples Beta(high, low) values per action from the device's own Beta sampler (DESIGN section 5) and keeps
     * the largest sum, evaluation the largest high / (high + low); ties go to the LAST maximal action.  Thread per env. */
    RL_ACTOR_BETA_THOMPSON = 7
} rl_actor_kind;

/* rl_actor_cfg.inner_kind: the agent RL_ACTOR_RESETTING_META rebuilds at each trial (the rl2-bandits baselines) */
typedef enum {
    RL_INNER_RANDOM = 0,    /* RandomAgent (src/agents/random.rs) */
    RL_INNER_TABULAR_Q = 1, /* BaseTabularQLearningAgent (src/agents/tabular.rs:84-232): values 0, counts 0 (build_agent
                             * ignores initial_action_count / initial_action_value, tabular.rs:61-77), epsilon-greedy with
                             * epsilon = exploration_rate */
    RL_INNER_UCB1 = 2,      /* BaseUCB1Agent (src/agents/bandits/ucb.rs:78-243): one success and one failure per arm,
                             * rewards scaled by the env's reward range, exploration_rate scales the bound */
    RL_INNER_BETA_THOMPSON = 3 /* BaseBetaThompsonSamplingAgent (src/agents/bandits/thompson_sampling.rs:94-212): counts
                                * (1, 1) per arm, the reward threshold halfway through the env's reward range,
                                * rl_actor_cfg.num_samples Beta draws per arm */
} rl_inner_agent_kind;

/* rl_actor_cfg.lanes_per_env value selecting the tensor-core rollout kernel (CartPole + 5/4-128-2 ReLU network) */
#define RL_LANES_TENSOR_CORE 128
/* rl_actor_cfg.lanes_per_env value selecting the warp-specialised rollout kernel K2q (policy and dynamics of an env on
 * different warps; CartPole + 5/4-128-2 ReLU network) at any size.  Its results are bit-identical to lanes_per_env = 8.
 * It serves the categorical actor on Philox noise only; any other actor or replayed noise is refused with
 * RL_ERR_UNSUPPORTED. */
#define RL_LANES_WARP_SPECIALIZED 160
typedef struct rl_actor_cfg {
    int32_t kind;                 /* rl_actor_kind */
    rl_mlp *net;                  /* CATEGORICAL_POLICY / EPS_GREEDY_Q with a feed-forward module */
    const uint8_t *actions_dev;   /* REPLAY_ACTIONS: u8 [T][E] */
    rl_tabq *table;               /* TABULAR_EPS_GREEDY */
    double exploration_rate;      /* EPS_GREEDY_Q / TABULAR_EPS_GREEDY; RESETTING_META: the inner tabular agent's epsilon
                                   * or the inner UCB1 agent's exploration rate (unused for the random inner agent) */
    int32_t training;             /* ActorMode::Training (src/agents/mod.rs:144) */
    int32_t lanes_per_env;        /* 0 = auto; threads cooperating on one env's MLP (1,2,4,8,16,32),
                                   * RL_LANES_TENSOR_CORE (128): 128-env tiles, hidden layer on tcgen05 (K2t), or
                                   * RL_LANES_WARP_SPECIALIZED (160): K2q */
    rl_grunet *seq_net;           /* CATEGORICAL_POLICY / EPS_GREEDY_Q with a recurrent module (Chain<Gru, Linear>) instead of
                                   * `net`; hidden state zero at every episode start.  EPS_GREEDY_Q keeps the reference's order:
                                   * gen_bool(eps), then gen_range(A) on an explored step WITHOUT stepping the module (its hidden
                                   * state does not advance), else the module step and the first maximal Q-value */
    rl_ucb1 *ucb;                 /* UCB1 (training: maximise the upper confidence bound; evaluation: the most selected action) */
    int32_t inner_kind;           /* RESETTING_META: rl_inner_agent_kind; read for no other kind */
    rl_bts *bts;                  /* BETA_THOMPSON (the draw count comes from the handle) */
    int32_t num_samples;          /* RESETTING_META with RL_INNER_BETA_THOMPSON: Beta draws summed per arm, 1 .. 1024 */
} rl_actor_cfg;

/* HistoryDataBound (src/agents/buffers/mod.rs:25-113), per lane */
typedef struct rl_bound { uint64_t min_steps, slack_steps; } rl_bound;

/* OnlineMeanVariance (src/utils/stats.rs:121-213) */
typedef struct rl_mean_var { double mean, squared_residual_sum; uint64_t count; } rl_mean_var;
/* StepsSummary (src/simulation/summary.rs:11-117) */
typedef struct rl_steps_summary {
    rl_mean_var step_reward, episode_reward, episode_length;
    uint64_t num_stored_steps;    /* steps kept after finalize_last_episode, all lanes */
    uint64_t num_stored_episodes;
} rl_steps_summary;

rl_status rl_traj_create(rl_env *env, uint64_t step_capacity, rl_traj **out);
rl_status rl_traj_destroy(rl_traj *traj);
typedef struct rl_traj_view {
    uint64_t num_lanes, step_capacity, num_features;
    const float *obs; const uint8_t *action; const float *reward; const uint8_t *succ; const float *next_obs;
    const uint32_t *lane_len; /* u32 [E] stored steps per lane */
    uint64_t num_steps;       /* valid steps on this device */
} rl_traj_view;
rl_status rl_traj_view_of(rl_traj *traj, rl_traj_view *out);
/* Fill a trajectory from caller data (parity/KAT entry point); arrays in the device layouts above. */
rl_status rl_traj_load(rl_traj *traj, uint64_t steps, const float *obs_dev, const uint8_t *action_dev,
                       const float *reward_dev, const uint8_t *succ_dev, const float *next_obs_dev);

/* summary may be NULL (then nothing is read back and the call does not synchronise). */
rl_status rl_rollout(rl_env *env, const rl_actor_cfg *actor, rl_bound bound, rl_traj *traj,
                     rl_steps_summary *summary);

/* ------------------------------------------------------------------------------------------ */
/* Scans (PackedTensor::discounted_cumsum_from_end src/torch/packed.rs:280-342;                 */
/*        reward_to_go / temporal_differences / gae src/torch/agents/critics/mod.rs:101-199)    */
/* ------------------------------------------------------------------------------------------ */
/* y[t][e] = x[t][e] + d * y[t+1][e], restarted after every step with succ != CONTINUE. */
rl_status rl_discounted_cumsum(rl_ctx *ctx, const float *x_dev, const uint8_t *succ_dev, uint64_t steps,
                               uint64_t lanes, float discount, float *y_dev);
/* Packed form of the reference (time-major ragged, longest first) for KATs; host arrays. */
rl_status rl_discounted_cumsum_packed(rl_ctx *ctx, float *x_host, uint64_t n, const uint64_t *batch_sizes,
                                      uint64_t n_batches, float discount);
/* Critic::advantages with AdvantageFn::Gae and StepValueTarget::RewardToGo in one pass:
 * value_fn may be NULL (then V == 0: advantages = reward-to-go with discount gamma*lambda).
 * adv_dev / rtg_dev: f32 [T][E], either may be NULL. */
rl_status rl_gae(rl_traj *traj, rl_mlp *value_fn, float gamma, float lambda, float *adv_dev, float *rtg_dev);

/* ------------------------------------------------------------------------------------------ */
/* TRPO  (Policy::update src/torch/agents/policies/trpo.rs:97-164 +                             */
/*        TrustRegionOptimizer src/torch/optimizers/conjugate_gradient.rs:115-403)              */
/* ------------------------------------------------------------------------------------------ */
typedef struct rl_trpo_cfg {
    double max_policy_step_kl;   /* 0.01 (trpo.rs:29-38) */
    uint64_t cg_iterations;      /* 10 (conjugate_gradient.rs:55-64) */
    uint64_t max_backtracks;     /* 15 */
    double backtrack_ratio;      /* 0.8 */
    double hpv_reg_coeff;        /* 1e-5 */
    int32_t accept_violation;    /* false */
} rl_trpo_cfg;
void rl_trpo_cfg_default(rl_trpo_cfg *cfg);
/* the reference's log keys (trpo.rs:119, conjugate_gradient.rs:164,200,219-226) */
typedef struct rl_trpo_stats {
    double entropy, step_size, loss_initial, loss_final, constraint_val_final, step_scale;
    int64_t num_backtracks;      /* -1 when no candidate was accepted */
    int64_t cg_iterations;
    uint64_t num_steps;          /* global N */
    float policy_update_ms;
} rl_trpo_stats;
/* Returns RL_OK or one of RL_STEP_* (then the policy parameters are unchanged).  `policy` may be any one-hidden-layer
 * module (<= 64 features, <= 1024 units, <= 16 actions; ReLU / tanh / sigmoid / identity); the reference's default
 * 5 -> 128 -> 2 ReLU policy runs on tensor cores.  The same holds for the other rl_*_update entry points below. */
rl_status rl_trpo_update(rl_traj *traj, const float *adv_dev, rl_mlp *policy, const rl_trpo_cfg *cfg,
                         rl_trpo_stats *stats);

/* The pieces of one TRPO step for diagnostics and parity checks: the loss_distance_fn closure of
 * trpo.rs:124-146 at the current parameters (loss, kl, entropy of the behaviour policy), the flat
 * loss gradient (conjugate_gradient.rs:127,143) and HessianVectorProduct::mat_vec_mul(vec)
 * (conjugate_gradient.rs:312-338).  grad_host / fvp_host: f32 [num_params]; any output may be NULL. */
rl_status rl_trpo_probe(rl_traj *traj, const float *adv_dev, rl_mlp *policy, const float *vec_host, double hpv_reg_coeff,
                        double *loss, double *kl, double *entropy, float *grad_host, float *fvp_host);

/* ------------------------------------------------------------------------------------------ */
/* Critic / Adam (Critic::update src/torch/agents/critics/opt.rs:100-127; n_backward_steps      */
/*   src/torch/agents/mod.rs:35-72; COptimizer/AdamConfig src/torch/optimizers/coptimizer.rs)   */
/* ------------------------------------------------------------------------------------------ */
typedef struct rl_adam_cfg { double learning_rate, beta1, beta2, weight_decay, eps; } rl_adam_cfg;
void rl_adam_cfg_default(rl_adam_cfg *cfg); /* lr 1e-3, betas .9/.999, wd 0, eps 1e-8 (libtorch) */
rl_status rl_adam_create(rl_mlp *mlp, const rl_adam_cfg *cfg, rl_adam **out);
rl_status rl_adam_destroy(rl_adam *adam);
typedef struct rl_opt_stats { double loss_first, loss_last; uint64_t num_steps; uint64_t opt_steps; float update_ms; } rl_opt_stats;
/* n_steps x { V(obs) forward, mse(V, targets), backward, Adam step } over all valid steps. */
rl_status rl_value_update(rl_traj *traj, const float *targets_dev, rl_mlp *value_fn, rl_adam *adam, int32_t n_steps,
                          rl_opt_stats *stats);

/* Which kernel runs the full-batch passes of the default networks (5 -> 128 -> 1 critic, 5 -> 128 -> 2 policy):
 * mlp_pass_tc_kernel (tcgen05 tensor cores + TMEM; the default) or mlp_pass_kernel (FP32 pipe; also selected by
 * RL_PASS_KERNEL=ffma in the environment).  Process-wide; for diagnostics and for parity checks between the two. */
enum { RL_PASS_KERNEL_FFMA = 0, RL_PASS_KERNEL_TCGEN05 = 1 };
rl_status rl_pass_kernel_select(int32_t kernel);

/* One full-batch pass of the critic for diagnostics and parity checks: mse_loss(V(obs), targets) (opt.rs:109-115)
 * and its flat gradient at the current parameters, computed by the named kernel (RL_PASS_KERNEL_*).
 * grad_host: f32 [num_params]; either output may be NULL. */
rl_status rl_value_probe(rl_traj *traj, const float *targets_dev, rl_mlp *value_fn, int32_t kernel, double *loss,
                         float *grad_host);

/* ------------------------------------------------------------------------------------------ */
/* The same updates for a recurrent module (Chain<Gru, Linear>; rl2-bandits.rs:379-430): TRPO with   */
/* back-propagation through time and a forward-tangent + BPTT Fisher-vector product in place of the  */
/* reference's autograd double backward, ValuesOpt with a GRU critic, GAE over SeqPacked values.     */
/* hidden <= 8 (features <= 20, outputs <= 16): one thread per lane (K9).  Up to hidden 128, 64       */
/* features, 32 outputs -- the rl2-sized GRU(14 -> 128) -> Linear(128 -> 10) -- as tiled GEMMs over  */
/* the lanes of a step (K10; hidden 128 on tcgen05 tensor cores).  RL_ERR_UNSUPPORTED beyond.        */
/* ------------------------------------------------------------------------------------------ */
rl_status rl_trpo_update_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, const rl_trpo_cfg *cfg,
                             rl_trpo_stats *stats);
rl_status rl_trpo_probe_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, const float *vec_host,
                            double hpv_reg_coeff, double *loss, double *kl, double *entropy, float *grad_host,
                            float *fvp_host);
rl_status rl_adam_create_seq(rl_grunet *net, const rl_adam_cfg *cfg, rl_adam **out);
rl_status rl_value_update_seq(rl_traj *traj, const float *targets_dev, rl_grunet *value_fn, rl_adam *adam, int32_t n_steps,
                              rl_opt_stats *stats);
rl_status rl_gae_seq(rl_traj *traj, rl_grunet *value_fn, float gamma, float lambda, float *adv_dev, float *rtg_dev);

/* ------------------------------------------------------------------------------------------ */
/* PPO and REINFORCE policies (Policy::update src/torch/agents/policies/ppo.rs:97-147,          */
/* reinforce.rs:64-89) -- same data path as TRPO with an Adam step in place of the CG step.     */
/* ------------------------------------------------------------------------------------------ */
typedef struct rl_ppo_cfg {
    uint64_t opt_steps_per_update; /* 10 (ppo.rs:33-41) */
    double clip_distance;          /* 0.2 */
} rl_ppo_cfg;
void rl_ppo_cfg_default(rl_ppo_cfg *cfg);
typedef struct rl_policy_opt_stats {
    double entropy;                /* logged "entropy" (ppo.rs:116-117, reinforce.rs:85-87) */
    double loss_first, loss_last;
    uint64_t num_steps, opt_steps;
    float update_ms;
} rl_policy_opt_stats;
/* no_grad initial log-probs, then opt_steps x { clipped surrogate loss, backward, Adam } */
rl_status rl_ppo_update(rl_traj *traj, const float *adv_dev, rl_mlp *policy, rl_adam *adam, const rl_ppo_cfg *cfg,
                        rl_policy_opt_stats *stats);
/* one backward_step on -(log_probs * advantages).mean() */
rl_status rl_reinforce_update(rl_traj *traj, const float *adv_dev, rl_mlp *policy, rl_adam *adam,
                              rl_policy_opt_stats *stats);
/* The same two updates for a recurrent policy (Chain<Gru, Linear> or Chain<Lstm, Linear>, the shapes of
 * rl_trpo_update_seq) with back-propagation through time; `adam` from rl_adam_create_seq on that policy. */
rl_status rl_ppo_update_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, rl_adam *adam, const rl_ppo_cfg *cfg,
                            rl_policy_opt_stats *stats);
rl_status rl_reinforce_update_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, rl_adam *adam,
                                  rl_policy_opt_stats *stats);

/* ------------------------------------------------------------------------------------------ */
/* Tabular Q (BaseTabularQLearningAgent src/agents/tabular.rs:84-232)                           */
/* One table per replica; a replica folds its own lane's steps in order (bit-exact f64/u64).     */
/* num_replicas = 1 with E > 1 lanes = the reference under train_parallel: every lane acts from  */
/* the one table and rl_tabq_update folds lane 0, lane 1, ... into it in order (train.rs:98-186).*/
/* ------------------------------------------------------------------------------------------ */
rl_status rl_tabq_create(rl_ctx *ctx, uint64_t num_replicas, int32_t num_observations, int32_t num_actions,
                         double discount_factor, rl_tabq **out);
rl_status rl_tabq_destroy(rl_tabq *t);
/* BatchUpdate::batch_update: replica r folds lane r of the trajectory; a single shared table folds every lane in
 * lane order (tabular.rs:197-207). */
rl_status rl_tabq_update(rl_tabq *t, rl_traj *traj);
/* q: f64 [R][S][A], counts: u64 [R][S][A] (host) */
rl_status rl_tabq_get_table(rl_tabq *t, double *q_host, uint64_t *counts_host);
rl_status rl_tabq_set_table(rl_tabq *t, const double *q_host, const uint64_t *counts_host);

/* UCB1Agent (src/agents/bandits/ucb.rs:20-243): UCB1 applied independently to each state of a finite observation space.
 * Tables per replica: mean reward f64 [S][A] (rewards scaled to [0, 1] by the env's reward range, :118-123), selection
 * count u64 [S][A], visit count u64 [S]; initialised to one success and one failure per arm (:125-128).  As for rl_tabq,
 * num_replicas = 1 is the reference under train_parallel (every lane acts from the one table, rl_ucb1_update folds lane 0,
 * lane 1, ... into it in order, :186-199), num_replicas = num_envs trains independent agents.  The actor is deterministic
 * given the tables; ties go to the LAST maximal action (utils/iter/cmp.rs:58-76). */
rl_status rl_ucb1_create(rl_ctx *ctx, uint64_t num_replicas, int32_t num_observations, int32_t num_actions, double reward_lo,
                         double reward_hi, double exploration_rate, rl_ucb1 **out);
rl_status rl_ucb1_destroy(rl_ucb1 *u);
rl_status rl_ucb1_update(rl_ucb1 *u, rl_traj *traj);
rl_status rl_ucb1_get_tables(rl_ucb1 *u, double *mean_host, uint64_t *action_count_host, uint64_t *visit_count_host);
rl_status rl_ucb1_set_tables(rl_ucb1 *u, const double *mean_host, const uint64_t *action_count_host,
                             const uint64_t *visit_count_host);

/* BetaThompsonSamplingAgent (src/agents/bandits/thompson_sampling.rs:20-212): Beta-Bernoulli Thompson sampling applied
 * independently to each state of a finite observation space.  Tables per replica: low and high reward counts u64 [S][A],
 * both starting at 1; a step counts as high when its reward is above (reward_lo + reward_hi) / 2 (f64, strict).  As for
 * rl_ucb1, num_replicas = 1 is one agent shared by every lane (train_parallel) and num_replicas = num_envs one agent per
 * lane; the counts are integer increments, so rl_bts_update's result does not depend on the order of the steps.
 * num_samples (1 .. 1024) is the number of Beta draws summed per action in training mode. */
rl_status rl_bts_create(rl_ctx *ctx, uint64_t num_replicas, int32_t num_observations, int32_t num_actions, double reward_lo,
                        double reward_hi, int32_t num_samples, rl_bts **out);
rl_status rl_bts_destroy(rl_bts *b);
rl_status rl_bts_update(rl_bts *b, rl_traj *traj);
rl_status rl_bts_get_counts(rl_bts *b, uint64_t *low_host, uint64_t *high_host);
rl_status rl_bts_set_counts(rl_bts *b, const uint64_t *low_host, const uint64_t *high_host);

/* ------------------------------------------------------------------------------------------ */
/* DQN (ReplayBuffer src/agents/buffers/replay.rs:11-126; DqnAgent::batch_update                 */
/*      src/torch/agents/dqn.rs:236-337; schedules.rs)                                          */
/* ------------------------------------------------------------------------------------------ */
rl_status rl_replay_create(rl_env *env, uint64_t step_capacity_per_lane, rl_replay **out);
rl_status rl_replay_destroy(rl_replay *rb);
/* WriteExperience::write_experience of every lane's thread of experience. */
rl_status rl_replay_append(rl_replay *rb, rl_traj *traj);
typedef struct rl_replay_stats { uint64_t num_steps, num_episodes, total_step_count; } rl_replay_stats;
rl_status rl_replay_stats_of(rl_replay *rb, rl_replay_stats *out);
typedef struct rl_dqn_cfg {
    uint64_t minibatch_steps;    /* 100_000 (dqn.rs:57-72) */
    int32_t opt_steps_per_update;/* 50 */
    int32_t target_one_step_td;  /* 0 = StepValueTarget::RewardToGo (default), 1 = OneStepTd */
    float discount_factor;
    uint64_t sample_seed;
} rl_dqn_cfg;
/* One sample_minibatch of dqn.rs:280-314 on this device: draw j takes lane j mod E (the round-robin over
 * buffers) and a uniformly random stored episode of it (Uniform::new(0, num_episodes)), episodes are
 * taken while the step total is below minibatch_steps, and targets are computed per cfg.  Draw words
 * come from rl_philox_slot(sample_seed, lane = j, step = draw_index, stream = 3, draw = 0, 1, ...).
 * Device pointers are valid until the next sample/update on this buffer. */
typedef struct rl_minibatch_view {
    uint64_t num_steps, num_episodes, capacity;
    const float *obs;      /* f32 [F][capacity], columns [0, num_steps) valid, episodes in draw order */
    const uint8_t *action; /* u8 [capacity] */
    const float *target;   /* f32 [capacity]  StepValueTarget::targets (critics/mod.rs:203-229) */
    const uint8_t *succ;   /* u8 [capacity]   0 = valid column, RL_PAD = unused */
} rl_minibatch_view;
rl_status rl_replay_sample(rl_replay *rb, const rl_dqn_cfg *cfg, rl_mlp *q, uint32_t draw_index, rl_minibatch_view *out);
/* Debug/parity read-back of one lane's buffer, oldest step first (ReplayBuffer::steps / episodes,
 * replay.rs:74-86).  obs/next_obs f32 [n][F] row-major; episode_len u64 [num_episodes]; any array may be NULL. */
rl_status rl_replay_read_lane(rl_replay *rb, uint64_t lane, uint64_t max_steps, float *obs_host, uint8_t *action_host,
                              float *reward_host, uint8_t *succ_host, float *next_obs_host, uint64_t *episode_len_host,
                              rl_replay_stats *lane_stats);
/* opt_steps_per_update x { sample_minibatch, mse(Q(obs).gather(action), targets), backward, Adam }
 * (dqn.rs:263-337); with a data-parallel group every rank samples its own minibatch_steps and the
 * gradient sums are all-reduced. */
rl_status rl_dqn_update(rl_replay *rb, rl_mlp *q, rl_adam *adam, const rl_dqn_cfg *cfg, rl_opt_stats *stats);
/* The same update with a recurrent action-value module (Chain<Gru, Linear>; DqnAgent over SeqPacked + SeqIterative modules,
 * dqn.rs:75-83,190-197,341-352).  Every optimizer step draws the episodes rl_dqn_update would draw (same sample_seed and draw
 * index) and lays them out as padded sequences, one episode per lane from a zero hidden state; the Q-loss is averaged over the
 * valid steps and back-propagated through time (hidden <= 8: one thread per episode; up to 128: GEMMs over the episodes of a
 * step).  OneStepTd targets come from a SeqPacked forward with the current parameters; an interrupted episode's successor
 * observation continues that episode's hidden state.  Synchronises once per optimizer step (the sampled sizes are read back). */
rl_status rl_dqn_update_seq(rl_replay *rb, rl_grunet *q, rl_adam *adam, const rl_dqn_cfg *cfg, rl_opt_stats *stats);
/* Diagnostic read of one sequence minibatch of rl_dqn_update_seq (synchronises): out->num_lanes = B episodes taken (in draw
 * order), out->step_capacity = L = the longest, out->lane_len = episode lengths, out->num_steps = M; planes in the device layouts
 * above with B lanes and L steps: succ is RL_CONTINUE inside an episode, its stored code on its last step and RL_PAD beyond;
 * next_obs is valid where succ == RL_INTERRUPT.  *target_dev: f32 [L][B] targets per cfg (q is needed for OneStepTd only).
 * Device pointers are valid until the next sample or update on this buffer. */
rl_status rl_replay_sample_seq(rl_replay *rb, const rl_dqn_cfg *cfg, rl_grunet *q, uint32_t draw_index, rl_traj_view *out,
                               const float **target_dev);
/* The Q-loss pass of rl_dqn_update_seq on the sequence minibatch of `draw_index`, for diagnostics and parity checks: the
 * mean loss (dqn.rs:316-326) and its flat gradient at the current parameters, no optimizer step.  grad_host: f32 [num_params];
 * either output may be NULL. */
rl_status rl_dqn_probe_seq(rl_replay *rb, const rl_dqn_cfg *cfg, rl_grunet *q, uint32_t draw_index, double *loss, float *grad_host);
/* ExplorationRateSchedule::LinearAnnealed (schedules.rs:35-45) */
double rl_exploration_rate(double start, double end, uint64_t period, uint64_t global_steps, int32_t training);

#ifdef __cplusplus
}
#endif
#endif /* RELEARN_B200_H */
