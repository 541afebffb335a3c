/*
 * evac_b200.h -- C ABI of the B200-native batched evacuation environment step.
 *
 * This is the drop-in boundary for the ONE hot path of cinemere/evacuation: the per-step
 * pedestrian dynamics + observation encoding behind `setup_env(...).reset()/step()`.
 * The reference has no FFI (it is pure Python); each entry point below names the Python
 * interface of the reference it replaces (paths relative to the reference root):
 *
 *   evac_create / evac_destroy   EvacuationEnv.__init__            src/env/env/env.py:41-84
 *                                EnvConfig / EnvWrappersConfig     src/env/env/config.py:3-100,
 *                                                                  src/env/wrappers/config.py:8-93
 *   evac_reset                   EvacuationEnv.reset               src/env/env/env.py:106-139
 *                                Pedestrians.reset                 src/env/env/pedestrians.py:16-27
 *   evac_step / evac_step_host   EvacuationEnv.step                src/env/env/env.py:141-171
 *                                Area.agent_step                   src/env/env/area.py:182-210
 *                                Area.pedestrians_step             src/env/env/area.py:76-180
 *                                update_statuses                   src/env/env/statuses.py:29-48
 *                                Reward.*                          src/env/env/reward.py:19-46
 *                                RelativePosition / PedestriansStatuses / MatrixObs
 *                                                                  src/env/wrappers/wrappers.py:8-96
 *                                GravityEncoding                   src/env/wrappers/gravity_encoding.py:41-81
 *   evac_rollout                 the caller's loop around step():  src/agents/rpo_agent.py:180-203 with
 *                                RandomAgent / RotatingAgent /     src/agents/random_agent.py:8-9,
 *                                WacuumCleaner                     src/agents/rotating_agent.py:12-16,
 *                                                                  src/agents/baseline_wacuum_cleaner.py:7-80
 *                                + pedestrians.status_stats        src/env/env/pedestrians.py:37-44 (efficiency curve,
 *                                                                  src/plotting_old/plot.py:165-201)
 *   evac_observe                 EvacuationEnv._get_observation + wrappers' observation()
 *                                                                  src/env/env/env.py:98-104
 *   evac_get_state/evac_set_state  env.unwrapped.{pedestrians,agent,time} attribute access
 *                                                                  (wrappers.py:35,48; gravity_encoding.py:50,64-65)
 *   evac_episode_stats           the per-episode logging dict      src/env/env/env.py:114-127
 *   evac_set_env_params /        one EnvConfig per environment     the reference's parameter sweeps (noise x enslaving
 *   evac_get_env_params          (gymnasium SyncVectorEnv over      x alpha grids) as one batch
 *                                differently configured envs)
 *
 * Conventions
 *   - plain C, no torch / C++ types; all array arguments are raw pointers.
 *   - unless a function name ends in `_host`, array pointers are DEVICE pointers on the
 *     handle's device and the call is asynchronous on `stream` (a cudaStream_t passed as void*;
 *     NULL = the legacy default stream).
 *   - every function returns 0 on success or a negative EVAC_ERR_* code; evac_last_error()
 *     returns a thread-local message for the last failure.
 *   - one handle per (process, GPU); a handle is not thread-safe.
 *   - there is NO CPU fallback: evac_create fails if no CUDA device is usable.
 *
 * Pedestrian status values (src/env/env/statuses.py:16-27): VISCEK=1, FOLLOWER=2, EXITING=3, ESCAPED=4.
 */
#ifndef EVAC_B200_H_
#define EVAC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVAC_ABI_VERSION 6

enum {
  EVAC_OK = 0,
  EVAC_ERR_INVALID = -1,     /* bad argument / unsupported configuration          */
  EVAC_ERR_CUDA = -2,        /* a CUDA runtime call failed                        */
  EVAC_ERR_UNSUPPORTED = -3, /* valid in the reference but not implemented (e.g. grav + Box, wrappers/config.py:80-81) */
  EVAC_ERR_NO_DEVICE = -4
};

enum { EVAC_STATUS_VISCEK = 1, EVAC_STATUS_FOLLOWER = 2, EVAC_STATUS_EXITING = 3, EVAC_STATUS_ESCAPED = 4 };
enum { EVAC_POS_ABS = 0, EVAC_POS_REL = 1, EVAC_POS_GRAV = 2 };     /* EnvWrappersConfig.positions */
enum { EVAC_STAT_NO = 0, EVAC_STAT_OHE = 1, EVAC_STAT_CAT = 2 };    /* EnvWrappersConfig.statuses  */
enum { EVAC_OBS_DICT = 0, EVAC_OBS_BOX = 1 };                       /* EnvWrappersConfig.type      */
enum { EVAC_PREC_F32 = 0, EVAC_PREC_F64 = 1 };                      /* pedestrian-state arithmetic */
enum { EVAC_AGENT_TABLE = 0, EVAC_AGENT_RANDOM = 1, EVAC_AGENT_ROTATING = 2, EVAC_AGENT_WACUUM = 3 }; /* evac_rollout action source */
/* neighbour search of the alignment pass (area.py:105-108 builds the full distance matrix):
 * AUTO = one-warp all-pairs tile for N <= 64, cell list (uniform grid, cell edge >= vision radius) above;
 * BRUTE = all-pairs shared-memory tiles for every N; CELLS = cell list whenever the shape supports it (N > 64, fp32) */
enum { EVAC_SEARCH_AUTO = 0, EVAC_SEARCH_BRUTE = 1, EVAC_SEARCH_CELLS = 2 };

/* Number of floats in one episode-statistics record, in the key order of env.py:115-125:
 * episode_intrinsic_reward, episode_status_reward, episode_reward, episode_length,
 * escaped_pedestrians, exiting_pedestrians, following_pedestrians, viscek_pedestrians,
 * overall_timesteps. */
#define EVAC_NUM_EPISODE_STATS 9

/* Plain-old-data mirror of EnvConfig (config.py:3-100) + EnvWrappersConfig (wrappers/config.py:8-44)
 * + SwitchDistances (distances.py:17-21).  Field names follow the reference. */
typedef struct EvacConfig {
  int32_t abi_version;            /* must be EVAC_ABI_VERSION */
  int32_t number_of_pedestrians;  /* N, 1 .. 32768 (all-pairs search: 1 .. 8192; fp64 parity mode: 1 .. 4096) */
  double width, height;           /* arena half-extents */
  double step_size;
  double noise_coef;
  double eps;
  double enslaving_degree;
  int32_t is_new_exiting_reward;
  int32_t is_new_followers_reward;
  double intrinsic_reward_coef;
  int32_t is_termination_agent_wall_collision;
  double init_reward_each_step;
  int32_t max_timesteps;
  /* observation wrappers */
  int32_t positions; /* EVAC_POS_*  */
  int32_t statuses;  /* EVAC_STAT_* */
  int32_t obs_type;  /* EVAC_OBS_*  */
  double alpha;      /* GravityEncoding alpha */
  /* SwitchDistances (constants.py:35-38): 0.2, 0.1 ("vision radius"), 0.4, 0.01 */
  double to_leader, to_pedestrian, to_exit, to_escape;
  /* batching extras (no counterpart in the reference) */
  int32_t auto_reset; /* 1: an env that terminates/truncates is reset inside the same step
                         (gymnasium vector-env "same-step" semantics, rpo_agent.py:193-203) */
  int32_t precision;  /* EVAC_PREC_F32 (product) or EVAC_PREC_F64 (parity mode) */
  int32_t neighbor_search; /* EVAC_SEARCH_* */
} EvacConfig;

/* Content hash (16 hex digits) of the sources this library was built from: SHA-256 over every .cu / .cuh file of csrc/ and
 * every .h file of include/ (evacuation_b200/build.py::source_hash).  The Python loader refuses a library whose id differs from the
 * tree's, so tests and benchmarks cannot run a stale binary. */
const char* evac_build_id(void);

typedef struct EvacHandle EvacHandle;

/* Fill `cfg` with the reference defaults (EnvConfig(), EnvWrappersConfig(), SwitchDistances). */
int evac_default_config(EvacConfig* cfg);

/* Create `num_envs` independent environments on CUDA device `device`.
 * `seed` keys the counter-based (Philox4x32-10) streams for reset layouts, noise and the
 * scripted agents; `env_index_offset` is added to the env index in the stream counter so a
 * batch sharded over several processes/GPUs draws the same numbers as one big batch. */
int evac_create(const EvacConfig* cfg, int32_t num_envs, int32_t device, uint64_t seed,
                int64_t env_index_offset, EvacHandle** out);
int evac_destroy(EvacHandle* h);

/* Floats per environment in one observation row (layout documented in DESIGN.md):
 *   Dict : [agent(2) | exit(2) | pedestrians(2N) | statuses(4N ohe, N cat, 0 no)]   (sorted-key order)
 *   Box  : [N+2, 2|3|6] row-major, rows = agent, exit, pedestrians                  (MatrixObs)
 *   grav : [agent(2) | grad_potential_exit(2) | grad_potential_pedestrians(2)] */
int32_t evac_obs_dim(const EvacHandle* h);
int32_t evac_num_envs(const EvacHandle* h);
/* number of cells of the neighbour-search grid (0 = all-pairs tiles) */
int32_t evac_num_cells(const EvacHandle* h);
/* bytes per element of the pedestrian state arrays exchanged by get/set_state (4 or 8) */
int32_t evac_state_elem_size(const EvacHandle* h);

/* Reset environments (all, or those with reset_mask[e] != 0) to a fresh random layout
 * (pedestrians.py:17-20 semantics: pos ~ U[-1,1)^2, dir = normalised U[-1,1)^2, agent at the
 * origin) drawn from the handle's Philox streams, then write observations to `obs`
 * ([E, obs_dim] float32, may be NULL). */
int evac_reset(EvacHandle* h, const uint8_t* reset_mask, float* obs, void* stream);

/* Overwrite / read the full simulation state.  Any pointer may be NULL (= leave / skip).
 * positions, directions: [E,N,2] float32 (EVAC_PREC_F32) or float64 (EVAC_PREC_F64);
 * statuses: [E,N] uint8 (set_state: NULL => recomputed from positions like pedestrians.py:21-26);
 * agent_position, agent_direction: [E,2] float32; now: [E] int32. */
int evac_set_state(EvacHandle* h, const void* positions, const void* directions, const uint8_t* statuses,
                   const float* agent_position, const float* agent_direction, const int32_t* now, void* stream);
int evac_get_state(EvacHandle* h, void* positions, void* directions, uint8_t* statuses,
                   float* agent_position, float* agent_direction, int32_t* now, void* stream);

/* Encode the observation of the CURRENT state into obs [E, obs_dim] float32. */
int evac_observe(EvacHandle* h, float* obs, void* stream);

/* One environment step for all E environments (env.py:141-171), ONE fused kernel launch.
 *   actions    [E,2] float32
 *   noise      [E,N] float32 or NULL.  NULL: the kernel draws U(-noise_coef/2, noise_coef/2)
 *              from its Philox stream.  Non-NULL: the injected-noise protocol -- entry [e,i]
 *              is the angular noise of pedestrian i and is used iff i is VISCEK or FOLLOWER
 *              (the k-th value the reference draws at area.py:124 goes to the k-th such i).
 *   obs        [E,obs_dim] float32 out (NULL to skip)
 *   reward     [E] float32 out; terminated, truncated: [E] uint8 out (any may be NULL) */
int evac_step(EvacHandle* h, const float* actions, const float* noise, float* obs, float* reward,
              uint8_t* terminated, uint8_t* truncated, void* stream);

/* Same call with HOST buffers: copies actions (and noise) host->device, steps, copies
 * obs / reward / flags device->host through the handle's pinned staging buffers and
 * synchronises.  This is the call a host-side Gymnasium user makes once per step.
 *   statuses   [E,N] uint8 out or NULL: the pedestrian statuses after the step (env.unwrapped.pedestrians.statuses,
 *              pedestrians.py:12; the rng="numpy" face needs them to draw the next step's |viscek + follower| noise
 *              values, area.py:124).  When obs, reward, terminated, truncated, statuses are page-locked and laid out back
 *              to back in that order, the whole result travels in ONE device->host copy.  When every buffer is page-locked
 *              and the batch is small (inputs + results <= 1 MB: the single environment up to a few hundred), nothing is copied at all: the
 *              kernel reads and writes the host buffers directly (unified addressing). */
int evac_step_host(EvacHandle* h, const float* actions, const float* noise, float* obs, float* reward,
                   uint8_t* terminated, uint8_t* truncated, uint8_t* statuses);

/* Checkpoint / resume: the COMPLETE device state of a handle -- pedestrian state, agent, time, episode index (the Philox
 * key word), running-episode accumulators, scripted-agent state, finished-episode statistics -- as one flat byte image in
 * DEVICE memory of evac_state_bytes(h) bytes.  The image is only meaningful for a handle created with the same
 * configuration, number of environments and library build; together with (seed, env_index_offset) it resumes a run
 * bit-identically (the random streams are counter-based: nothing else carries state).  Per-environment parameters
 * (evac_set_env_params) are configuration and are not part of the image.
 * [the reference has no checkpointing of the environment; SURVEY.md section 5] */
int64_t evac_state_bytes(EvacHandle* h);
int evac_save_state(EvacHandle* h, void* image, void* stream);
int evac_load_state(EvacHandle* h, const void* image, void* stream);

/* `num_steps` consecutive steps in ONE kernel launch with the state kept on chip.
 *   agent_kind EVAC_AGENT_TABLE: actions [num_steps,E,2] float32; EVAC_AGENT_RANDOM: U[-1,1)^2
 *              from the Philox stream (RandomAgent); EVAC_AGENT_ROTATING: (sin, cos)(0.05 k);
 *              EVAC_AGENT_WACUUM: the scripted sweep baseline (per-env state machine kept in the handle,
 *              re-armed by a reset, a same-step auto-reset or evac_set_state(agent_position))
 *   noise      NULL or [num_steps,E,N] float32 (injected)
 *   obs        [E,obs_dim] (observation after the last step) or, if obs_every_step != 0,
 *              [num_steps,E,obs_dim]; NULL to skip
 *   reward_sum [E] float32: sum of the rewards of the num_steps steps (NULL to skip)
 *   terminated, truncated: [E] uint8, OR over the steps (NULL to skip)
 *   status_counts [num_steps,E,4] uint16 or NULL: escaped, exiting, following, viscek pedestrians after every step
 *              (before a same-step auto-reset) -- the "escaped vs time" evacuation-efficiency statistic */
int evac_rollout(EvacHandle* h, int32_t num_steps, int32_t agent_kind, const float* actions, const float* noise,
                 float* obs, int32_t obs_every_step, float* reward_sum, uint8_t* terminated, uint8_t* truncated,
                 uint16_t* status_counts, void* stream);

/* Per-env statistics of the most recently FINISHED episode (auto_reset) -- [E, EVAC_NUM_EPISODE_STATS]
 * float32 plus finished[E] uint8 (1 if that env finished an episode since the last call; cleared by the call).
 * `totals` (may be NULL): [1 + EVAC_NUM_EPISODE_STATS] float64 = number of finished episodes and the sums of
 * their statistics since creation -- the vector that is all-gathered across ranks. */
int evac_episode_stats(EvacHandle* h, float* stats, uint8_t* finished, double* totals, void* stream);

/* Running accumulators of the CURRENT episode of every env (env.py:65-67,168-170) and the overall step counter
 * (area.py:42-59): acc [E,3] float64 = episode_reward, episode_intrinsic_reward, episode_status_reward;
 * overall_timesteps [E] int64.  Device pointers; either may be NULL. */
int evac_get_accumulators(EvacHandle* h, double* acc, int64_t* overall_timesteps, void* stream);

/* ---- per-environment dynamics and reward parameters: one handle runs a whole parameter grid (or domain randomisation)
 * in one launch per step, where a uniform handle needs one handle per configuration.
 *
 * The fields are the EvacConfig fields that enter one environment's own arithmetic.  Left out, and uniform over the handle:
 *   - width, height, to_pedestrian: they size the neighbour-search grid (cell list, cell masks, cluster grid);
 *   - to_leader, width, height, step_size: they place the WacuumCleaner's lanes;
 *   - eps, to_exit, to_escape: the reference's parameter sweeps do not vary them;
 *   - number_of_pedestrians and the observation modes: they are shapes.
 * Each record is converted exactly as evac_create converts the same EvacConfig fields, and the random streams are keyed by
 * (seed, global env index, episode, step), not by these values: environment e of a handle with per-env parameters computes
 * bit for bit what environment e of a uniform handle created with e's values (same E, seed and env_index_offset) computes. */
typedef struct EvacEnvParams {
  double noise_coef;
  double enslaving_degree;
  double alpha;                                /* GravityEncoding alpha (observation and reset / evac_observe) */
  double intrinsic_reward_coef;
  double init_reward_each_step;
  int32_t is_new_exiting_reward;
  int32_t is_new_followers_reward;
  int32_t is_termination_agent_wall_collision;
  int32_t max_timesteps;                       /* 1 .. 2^21, like EvacConfig */
} EvacEnvParams;

/* `params`: HOST array of E records, or NULL to return to the handle's uniform EvacConfig values.  Stream-ordered on
 * `stream`: steps enqueued before the call use the old values, steps after it the new ones (the host array may be reused as
 * soon as the call returns).  The device copy is allocated once per handle, so a CUDA graph captured while per-env parameters
 * are set reads the values of later calls.  Setting or clearing them switches the step / observe kernels between their uniform
 * and per-environment instances: a graph captured before the switch still runs the other instance and must be re-captured.
 * The parameters are configuration, not state: evac_state_bytes / evac_save_state / evac_load_state do not include them. */
int evac_set_env_params(EvacHandle* h, const EvacEnvParams* params, void* stream);
/* out: HOST array of E records -- the per-env values, or the EvacConfig values of every env of a uniform handle. */
int evac_get_env_params(const EvacHandle* h, EvacEnvParams* out);

/* Number of kernels this library launched since the handle was created. */
int64_t evac_launch_count(const EvacHandle* h);

const char* evac_last_error(void);
int32_t evac_abi_version(void);

/* ---- rollout-loop glue for BASELINE config 5 (SURVEY section 8 row f1): the CALLER of step() --------------------
 *
 *   evac_policy_*            RPOTransformerEmbedding.get_action_and_value / get_value, forward only
 *                                                                  src/agents/networks/rpo_transformer_agent_network.py:36-163
 *                                                                  src/agents/networks/rpo_linear_agent_network.py:19-61
 *                            or, with num_blocks = 0, RPOLinearNetwork on the flattened observation (the gravity-encoding
 *                            and flat-observation configs): no embedding kernel, the heads read the observation
 *                            + (optional, fused) gymnasium NormalizeObservation + clip(-1, 1), ClipAction
 *                                                                  src/agents/rpo_agent.py:24-33,186-193
 *   evac_normalize_reward    gymnasium NormalizeReward(gamma) + clip(-100, 100)      src/agents/rpo_agent.py:31-32
 *
 * The policy reads the [E, (N+2)*d_model] MatrixObs rows evac_step writes and produces the [E,2] actions evac_step
 * consumes, so policy -> step -> normalise stays on the device (two launches for the policy, one for the step; one for the
 * linear policy).  For the gravity encoding (K = 6) evac_rollout_policy (below) runs the whole loop, num_steps iterations per
 * step-kernel launch.
 *
 * num_blocks = 0 means "RPOLinearNetwork directly on the observation": K = seq_len * d_model is the observation width
 * (evac_policy_default_linear_config: seq_len 1, d_model = obs_dim), 1 <= K <= 4096, num_heads / dim_feedforward / use_resid /
 * dropout / layer_norm_eps are unused, and the weights are the heads part of the layout below only. */
typedef struct EvacPolicyConfig {
  int32_t abi_version;      /* must be EVAC_ABI_VERSION */
  int32_t seq_len;          /* S = number_of_pedestrians + 2 rows of the observation, 1 .. 64 (num_blocks = 0: 1) */
  int32_t d_model;          /* values per row: 6 (ohe), 3 (cat) or 2 (no statuses) (num_blocks = 0: the observation width) */
  int32_t num_heads;        /* RPOTransformerEmbeddingConfig.num_heads (3); 1 .. 4 (every (d_model, num_heads) pair is instantiated) */
  int32_t dim_feedforward;  /* .dim_feedforward (96) */
  int32_t num_blocks;       /* .num_blocks (2); 0 .. 8, 0 = the linear policy without embedding */
  int32_t use_resid;        /* .use_resid (0) */
  float dropout;            /* .dropout (0.1); applied only when EvacPolicyIO.training != 0 */
  float layer_norm_eps;     /* nn.LayerNorm default 1e-5 */
  int32_t num_hidden;       /* RPOLinearNetworkConfig.num_hidden (64); multiple of 4, <= 64 */
  int32_t action_dim;       /* 2; <= 3 */
} EvacPolicyConfig;

typedef struct EvacPolicy EvacPolicy;

int evac_policy_default_config(EvacPolicyConfig* cfg, int32_t number_of_pedestrians, int32_t d_model);
/* RPOLinearNetwork defaults (num_hidden 64, action_dim 2) on an observation of obs_dim floats: num_blocks 0, seq_len 1,
 * d_model obs_dim. */
int evac_policy_default_linear_config(EvacPolicyConfig* cfg, int32_t obs_dim);
int evac_policy_create(const EvacPolicyConfig* cfg, int32_t device, EvacPolicy** out);
int evac_policy_destroy(EvacPolicy* p);
/* Number of floats evac_policy_load_weights expects, in this order (PyTorch parameter layouts, row-major):
 *   for every block b: attention.Wq.weight [H*D, D], .bias [H*D], Wk.weight, Wk.bias, Wv.weight, Wv.bias,
 *                      attention.dense.weight [D, H*D], .bias [D], ff.0.weight [F, D], ff.0.bias [F],
 *                      ff.3.weight [D, F], ff.3.bias [D], norm1.weight [D], norm1.bias [D], norm2.weight [D], norm2.bias [D]
 *   critic.0.weight [NH, S*D], .bias [NH], critic.2.weight [NH, NH], .bias [NH], critic.4.weight [1, NH], .bias [1],
 *   actor_mean.0.weight [NH, S*D], .bias [NH], actor_mean.2.weight [NH, NH], .bias [NH], actor_mean.4.weight [A, NH], .bias [A],
 *   actor_logstd [A] */
int64_t evac_policy_num_weights(const EvacPolicy* p);
/* `weights` is a HOST pointer; the library repacks it for the kernels and uploads it (synchronous). */
int evac_policy_load_weights(EvacPolicy* p, const float* weights, int64_t count);
/* Pre-allocate the internal embedding scratch for up to `max_envs` environments (needed before a forward call is
 * captured in a CUDA graph without an `embedding` output buffer).  No-op for the linear policy. */
int evac_policy_reserve(EvacPolicy* p, int32_t max_envs);

typedef struct EvacPolicyIO {
  int32_t num_envs;
  const float* obs;          /* [E, S*D] float32 (device) */
  /* optional fused NormalizeObservation + clip: running mean / variance [E, S*D] updated in place with this step's
   * observation (gymnasium RunningMeanStd, one sample per env and step), *norm_count = samples seen BEFORE this call
   * (device double; the caller advances it), obs_norm (may be NULL) receives the normalised clipped observation */
  float* norm_mean;
  float* norm_var;
  const double* norm_count;
  float* obs_norm;
  float norm_eps, norm_clip;
  /* outputs (device), any may be NULL */
  float* embedding;          /* [E, S*D] output of the transformer blocks; must be NULL for the linear policy */
  float* mean;               /* [E, A] actor mean */
  float* value;              /* [E] critic */
  float* action;             /* [E, A] Normal(mean, exp(logstd)).sample() (or `given_action`, or the mean if !sample) */
  float* action_clipped;     /* [E, A] clip(action, -1, 1) -- what evac_step consumes */
  float* logprob;            /* [E] */
  float* entropy;            /* [E] */
  const float* given_action; /* optional [E, A]: evaluate the log-probability of this action instead of sampling */
  int32_t sample;
  int32_t training;          /* != 0: dropout active (the reference's rollouts never call .eval()) */
  uint64_t seed, offset;     /* counter-based streams (dropout masks, Normal sampling): vary `offset` per call ... */
  const uint64_t* offset_device; /* ... or point this at a DEVICE counter that is added to `offset` (NULL = unused): a
                                    forward captured in a CUDA graph then draws fresh numbers on every replay */
  int64_t env_index_offset;  /* global index of env 0 (sharding-invariant streams, like evac_create) */
  /* != 0: evaluation -- the normaliser's statistics are used frozen, like gymnasium's NormalizeObservation at test time.
   * norm_mean, norm_var and *norm_count are only read and stay bit for bit as they were (norm_count must still be given with
   * them); obs_norm, when given, still receives the normalised clipped observation.  Per element, op for op the one-warp
   * kernel's frozen normaliser (evac_rollout_policy with norm_update = 0):
   *     z = clip(__fmul_rn(__fsub_rn(x, mean), rsqrtf(__fadd_rn(var, norm_eps))), -norm_clip, norm_clip)
   * with NaN-propagating min / max (a NaN observation or statistic stays NaN and poisons only its own environment).
   * Evaluation runs without dropout: norm_frozen together with training != 0 on a transformer policy (num_blocks > 0) fails
   * with EVAC_ERR_UNSUPPORTED.  0 (a zero-initialised struct) updates the statistics as described above. */
  int32_t norm_frozen;
} EvacPolicyIO;

/* embedding kernel (+ heads kernel if any head output is requested), asynchronous on `stream`.  The heads -- the 372 x 128 and
 * 64 x 64 dense layers of rpo_linear_agent_network.py:23-42, the one dense contraction on this path -- run as 3xTF32 tcgen05.mma with
 * the accumulators in tensor memory (csrc/evac_policy_tc.cuh) whenever S * D is a multiple of 4; otherwise, or with EVAC_POLICY_TC=0 in
 * the environment at evac_policy_create, on the CUDA cores.  Both agree with a float64 evaluation to 3e-6.
 * Linear policy (num_blocks = 0): ONE launch, the heads kernel on `obs` (always, so that the normaliser runs even without head
 * outputs); the NormalizeObservation update + clip runs in the heads' load of X, and `obs` (plus norm_mean / norm_var / obs_norm
 * when K is a multiple of 4) must be 16-byte aligned.
 * Frozen normaliser (io->norm_frozen): the embedding kernel's prologue, or the heads' load of X, reads the statistics and writes only
 * obs_norm; on the tensor cores the frozen load takes the normaliser-free kernel's column tiling (64 columns below 296 row tiles of
 * 128 environments, 128 above), where the updating load always takes 128. */
int evac_policy_forward(EvacPolicy* p, const EvacPolicyIO* io, void* stream);
int64_t evac_policy_launch_count(const EvacPolicy* p);

/* NormalizeReward(gamma) + clip for E environments (all pointers device, in place on returns / ret_mean / ret_var;
 * *count = samples seen before this call).  Optionally (truncated, done_out non-NULL) also writes the rollout loop's
 * next_done = float(terminated | truncated) (rpo_agent.py:194) in the same pass. */
int evac_normalize_reward(int32_t num_envs, const float* reward, const uint8_t* terminated, const uint8_t* truncated, float* returns,
                          float* ret_mean, float* ret_var, const double* count, float* out, float* done_out, float gamma, float eps,
                          float clip, void* stream);

/* ---- the gravity-encoding rollout loop in ONE step-kernel launch per num_steps iterations ------------------------------
 *
 *   evac_rollout_policy      num_steps iterations of rpo_agent.py:180-203 for every environment, with the linear policy
 *                            (num_blocks = 0) as the agent of the one-warp step kernel: NormalizeObservation + clip, the heads,
 *                            Normal sampling (or the mean), ClipAction, the step with same-step auto-reset, NormalizeReward +
 *                            clip and next_done.  The state, both normalisers' per-env statistics and the loop's next_done stay
 *                            on chip for the whole launch.
 *
 * Every value is bit-identical to num_steps iterations of the per-step loop (evac_policy_forward with the fused normaliser on
 * obs, evac_step on the clipped action, evac_normalize_reward with done_out, and `count += 1.0` / `offset += 1` after each):
 * the heads are the CUDA-core heads kernel's sums (the kernel K = 6 takes) in the same order.
 *
 * Supported, anything else fails with EVAC_ERR_UNSUPPORTED: a handle that runs the one-warp kernel (float32, N <= 64) with
 * positions = grav (obs_dim 6), uniform or per-environment parameters; a policy with num_blocks = 0, K = 6 and action_dim 2, any
 * num_hidden it accepts.  The flat-observation linear policy is not taken: at K = 364 layer 1 of the two heads alone is 47 k FMAs
 * and 186 KB of weights per environment and step -- work for the tensor-core heads kernel, not for one warp.
 * Noise is always the in-kernel stream.  Sampling draws of iteration s use stream offset offset + *offset_device + s and the
 * policy's env_index_offset (in the io struct); the environment streams use the handle's.
 *
 * Launches (counted on the handle, evac_launch_count): the step kernel, plus one single-thread kernel that advances norm_count
 * (when norm_update != 0), ret_count and *offset_device by num_steps when any of them is given.  They are advanced after the
 * step kernel because every CTA of it reads them at its start. */
typedef struct EvacPolicyRolloutIO {
  /* inputs and carried state (device) */
  float* obs;                /* [E, 6] raw observation: read before the first iteration, overwritten with the one after the last */
  float* next_done;          /* [E] in / out */
  float* norm_mean;          /* [E, 6] NormalizeObservation running mean / variance (in place), or NULL: no normaliser */
  float* norm_var;
  double* norm_count;        /* device scalar: samples seen before the call */
  float norm_eps, norm_clip;
  int32_t norm_update;       /* 1: update the statistics (evac_policy_forward's fused normaliser), 0: use them frozen (evaluation) */
  float* returns;            /* [E] NormalizeReward state (in place), or NULL: no reward normaliser */
  float* ret_mean;
  float* ret_var;
  double* ret_count;         /* device scalar: samples seen before the call */
  float gamma, eps, clip;
  int32_t sample;            /* 0: the action is the actor mean */
  uint64_t seed, offset;     /* as in EvacPolicyIO */
  uint64_t* offset_device;   /* NULL or a DEVICE counter added to offset; advanced by num_steps */
  int64_t env_index_offset;  /* global index of env 0 in the POLICY's Normal draws (EvacPolicyIO.env_index_offset); the
                                environment streams are keyed by the handle's own env_index_offset */
  /* per-step outputs [num_steps, E, ...] (device), any may be NULL */
  float* obs_norm;           /* [T, E, 6] the normalised observation the policy saw */
  float* action;             /* [T, E, 2] the action before ClipAction */
  float* logprob;            /* [T, E] */
  float* value;              /* [T, E]; NULL skips the critic */
  float* reward_norm;        /* [T, E] the normalised, clipped reward (needs the reward normaliser) */
  float* dones;              /* [T, E] next_done BEFORE the step */
  uint16_t* status_counts;   /* [T, E, 4] as evac_rollout writes them */
  /* per-launch outputs [E] (device), any may be NULL: as in evac_rollout */
  float* reward_sum;
  uint8_t* terminated;
  uint8_t* truncated;
} EvacPolicyRolloutIO;

int evac_rollout_policy(EvacHandle* h, const EvacPolicy* p, int32_t num_steps, const EvacPolicyRolloutIO* io, void* stream);

/* ---- measurement helpers (used by bench.py; not part of the reference surface) ---- */
/* FP32 FMA-pipe peak probe: every thread runs `iters` x 8 independent FMA chains; packed != 0 uses
 * fma.rn.f32x2.  Returns elapsed milliseconds (CUDA events) in *ms and the flop count in *flops. */
int evac_probe_fma(int32_t device, int32_t packed, int32_t iters, float* ms, double* flops);
/* Standalone launch of the SAME pairwise neighbour-alignment device function the fused step uses:
 * E envs x N pedestrians, `reps` passes over a resident tile.  *ms = elapsed, *pairs = ordered pairs evaluated. */
int evac_probe_pairwise(int32_t device, int32_t num_envs, int32_t n, int32_t reps, float* ms, double* pairs);

#ifdef __cplusplus
}
#endif
#endif /* EVAC_B200_H_ */
