/*
 * ssd_b200.h — C ABI of libssd_b200.so, the B200 (sm_100a) batched simulator for the
 * sequential-social-dilemma environments of Algorithmic-Alignment-Lab/contracts.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference has no FFI of its own: the
 * interface it exposes for this path is the Python MultiAgentEnv `reset()/step()` of the
 * classes built by `utils/env_creator_functions.py:12-34`.  Each entry point below replaces
 * the batched equivalent of one reference method (cited per function; paths relative to the
 * reference root).  The Python binding a maintainer adds is a ctypes stub — see
 * INTEGRATION.md and contracts_b200/_lib.py.
 *
 * Conventions
 *   - plain C: opaque handle, POD config, raw pointers + sizes, no C++/torch types;
 *   - every function returns 0 on success or a negative SSD_E* code; the message is
 *     available through ssd_last_error(handle) (or ssd_last_error(NULL) for create errors);
 *   - all `_dev` pointers are device pointers owned by the CALLER (e.g. torch tensors via
 *     tensor.data_ptr()); the library owns only the persistent per-env state;
 *   - every call is asynchronous on the given `stream` (a cudaStream_t passed as void*;
 *     NULL = legacy default stream) and performs no host synchronisation;
 *   - a handle is bound to one device and is not thread-safe; calls must be stream-ordered.
 *   - env i of a handle has global id `first_env_id + i`; its random stream is
 *     Philox4x32-10 keyed (seed, global id), so trajectories do not depend on how envs are
 *     sharded over handles / GPUs.
 */
#ifndef SSD_B200_H
#define SSD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSD_ABI_VERSION 3

/* env_kind: which reference class the handle simulates */
#define SSD_ENV_CLEANUP 0           /* environments/cleanup_new.py  CleanupEnv   ('CleanupNew') */
#define SSD_ENV_HARVEST 1           /* environments/harvest_new.py  HarvestEnv   ('HarvestNew') */
#define SSD_ENV_CLEANUP_FEATURES 2  /* environments/cleanup_features.py CleanupFeatures ('Cleanup') */
#define SSD_ENV_HARVEST_FEATURES 3  /* environments/harvest_features.py HarvestFeatures ('Harvest') */
#define SSD_ENV_SELFDRIVE 4         /* environments/self_driving_car_accelerate.py ('SelfDrive') */

/* contract_kind: contract/contract_list.py classes fused into the reward write */
#define SSD_CONTRACT_NONE 0
#define SSD_CONTRACT_CLEANUP 1              /* CleanupContract                 :7-27  */
#define SSD_CONTRACT_HARVEST_LOCAL 2        /* HarvestFeaturemodLocalContract  :29-54 */
#define SSD_CONTRACT_SELFDRIVE_DISTPROP 3   /* SelfdriveContractDistprop       :56-102 */

#define SSD_MAX_AGENTS 8
#define SSD_OBS_BYTES_PER_AGENT 675         /* 15 x 15 x 3 uint8 (map_env.py:397-411) */
#define SSD_METRIC_STRIDE 56                /* doubles per env written by ssd_get_metrics */

#define SSD_OK 0
#define SSD_EINVAL (-1)
#define SSD_ENOMEM (-2)
#define SSD_ECUDA (-3)
#define SSD_EUNSUPPORTED (-4)

typedef struct ssd_handle ssd_handle;

/* ssd_config.flags, cleanup_new / harvest_new: MapEnv kwargs use_collective_reward and
 * inequity_averse_reward (map_env.py:69-70): reward shaping at the end of MapEnv.step (map_env.py:289-301) */
#define SSD_FLAG_COLLECTIVE_REWARD 1
#define SSD_FLAG_INEQUITY_AVERSE 2

typedef struct ssd_config {
    int32_t abi_version;      /* SSD_ABI_VERSION */
    int32_t struct_size;      /* sizeof(ssd_config) as the caller compiled / declared it: ssd_create rejects a struct
                                 that is shorter than the library's (a stale binding would otherwise be read past its end) */
    int32_t env_kind;
    int32_t num_envs;         /* E, envs stepped per launch by this handle */
    int32_t num_agents;       /* n in [1, 8] */
    int32_t map_h, map_w;     /* gridworlds: ascii map size; ignored by selfdrive */
    const char* ascii_map;    /* map_h * map_w chars, row-major (CLEANUP_MAP / HARVEST_MAP layout) */
    int32_t horizon;          /* env `horizon` kwarg (cleanup_new.py:71): done when t == horizon */
    int32_t contract_kind;
    double theta_low;         /* contract_space.low[0]  (a float32 value, e.g. 0) */
    double theta_high;        /* contract_space.high[0] (a float32 value, e.g. float32(0.2)) */
    double null_prob;         /* SeparateContractSubgameStage null_prob (two_stage_train.py:152-166) */
    uint32_t seed;            /* Philox key word 0 */
    uint32_t first_env_id;    /* global id of env 0 (Philox key word 1 = first_env_id + i) */
    int32_t device;           /* CUDA device ordinal */
    int32_t flags;            /* SSD_FLAG_* bits (gridworlds), else 0 */
    double env_params[8];     /* selfdrive: low_bound, high_bound, start_vel, start_vel_ambulance
                                 (SelfAcceleratingCarEnv.__init__, self_driving_car_accelerate.py:19);
                                 cleanup_new / harvest_new: alpha, beta of inequity_averse_reward
                                 (map_env.py:71-72,293-300); else unused */
} ssd_config;

/* Buffers of one step.  Gridworld / feature envs: actions are uint8 [E][n] action ids
 * (Agent.py:8-16,161-162,198-199); selfdrive: float32 [E][n] accelerations.
 * NULL is allowed for every output except obs and rew (rew_dev may be NULL in ssd_step_host_async, whose result
 * block carries the rewards). */
typedef struct ssd_step_io {
    const void* actions_dev;
    uint8_t* obs_dev;         /* gridworlds: uint8 [E][n][15][15][3] (MapEnv.step 'curr_obs', map_env.py:269,284) */
    int64_t obs_env_stride;   /* bytes between consecutive envs in obs_dev (>= n*675; 0 = dense) */
    double* rew_dev;          /* [E][n] rewards AFTER contract transfers (two_stage_train.py:69-90) */
    double* base_rew_dev;     /* [E][n] env rewards before transfers (MapEnv.step rewards, map_env.py:285) */
    double* transfers_dev;    /* [E][n] Contract.compute_transfer values (contract_list.py) */
    uint8_t* info_dev;        /* [E][n][4]: eaten_apples, cleaned_squares|eaten_close_apples, total_close_apples, 0 */
    double* feature_obs_dev;  /* [E][n][F] infos['feature_obs'] (cleanup_new.py:243-251 F=12+n, harvest_new.py:215-222 F=10+2n) */
    uint8_t* done_dev;        /* [E] dones['__all__'] (cleanup_new.py:242) */
    /* Vectorised-sampler mode (what RLlib's rollout worker does with a vector env, utils/ray_config_utils.py:140: reset
     * an env as soon as it is done).  auto_reset != 0: every env that finishes in this step (t == horizon) is reset
     * by the step itself, exactly as ssd_reset with mask = done would (same draws, same episode statistics hand-off):
     * its rewards / dones / infos are those of the final step, its observation is the RESET observation of the next
     * episode.  With neg_proposals_dev / neg_accept_dev (double [E] / [E][n], the policy's negotiation outputs for every
     * env; only the rows of the resetting envs are read) the agreement stage of ssd_negotiate also runs for them
     * (neg_decision_dev uint8 [E], nullable, receives their decisions).  Needs done_dev.  One masked launch behind the step. */
    int32_t auto_reset;
    const double* neg_proposals_dev;
    const double* neg_accept_dev;
    uint8_t* neg_decision_dev;
} ssd_step_io;

/* --- lifetime ------------------------------------------------------------------------------- */
/* Replaces env_creator(name, config) (utils/env_creator_functions.py:12-34) for E envs at once:
 * parses the ascii map like MapEnv.__init__/CleanupEnv.__init__ (map_env.py:92-130,
 * cleanup_new.py:106-125), uploads point lists / palette / spawn-probability thresholds. */
int ssd_create(const ssd_config* cfg, ssd_handle** out);
void ssd_destroy(ssd_handle* h);
const char* ssd_last_error(const ssd_handle* h);

/* --- the hot path ----------------------------------------------------------------------------- */
/* MapEnv.reset + CleanupEnv/HarvestEnv.custom_reset + SeparateContractSubgameStage.reset
 * (map_env.py:306-342, cleanup_new.py:171-209, harvest_new.py:143-176, two_stage_train.py:159-187)
 * for the envs with mask_dev[i] != 0 (all envs when mask_dev is NULL).  Writes the reset
 * observation of those envs (agents are NOT drawn in it, as in the reference). */
int ssd_reset(ssd_handle* h, const uint8_t* mask_dev, uint8_t* obs_dev, int64_t obs_env_stride, void* stream);

/* MapEnv.step (map_env.py:216-304) + env step tail (cleanup_new.py:211-267 / harvest_new.py:181-239)
 * + SeparateContractEnv.step reward redistribution (two_stage_train.py:62-121), one launch for E envs. */
int ssd_step(ssd_handle* h, const ssd_step_io* io, void* stream);
/* Error surface of the step.  ssd_step returns SSD_OK as soon as the launch is enqueued; conditions that only the
 * kernel can see are recorded in a STICKY per-env flag word that lasts until the env is reset and is reported as
 * `err_flags` by ssd_get_metrics (out[5]) / ssd_set_episode_stats (max over envs):
 *   2  the reference would have raised KeyError in update_moves (map_env.py:640, agent_by_pos lookup)
 *   8  an action id outside the env's action space (the agent stays in place; the reference raises KeyError in
 *      Agent.action_map, Agent.py:161-162)
 *   16 ssd_set_state was given a map character that is not one of ' @AHRS'
 * The reference checks none of these eagerly either; callers that want a hard failure read err_flags at episode end
 * (contracts_b200/environments/gridworld.py does and raises).  There is no `rng_mode=injected` / ssd_set_injected_draws:
 * the only random stream is the counter-based Philox one (key = seed, global env id), which the parity harness injects
 * into the unmodified reference instead (oracle/ref_harness.py). */
/* The same step for a caller that holds HOST buffers (a CPU rollout worker, RLlib's sampler): copies
 * actions_host (uint8 [E][n], pinned for asynchronous copies) into io->actions_dev, steps, copies the rewards
 * (double [E][n], after transfers) and dones (uint8 [E], nullable) back, and returns when they are valid.  The device ->
 * host copy starts as soon as the rewards exist — for cleanup_new that is before the observe kernel, so it overlaps
 * it; the observations stay in the device batch tensor io->obs_dev. */
int ssd_step_host(ssd_handle* h, const ssd_step_io* io, const void* actions_host, double* rew_host, uint8_t* done_host,
                  void* stream);

/* Pipelined form of ssd_step_host (what RLlib's BaseEnv.send_actions() / poll() pair is to a vector env,
 * utils/ray_config_utils.py:140 -> rollout worker): submit step k + 1 before waiting for step k.  Two slots.
 *   ssd_step_host_async  uploads actions_host (uint8 [E][n], pinned) on a library-owned copy-in stream into the slot's
 *                        device action buffer (io->actions_dev is ignored), runs the step on `stream`, and — as soon as
 *                        the rewards exist, i.e. overlapping the observe kernel — copies ONE result block to
 *                        result_host (pinned, ssd_host_result_layout().total_bytes) on a copy-out stream.  Returns
 *                        without any host synchronisation; *ticket_out identifies the step (ticket & 1 = slot).
 *   ssd_step_host_wait   blocks until that step's result block is valid in host memory (and the slot can be reused).
 * At most two steps may be in flight; a slot must be waited for before it is submitted again (SSD_EINVAL otherwise).
 *
 * The result block is a LOSSLESS compact form of (rewards after transfers, dones).  Rewards on this path are small
 * integers except in envs where a contract transfer was paid this step, so the block holds
 *   count    uint32         number of records below
 *   done     uint8 [E]      dones['__all__']
 *   rew_i8   int8 [E][n]    the reward, valid for every env that is NOT in the record list
 *   records  [count] x { int32 env; int32 0; double rew[n] }   envs with a reward that is not an integer in
 *                           [-127, 127] (bit pattern compared, so -0.0 also lands here): all n exact float64 rewards;
 *                           order unspecified (warp-aggregated atomics)
 * at the byte offsets ssd_host_result_layout() reports.  Only the leading `count` records travel: the copy size is
 * predicted from the previous steps and ssd_step_host_wait fetches the remainder in the (rare) case of a miss.
 * ssd_host_result_expand() is the host-side convenience that rebuilds the dense float64 [E][n] matrix. */
typedef struct ssd_host_layout {
    int64_t total_bytes;      /* size of a result block (worst case: every env in the record list) */
    int64_t count_offset;     /* uint32 */
    int64_t done_offset;      /* uint8 [E] */
    int64_t rew_i8_offset;    /* int8 [E][n] */
    int64_t records_offset;   /* records, record_bytes each */
    int32_t record_bytes;     /* 8 + 8 n */
    int32_t record_capacity;  /* E */
} ssd_host_layout;
int ssd_host_result_layout(const ssd_handle* h, ssd_host_layout* out);
int ssd_step_host_async(ssd_handle* h, const ssd_step_io* io, const void* actions_host, void* result_host,
                        int64_t* ticket_out, void* stream);
int ssd_step_host_wait(ssd_handle* h, int64_t ticket);
/* The same pipelined form for the feature envs and selfdrive (declared with their io structs below): one kernel per step,
 * io->actions_dev ignored, io->rew_dev may be NULL.  ssd_host_result_layout / ssd_step_host_wait / ssd_host_result_expand
 * serve every env kind; the block's `done` field is uint8 [E] for the gridworlds and the feature envs and uint8 [E][n+1]
 * (per-car dones, then '__all__') for selfdrive, whose actions_host is float32 [E][n]. */
/* host code only: rew_out double [E][n] from a valid result block */
int ssd_host_result_expand(const ssd_handle* h, const void* result_host, double* rew_out);

/* --- contract parameters / negotiation ----------------------------------------------------------- */
/* theta_dev: double [E].  What SeparateContractNegotiateStage does with a0's proposal
 * (two_stage_train.py:258-262) / a caller-chosen contract. */
int ssd_set_contract_params(ssd_handle* h, const double* theta_dev, void* stream);
/* Agreement stage of SeparateContractNegotiateStage.step (two_stage_train.py:266-281):
 * proposals_dev double [E] (a0's action[:-1]), accept_dev double [E][n] (each agent's action[-1]),
 * decision_dev uint8 [E] out.  Chooses 2 of agents 1..n-1 when n > 3, multiplies their accept
 * values, draws once and keeps the proposal as theta or zeroes it.  Every env kind. */
int ssd_negotiate(ssd_handle* h, const uint8_t* mask_dev, const double* proposals_dev, const double* accept_dev,
                  uint8_t* decision_dev, void* stream);
/* mask_dev (nullable, uint8 [E]): negotiate only in the envs with mask_dev[i] != 0 — the envs that were just reset when
 * every env of the batch is at its own point of its episode (a vectorised sampler in steady state). */

/* --- JointEnv output layouts (environments/two_stage_train.py:476-617) ----------------------------- */
/* `global_obs`: MapEnv.global_view() (map_env.py:394-395; base_env.get_global_obs(), cleanup_new.py:299-300,
 * harvest_new.py:178-179, before the / 255): the whole colour map with agents, uint8 [E][H][W][3]. */
int ssd_global_view(ssd_handle* h, uint8_t* out_dev, void* stream);
/* `concatenated_obs`: np.concatenate of the agents' windows along the channel axis (two_stage_train.py:527-533,
 * 604-609): obs_dev uint8 [E][n][15][15][3] (env stride obs_env_stride, 0 = dense) -> out_dev uint8 [E][15][15][3n]. */
int ssd_concat_obs(ssd_handle* h, const uint8_t* obs_dev, int64_t obs_env_stride, uint8_t* out_dev, void* stream);

/* --- render path (environments/map_env.py:389-392,460-475) --------------------------------------------- */
/* MapEnv.beam_pos (map_env.py:231,812) is only ever shown by render(): recording it is optional.  When enabled, every
 * step also stores the cells its beams crossed (library-owned overlay, cleared at each step / reset). */
int ssd_record_beams(ssd_handle* h, int32_t enable);
/* MapEnv.full_map_to_colors() = render(mode='rgb_array') (map_env.py:389-392): the map with the agents and, when recorded,
 * the beams of the last step on top (get_map_with_agents, map_env.py:354-375).  out_dev uint8 [E][H][W][3]. */
int ssd_render(ssd_handle* h, uint8_t* out_dev, void* stream);

/* --- policy-side consumer (environments/Networks/vision_net.py:150-181) --------------------------------- */
#define SSD_POLICY_F32 0
#define SSD_POLICY_F16 1
#define SSD_POLICY_BF16 2
/* The observation as VisionNetwork.forward feeds its first convolution, in one pass over the uint8 batch tensor:
 * image_dev T [E*n][3][15][15] = (`curr_obs / 255` as float32).permute(0, 3, 1, 2) (:159,167) cast to T;
 * contract_dev (nullable) T [E*n][10] = (theta, 0) repeated 5 times (:160-161).  T by `dtype`. */
int ssd_policy_inputs(ssd_handle* h, const uint8_t* obs_dev, int64_t obs_env_stride, int32_t dtype, void* image_dev,
                      void* contract_dev, void* stream);
/* The same tensors written by the environment itself instead of by a second pass over the uint8 windows. */
typedef struct ssd_policy_out {
    int32_t struct_size;    /* sizeof(ssd_policy_out) (a smaller value is rejected) */
    int32_t dtype;          /* SSD_POLICY_F32 / _F16 / _BF16 */
    void*   image_dev;      /* T [E*n][3][15][15], 16-byte aligned: the tensor ssd_policy_inputs writes */
    void*   contract_dev;   /* T [E*n][10] = (theta, 0) x 5, nullable */
} ssd_policy_out;
/* Gridworld kinds.  While set (sticky, like ssd_set_episode_stats / ssd_record_beams; NULL switches it off), the handle
 * has one observation form, the policy's:
 *   - every call that writes uint8 windows — ssd_step, ssd_step_host, ssd_step_host_async, ssd_reset (masked or not) and
 *     the auto_reset behind a step — writes the image rows of the same envs instead, with exactly the values
 *     ssd_policy_inputs(dtype) would produce from the windows.  obs_dev must be NULL in these calls (else SSD_EINVAL);
 *   - every call that changes theta leaves the contract rows of the envs it changes current: ssd_reset, auto_reset with
 *     negotiation, ssd_negotiate, ssd_set_contract_params, ssd_solver_choose and ssd_checkpoint_load.  ssd_set_state, a
 *     parity tool, does not (call ssd_set_contract_params afterwards when it changed theta).
 * Validates before storing anything: SSD_EINVAL for a struct_size too small, an unknown dtype, a NULL or misaligned
 * image_dev, a contract_dev not aligned to its element, or a feature-env or selfdrive handle.  The caller keeps both
 * tensors alive while they are set. */
int ssd_set_policy_output(ssd_handle* h, const ssd_policy_out* out);
/* The flat rows a policy on the feature envs and selfdrive consumes (SeparateContractEnv, two_stage_train.py:113-121),
 * written by the environment itself.  Row e*n + a of obs_dev T [E*n][W] is agent a of env e:
 *   - with a contract (contract_kind != SSD_CONTRACT_NONE): W = F + 2, the row is features ++ [theta, 0] (theta: the env's
 *     contract parameter; the last column is the subgame stage, 0 on the device);
 *   - without a contract: W = F, the features alone.
 * F = ssd_feature_dim(h): 12 + n (cleanup features), 10 + 2n (harvest features), 2n + 5 (selfdrive).  Each element is
 * T(float32(x)), x the float64 the step writes without this mode (or theta): float64 -> float32 -> T, round to nearest
 * even.  Rows are W * sizeof(T) bytes and may start on any multiple of 2 bytes. */
typedef struct ssd_flat_policy_out {
    int32_t struct_size;    /* sizeof(ssd_flat_policy_out) (a smaller value is rejected) */
    int32_t dtype;          /* SSD_POLICY_F32 / _F16 / _BF16 */
    void*   obs_dev;        /* T [E*n][W], 16-byte aligned */
} ssd_flat_policy_out;
/* Feature-env and selfdrive kinds.  While set (sticky; NULL switches it off), the handle has one observation form, the
 * policy's:
 *   - every call that writes float64 rows — ssd_feat_step / ssd_selfdrive_step, their _host_async forms, ssd_feat_reset /
 *     ssd_selfdrive_reset (masked or not) and the auto_reset behind a step — writes the flat rows of the same envs
 *     instead (selfdrive: the rows of cars that did not act too).  obs_dev must be NULL in these calls (else SSD_EINVAL);
 *   - every call that changes theta leaves the theta column of the envs it changes current: ssd_set_contract_params,
 *     ssd_negotiate, ssd_solver_choose and ssd_checkpoint_load.
 * Validates before storing anything: SSD_EINVAL for a struct_size too small, an unknown dtype, a NULL or not 16-byte
 * aligned obs_dev, or a gridworld handle (those have ssd_set_policy_output).  The caller keeps the tensor alive while it
 * is set. */
int ssd_set_flat_policy_output(ssd_handle* h, const ssd_flat_policy_out* out);
/* The grid worlds' feature observation (image_obs=False: cleanup_new.py:193-202,243-254, harvest_new.py:160-168,212-222)
 * as the handle's observation, written on the device at every step and reset, with no observation windows:
 *   - SSD_FEATURE_F64: obs_dev double [E][n][F], each value what infos['feature_obs'] (the image_obs=False observation)
 *     holds; F = ssd_feature_dim(h) = 12 + n (cleanup), 10 + 2n (harvest);
 *   - SSD_POLICY_F32 / _F16 / _BF16: obs_dev T [E*n][W], the rows of ssd_set_flat_policy_output: W = F + 2 and the row
 *     features ++ [theta, 0] with a contract, W = F and the features alone without one; each element T(float32(x)).
 * Grid-world kinds.  While set (sticky; NULL switches the handle back to uint8 windows, and ssd_set_policy_output or
 * ssd_set_global_output replaces it, as it replaces them), the handle has this one observation form:
 *   - ssd_reset (masked or not) writes the reset rows of the envs it resets: the reset observation of the reference
 *     (cleanup: the apple / waste caches from before the reset-time spawn; harvest: the map after it), and ssd_step,
 *     ssd_step_host, ssd_step_host_async write the step's rows; the auto_reset behind a step writes the new episode's reset
 *     rows of the envs it restarts.  obs_dev and feature_obs_dev must be NULL in these calls (else SSD_EINVAL);
 *   - with a policy dtype under a contract, every call that changes theta leaves the theta column of the envs it changes
 *     current: ssd_reset, auto_reset with negotiation, ssd_negotiate, ssd_set_contract_params, ssd_solver_choose and
 *     ssd_checkpoint_load (ssd_set_state does not; the next step writes it).
 * Rewards, dones, infos, state, metrics, episode statistics and the episode log are those of the uint8 form.
 * Validates before storing anything: SSD_EINVAL for a struct_size too small, an unknown dtype, a NULL or not 16-byte aligned
 * obs_dev, or a feature-env or selfdrive handle.  The caller keeps the tensor alive while it is set. */
#define SSD_FEATURE_F64 3        /* accepted by ssd_set_feature_output only */
typedef struct ssd_feature_out {
    int32_t struct_size;    /* sizeof(ssd_feature_out) (a smaller value is rejected) */
    int32_t dtype;          /* SSD_FEATURE_F64, SSD_POLICY_F32 / _F16 / _BF16 */
    void*   obs_dev;        /* double [E][n][F] or T [E*n][W], 16-byte aligned */
} ssd_feature_out;
int ssd_set_feature_output(ssd_handle* h, const ssd_feature_out* out);
/* JointEnv's global observation (global_obs=True: two_stage_train.py:572-617, get_global_obs = global_view() / 255,
 * cleanup_new.py:299-300, harvest_new.py:178-179) as the handle's observation, written on the device at every step and
 * reset, with no observation windows:
 *   - SSD_GLOBAL_U8: obs_dev uint8 [E][H][W][3], byte for byte what ssd_global_view returns for the same state;
 *   - SSD_POLICY_F32 / _F16 / _BF16: obs_dev T [E][3][H][W], each element T(float32(u8 / 255.0)) of that view (the
 *     rounding of ssd_policy_inputs: VisionNetwork.forward's preprocessing of get_global_obs()).
 * Grid-world kinds without a contract (JointEnv wraps the bare base env).  While set (sticky; NULL switches the handle back
 * to uint8 windows, and each of ssd_set_policy_output / ssd_set_feature_output replaces it, as this call replaces them),
 * the handle has this one observation form:
 *   - ssd_reset (masked or not) writes the view of the envs it resets (the agents are not painted at t == 0, as
 *     MapEnv.reset leaves them out of the colour map), ssd_step, ssd_step_host and ssd_step_host_async write the view after
 *     the step, and the auto_reset behind a step writes the reset view of the envs it restarts.  obs_dev and
 *     feature_obs_dev must be NULL in these calls (else SSD_EINVAL).
 * Rewards, dones, infos, state, metrics, episode statistics, the episode log, ssd_global_view, ssd_render and beam recording
 * are those of the uint8 form.
 * Validates before storing anything: SSD_EINVAL for a struct_size too small, an unknown dtype, a NULL or not 16-byte aligned
 * obs_dev, a handle with a contract, or a feature-env or selfdrive handle.  The caller keeps the tensor alive while it is
 * set. */
#define SSD_GLOBAL_U8 4          /* accepted by ssd_set_global_output only */
typedef struct ssd_global_out {
    int32_t struct_size;    /* sizeof(ssd_global_out) (a smaller value is rejected) */
    int32_t dtype;          /* SSD_GLOBAL_U8, SSD_POLICY_F32 / _F16 / _BF16 */
    void*   obs_dev;        /* uint8 [E][H][W][3] or T [E][3][H][W], 16-byte aligned */
} ssd_global_out;
int ssd_set_global_output(ssd_handle* h, const ssd_global_out* out);

/* --- NegotiationSolver (environments/two_stage_train.py:619-776); every env kind ------------------- */
#define SSD_SOLVER_RULE_MAX 0        /* decision_rule 'max'      (:751-757) */
#define SSD_SOLVER_RULE_MAJORITY 1   /* decision_rule 'majority' (:758-773) */
/* negotiate() :705-746, the candidate contracts: params_dev double [E][1 + num_samples]; [e][0] = contract_space.low
 * (the null contract), [e][1 + i] = contract_param_space.sample() = float32(uniform(low, high)) from the env's
 * Philox stream.  The caller evaluates its value function V(s, c) per agent for every candidate (compute_vals
 * :693-703 — an RLlib policy forward in the reference). */
int ssd_solver_sample(ssd_handle* h, int32_t num_samples, double* params_dev, void* stream);
/* compute_best_param() :748-776 on vals_dev double [E][1 + num_samples][n]; the chosen parameter becomes the env's
 * contract parameter (reset :675-676) and is also written to best_param_dev double [E] / best_index_dev int32 [E]
 * (either may be NULL). */
int ssd_solver_choose(ssd_handle* h, int32_t num_samples, int32_t rule, const double* params_dev, const double* vals_dev,
                      double* best_param_dev, int32_t* best_index_dev, void* stream);

/* The solver inside a vectorised sampler, where every env is at its own point of its episode and only the envs that were
 * just reset choose a contract.  An env is PENDING when it is at the start of an episode (reset, t == 0) whose contract the
 * solver has not chosen yet.  Pending envs are taken in windows of at most `capacity` (C) envs in ascending env order:
 *   ssd_solver_rows     finds the window, samples its candidates and writes the value-query rows;
 *   (the caller)        runs its value function on all C x (1 + S) x n rows;
 *   ssd_solver_resolve  applies compute_best_param (two_stage_train.py:748-776) to the window and clears it from pending.
 * Each env ends with exactly what ssd_solver_sample + ssd_solver_choose give it on the same values.  Both calls are
 * asynchronous, synchronise nothing and can be captured in a CUDA graph: (step with auto_reset, rows, value function,
 * resolve) per step, with C >= the resets of a step; after a full reset, loop windows until pending (count_dev[1]) is 0.
 * Pending status is read from t and the episode counter, which every reset writes: no step or reset kernel changes. */
typedef struct ssd_solver_window {
    int32_t struct_size;      /* sizeof(ssd_solver_window) (a smaller value is rejected) */
    int32_t num_samples;      /* S >= 0 (contract_samples) */
    int32_t capacity;         /* C in [1, E] */
    int32_t* env_dev;         /* int32 [C]: the window's envs (local indices), -1 beyond the window */
    uint32_t* episode_dev;    /* uint32 [C]: their episode counters when the rows were written */
    uint32_t* count_dev;      /* uint32 [2]: envs in the window, pending envs in total (window included) */
    double* params_dev;       /* double [C][1 + S]: the candidates of ssd_solver_sample, 0 beyond the window */
    void* rows_dev;           /* [C][1 + S][n][W] value-query rows in the handle's observation form (below), 16-byte aligned */
} ssd_solver_window;
/* Every env kind with a contract.  on != 0 allocates the per-env record of resolved episodes and marks every env as
 * having none; 0 switches the queue off.  An env that was never reset is never pending; ssd_checkpoint_load marks the
 * envs it loads as resolved (their theta comes back with them). */
int ssd_solver_enable(ssd_handle* h, int32_t on);
/* Rows [C][1 + S][n][W] by the handle's observation form; row (c, k, a) is agent a of window env c with candidate k:
 *   - flat forms (feature envs and selfdrive, grid worlds with ssd_set_feature_output), W = F + 2: obs[e][a] ++ [param, 0]
 *       float64: what NegotiationSolver._obs_with builds (two_stage_train.py:316-325), obs = the float64 observation:
 *                obs_dev double [E][n][F] for the feature envs and selfdrive, the handle's feature rows for the grid worlds;
 *       policy dtype T: the handle's policy rows with the feature columns copied bit for bit, then T(float32(param)), 0;
 *   - image forms (grid worlds): the contract part alone, the image being the same for every candidate:
 *       uint8 windows: double (param, 0), W = 2;  policy image: T (param, 0) x 5, W = 10 (the contract rows).
 * obs_dev is required for the float64 form of the feature envs and selfdrive (their observation is passed per call) and
 * must be NULL otherwise.  Rows, candidates and env ids beyond the window count are zero / zero / -1. */
int ssd_solver_rows(ssd_handle* h, const ssd_solver_window* win, const void* obs_dev, void* stream);
/* vals_dev double [C][1 + S][n].  For each env of the window: the chosen parameter becomes its theta (and the policy
 * output's rows that carry it follow), best_param_dev[c] / best_index_dev[c] (nullable, double [C] / int32 [C]) receive it
 * and its candidate index, and its episode counts as resolved.  An env that was stepped or reset again since the rows
 * call is left unchanged: best_index -1, best_param its current theta, and stale_dev (nullable, uint32 [1]) counts it.
 * Slots beyond the window get best_index -1, best_param 0. */
int ssd_solver_resolve(ssd_handle* h, const ssd_solver_window* win, int32_t rule, const double* vals_dev, double* best_param_dev,
                       int32_t* best_index_dev, uint32_t* stale_dev, void* stream);

/* --- state access (parity tests, checkpointing) ---------------------------------------------------- */
/* map: uint8 chars [E][H][W] (MapEnv.world_map); pos: int32 [E][n][2] (row, col); ori: int32 [E][n]
 * (Agent.int_orientation); t: int32 [E] (MapEnv.timesteps); theta: double [E].  NULL pointers are skipped. */
int ssd_get_state(ssd_handle* h, uint8_t* map_dev, int32_t* pos_dev, int32_t* ori_dev, int32_t* t_dev,
                  double* theta_dev, void* stream);
int ssd_set_state(ssd_handle* h, const uint8_t* map_dev, const int32_t* pos_dev, const int32_t* ori_dev,
                  const int32_t* t_dev, const double* theta_dev, void* stream);
/* Episode accumulators behind env.metrics (cleanup_new.py:186-189,213-232,264-266; two_stage_train.py:92-99).
 * out_dev: double [E][SSD_METRIC_STRIDE] =
 *   [apples_eaten, low_density_eaten, raw_env_rewards, transfers, dirt_cleaned, err_flags, 0, 0,
 *    agent_a[8], agent_b[8], sum_raw[8], tsum_raw[8], sum_transferred[8], tsum_transferred[8]] */
int ssd_get_metrics(ssd_handle* h, double* out_dev, void* stream);
/* Episode statistics without a pass over all envs (the MetricsCallback hand-off, utils/logger_utils.py:126-151):
 * while stats_dev (double [SSD_STATS_LEN], caller-owned, caller-zeroed) is set, every ssd_reset adds the accumulators
 * of each FINISHED episode it replaces (envs that had been reset before) to it with device atomics:
 *   [apples_eaten, raw_env_rewards, transfers, dirt_cleaned, sum of transferred rewards, sum of raw rewards,
 *    episodes, max err_flags].  NULL switches it off.  Gridworld kinds. */
#define SSD_STATS_LEN 8
int ssd_set_episode_stats(ssd_handle* h, double* stats_dev);

/* Episode log: one record per finished episode, for every env kind (the per-episode form of the MetricsCallback hand-off,
 * utils/logger_utils.py:126-151).  While a log is set (sticky; NULL switches it off), the kernel that resets an env whose
 * episode it replaces appends one record to a caller-owned ring buffer on the device: ssd_reset / ssd_feat_reset /
 * ssd_selfdrive_reset (masked or not), the grid auto_reset behind a step, the next-step auto_reset of the feature and
 * selfdrive steps, and the pipelined host-buffer steps, which run the same kernels.  Nothing is read or synchronised per
 * step, and the appends work inside a captured CUDA graph.
 *   - only resets append: ssd_checkpoint_load and ssd_set_state are not episode ends;
 *   - an env that was never reset has no episode to log; a reset at t = 0 logs a zero-length episode (what
 *     ssd_set_episode_stats counts as an episode too);
 *   - the order of the records of one launch is unspecified, their contents are deterministic;
 *   - the caller keeps both buffers alive while the log is set. */
typedef struct ssd_episode_record {      /* 480 bytes, 16-byte aligned in the buffer */
    uint32_t env_id;     /* global id (first_env_id + i) */
    uint32_t episode;    /* number of the finished episode (0 = the env's first) */
    int32_t  t;          /* steps it ran */
    uint32_t ended;      /* 1: it ended by itself (grid / feature: t == horizon; selfdrive: every car done); 0: a reset cut it short */
    double   theta;      /* its contract parameter */
    double   pad;        /* 0 */
    double   metrics[SSD_METRIC_STRIDE];   /* grid: the ssd_get_metrics row; feature envs: the ssd_feat_get_metrics row
                                              (40 values, the rest 0); selfdrive: [0] = the transfers metric, the rest 0 --
                                              each exactly as the getter would have returned it just before the reset */
} ssd_episode_record;

typedef struct ssd_episode_log {
    int32_t struct_size;                 /* sizeof(ssd_episode_log); smaller is rejected */
    int32_t capacity;                    /* records in records_dev, >= 1 */
    ssd_episode_record* records_dev;     /* [capacity], 16-byte aligned */
    unsigned long long* count_dev;       /* records appended since it was zeroed (by the caller); record k lands in slot k % capacity */
} ssd_episode_log;

/* Every env kind.  Validates before storing anything: SSD_EINVAL for a struct_size too small, capacity < 1, a NULL or
 * misaligned records_dev (16 bytes) or count_dev (8 bytes). */
int ssd_set_episode_log(ssd_handle* h, const ssd_episode_log* log);

/* --- SelfAcceleratingCarEnv (env_kind SSD_ENV_SELFDRIVE) -------------------------------------------------
 * environments/self_driving_car_accelerate.py reset :49-79 / step :151-250 (collision_on=False), optionally with
 * SelfdriveContractDistprop (contract/contract_list.py:66-102) + SeparateContractSubgameStage
 * (two_stage_train.py:62-121,159-187) fused.  Agents that are done stop acting (RLlib semantics).  All values are
 * float64; D = 2 (n + 1) + 3 observation elements per car (ssd_feature_dim returns D). */
typedef struct ssd_selfdrive_io {
    const float* actions_dev;   /* [E][n] accelerations */
    double* obs_dev;            /* [E][n][D]  (rows of cars that did not act this step are still written) */
    double* rew_dev;            /* [E][n] after transfers; 0 for cars that did not act */
    double* base_rew_dev;       /* [E][n] nullable */
    double* transfers_dev;      /* [E][n] nullable: value of each car's transfer tuple */
    double* info_dev;           /* [E][n][4] nullable: just_passed, acted, ambulance_rank, ambulance_dist_to_front
                                   (last two in the row of the first acting car, like infos[key_lst[0]]) */
    uint8_t* done_dev;          /* [E][n+1] nullable: per-car dones, then '__all__' */
    int32_t auto_reset;         /* next-step auto-reset: an env whose episode ended ('__all__') in the previous step is reset
                                   by this step instead of being stepped — reset observation, zero rewards, dones cleared,
                                   its actions ignored (what ssd_selfdrive_reset with mask = done[:, n] would do, no launch) */
} ssd_selfdrive_io;
int ssd_selfdrive_reset(ssd_handle* h, const uint8_t* mask_dev, double* obs_dev, void* stream);
int ssd_selfdrive_step(ssd_handle* h, const ssd_selfdrive_io* io, void* stream);
/* host actions in (float32 [E][n], pinned), compact result block out: see ssd_step_host_async */
int ssd_selfdrive_step_host_async(ssd_handle* h, const ssd_selfdrive_io* io, const void* actions_host, void* result_host,
                                  int64_t* ticket_out, void* stream);
/* pos/vel double [E][n], theta / transfers metric double [E], t int32 [E]; NULL pointers are skipped */
int ssd_selfdrive_get_state(ssd_handle* h, double* pos_dev, double* vel_dev, double* theta_dev, double* transfers_dev,
                            int32_t* t_dev, void* stream);
/* uniform float32 accelerations in [lo, hi) for benchmark rollouts, [E][n] */
int ssd_selfdrive_random_actions(ssd_handle* h, uint32_t step_index, float lo, float hi, float* actions_dev, void* stream);

/* --- CleanupFeatures / HarvestFeatures (env_kind SSD_ENV_CLEANUP_FEATURES / SSD_ENV_HARVEST_FEATURES) ----------
 * environments/cleanup_features.py step :156-254 / reset :256-284, environments/harvest_features.py step :173-287 /
 * reset :289-336, optionally with CleanupContract / HarvestFeaturemodLocalContract + SeparateContractSubgameStage
 * fused (two_stage_train.py:62-121,159-187).  ssd_create takes the same ascii map as the gridworld kinds.
 * F = ssd_feature_dim(h) = 12 + n (cleanup) or 10 + 2 n (harvest) float64 features per agent. */
typedef struct ssd_feat_io {
    const uint8_t* actions_dev; /* [E][n] action ids (cleanup 0-8: moves, stay, turns, clean 7, fire 8; harvest 0-7) */
    double* obs_dev;            /* [E][n][F] */
    double* rew_dev;            /* [E][n] after transfers */
    double* base_rew_dev;       /* [E][n] nullable */
    double* transfers_dev;      /* [E][n] nullable */
    uint8_t* info_dev;          /* [E][n][4] nullable: cleanup (cleaned_squares,0,0,0); harvest (eaten_apples, eaten_close_apples,0,0) */
    uint8_t* done_dev;          /* [E] nullable: dones['__all__'] (timesteps == horizon) */
    int32_t auto_reset;         /* next-step auto-reset, as in ssd_selfdrive_io */
} ssd_feat_io;
int ssd_feat_reset(ssd_handle* h, const uint8_t* mask_dev, double* obs_dev, void* stream);
int ssd_feat_step(ssd_handle* h, const ssd_feat_io* io, void* stream);
/* host actions in (uint8 [E][n], pinned), compact result block out: see ssd_step_host_async */
int ssd_feat_step_host_async(ssd_handle* h, const ssd_feat_io* io, const void* actions_host, void* result_host,
                             int64_t* ticket_out, void* stream);
/* pos int32 [E][n][2], ori int32 [E][n], cells uint8 [E][H][W] (1 = apple, 2 = waste in the current lists),
 * theta double [E], t int32 [E]; NULL pointers are skipped */
int ssd_feat_get_state(ssd_handle* h, int32_t* pos_dev, int32_t* ori_dev, uint8_t* cells_dev, double* theta_dev,
                       int32_t* t_dev, void* stream);
/* double [E][40]: dirt_cleaned, raw_env_rewards, transfers, total_apples_eaten, low_density_apples_eaten,
 * err_flags (always 0 since the lists are kept in birth order; was: 16-bit birth stamps wrapped), 0, 0,
 * per agent: sum r [8], sum t*r [8], sum transferred r [8], sum t * transferred r [8] */
int ssd_feat_get_metrics(ssd_handle* h, double* out_dev, void* stream);

/* --- checkpoint / restore / copy of env state (every env_kind) ------------------------------------------------
 * One primitive behind resuming a run, re-sharding it over another number of handles and branching an env into others:
 * the complete mutable state of an env as one ROW of row_bytes bytes, and rows loaded back.  A row holds every byte a
 * later step, reset, negotiation, metrics call or auto_reset reads (flags and sticky error bits, the episode counter —
 * a word of every Philox counter —, the episode accumulators), and nothing the caller owns (observations, rewards,
 * infos, the episode-statistics vector), nor the per-step scratch, the beam overlay, the SSD_STEP_AUTO counter or the
 * pipelined host path's copy-size prediction.  A row loaded into env i continues on env i's own random stream
 * (seed, first_env_id + i): loaded into the env of the same global id it continues exactly as if it had never stopped.
 *
 * Row layouts (byte offsets; n = num_agents; unlisted bytes are padding and saved as 0):
 *   cleanup_new / harvest_new: the env record, row_bytes = 512 (640 with SSD_FLAG_COLLECTIVE_REWARD / _INEQUITY_AVERSE)
 *     0 u32 agent[8] (row | col << 8 | ori << 16)   32 i32 t   36 u32 episode   40 f64 theta
 *     48 u32 flags (bit 31 initialised, bit 0 stale apple list, bits 8.. sticky err_flags)   52 u32 #waste cells
 *     64 u32 apple mask[8]   96 u32 waste mask[8] (bit j = point j of the row-major point list)
 *     128.. episode accumulators (apples, low density, dirt, transfers, per-agent sums; 440..575 float64 shaped sums)
 *   cleanup / harvest (feature envs): row_bytes = L + LS, L = round16(192 + 28 n), LS = both list capacities
 *     0 u32 agent[8]   32 u32 apple list length   36 u32 waste list length   40 i32 t   44 u32 episode | init << 31
 *     48 f64 theta   64 u32 apple mask[8]   96 u32 waste mask[8]   128 f64 metrics[8]
 *     192 u64 sum t*r[n]   192+8n f64 sum transferred[n]   192+16n f64 sum t*transferred[n]   192+24n u32 sum r[n]
 *     L uint8 apple list (point indices, birth order; capacity LA = max(16, round16(#apple points)))   L+LA waste list
 *     (the bytes behind each list's length are saved as 0)
 *   selfdrive: row_bytes = round16(16 n + 40)
 *     0 f64 pos[n]   8n f64 vel[n]   16n f64 theta   16n+8 f64 transfers metric   16n+16 f64 dist_to_front
 *     16n+24 u32 crossing order (4 bits per entry)   16n+28 u32 n_crossed | done mask << 8 | all_done << 16 | init << 31
 *     16n+32 i32 t   16n+36 u32 episode
 * config_tag hashes a layout version and every ssd_config field except num_envs, first_env_id, seed, device and
 * struct_size: rows move between handles of the same configuration whatever their size or place in a sharded run. */
typedef struct ssd_checkpoint_layout {
    int64_t row_bytes;        /* bytes of one env's row, a multiple of 16 */
    uint64_t config_tag;      /* hash of everything that gives the row its meaning */
} ssd_checkpoint_layout;
int ssd_checkpoint_get_layout(const ssd_handle* h, ssd_checkpoint_layout* out);
/* rows_dev uint8 [count][row_bytes] (16-byte aligned) <- the envs env_idx_dev[0..count) (int32 local indices; NULL: envs
 * 0..count-1).  A row whose index is outside [0, E) is saved as zeros. */
int ssd_checkpoint_save(ssd_handle* h, const int32_t* env_idx_dev, int32_t count, uint8_t* rows_dev, void* stream);
/* rows_dev -> the envs env_idx_dev[0..count) (NULL: 0..count-1).  SSD_EINVAL before any launch when config_tag is not the
 * handle's.  Each row is validated first — agents inside the map, orientation <= 3, no mask bits beyond the point lists,
 * #waste = popcount of the waste mask, 0 <= t <= horizon (grid worlds); list lengths <= point counts, entries < point
 * counts, each list setting exactly the bits of its presence mask (feature envs); n_crossed <= n, crossing-order entries
 * < n, no entries beyond n_crossed (selfdrive) — and, like a row whose index is outside [0, E), written only when it
 * passes: row_ok_dev[r] (uint8, nullable) = 1 if row r was loaded, else 0.  Duplicate destinations are the caller's error.
 * With the solver queue on (ssd_solver_enable), the loaded envs' episodes count as resolved: their theta came with them. */
int ssd_checkpoint_load(ssd_handle* h, uint64_t config_tag, const int32_t* env_idx_dev, int32_t count, const uint8_t* rows_dev,
                        uint8_t* row_ok_dev, void* stream);

/* --- utilities ------------------------------------------------------------------------------------------ */
/* uniform random action ids in [0, num_actions) for benchmark rollouts, uint8 [E][n];
 * drawn from Philox site 13 at counter `step_index` (no reference equivalent: RLlib's policy).
 * step_index == SSD_STEP_AUTO takes (and then bumps) a per-handle device counter instead, so the call can be
 * captured in a CUDA graph and still draw fresh actions at every replay (the last CTA to finish bumps the counter). */
#define SSD_STEP_AUTO 0xFFFFFFFFu
int ssd_random_actions(ssd_handle* h, uint32_t step_index, int32_t num_actions, uint8_t* actions_dev, void* stream);   /* gridworld and feature kinds */
/* host-side Philox4x32-10 (so tests can pin the generator: KATs in tests/test_philox.py) */
void ssd_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
int ssd_abi_version(void);
int ssd_feature_dim(const ssd_handle* h);          /* F of feature_obs_dev */
int64_t ssd_state_bytes_per_env(const ssd_handle* h);
/* Measurement only (bench.py roofline): with timing on, ssd_step brackets its kernels with CUDA events on the
 * launch stream (not capturable in a CUDA graph).  ssd_get_step_times waits for the last step and returns
 * out_ms[0] = logic kernel, out_ms[1] = observe (+ harvest reward) kernel, in milliseconds. */
int ssd_enable_timing(ssd_handle* h, int32_t on);
int ssd_get_step_times(ssd_handle* h, double* out_ms);
int64_t ssd_kernel_launches(const ssd_handle* h);  /* kernels launched through this handle so far */

#ifdef __cplusplus
}
#endif
#endif /* SSD_B200_H */
