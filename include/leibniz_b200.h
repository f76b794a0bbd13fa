/*
 * leibniz_b200 — C ABI of the B200-native TriFinger MDP hot path.
 *
 * This is the drop-in boundary for the per-step reward + observation/state + reset
 * path of pairlab/leibnizgym (BASELINE.json north_star, SURVEY.md §8).  The reference
 * is pure Python/TorchScript, so there is no existing FFI to mirror: each entry point
 * replaces the chain of ATen ops the cited reference function issues.  All paths below
 * are relative to /root/reference/leibnizgym/.
 *
 * Conventions (every entry point):
 *   - returns 0 on success, a negative LG_ERR_* code otherwise; the message of the last
 *     error on the calling thread is available from lg_last_error();
 *   - all pointers are DEVICE pointers unless the name ends in _host; nothing is
 *     allocated, freed or retained; no host synchronisation happens inside;
 *   - `stream` is a cudaStream_t passed as void*; every launch goes onto it, so calls
 *     compose with CUDA graphs (stream capture);
 *   - float tensors are fp32, row-major, densely packed with the reference's shapes;
 *     bool tensors are 1 byte per element (torch.bool); step counters are int64.
 */
#ifndef LEIBNIZ_B200_H_
#define LEIBNIZ_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LG_VERSION 111            /* 1.1.1 */
#define LG_MAX_ACTION_DIM 18      /* position_impedance: 9 positions + 9 stiffnesses */
#define LG_MAX_STATE_DIM 122      /* 50 + 6 + 39 + 9 + 18 */
#define LG_NUM_TERMS 7            /* six reference terms + the keypoint extension */
#define LG_NUM_STATS 16
#define LG_INJECT_U_COLS 24
#define LG_INJECT_N_COLS 8
#define LG_HISTORY_COLS 16        /* 9 fingertip position floats + 7 object pose floats */

enum LgError {
  LG_OK = 0,
  LG_ERR_BAD_ARG = -1,     /* null / misaligned pointer, negative size, unknown enum   */
  LG_ERR_CUDA = -2,        /* a CUDA runtime call failed; text in lg_last_error()      */
  LG_ERR_UNSUPPORTED = -3  /* valid in the reference but not built (none at present)   */
};

/* order in which the reference evaluates and accumulates the terms
 * (envs/trifinger/trifinger_env.py:513-553) */
enum LgTerm {
  LG_TERM_FINGER_REACH_OBJECT_RATE = 0, /* envs/trifinger/rewards.py:187-235 */
  LG_TERM_FINGER_MOVE_PENALTY = 1,      /* rewards.py:238-263 */
  LG_TERM_OBJECT_DIST = 2,              /* rewards.py:37-63 */
  LG_TERM_OBJECT_ROT = 3,               /* rewards.py:94-139 */
  LG_TERM_OBJECT_ROT_DELTA = 4,         /* rewards.py:142-184 */
  LG_TERM_OBJECT_MOVE = 5,              /* rewards.py:65-91 */
  LG_TERM_KEYPOINT = 6                  /* extension, no reference code (SURVEY.md §8c) */
};

enum LgCommandMode { LG_CMD_POSITION = 0, LG_CMD_TORQUE = 1, LG_CMD_POSITION_IMPEDANCE = 2 };
enum LgResetKind { LG_RESET_NONE = 0, LG_RESET_DEFAULT = 1, LG_RESET_RANDOM = 2 };
/* Where reset and goal samples come from (LgParams.rng_stream):
 *   LG_RNG_PHILOX  the library's own Philox stream keyed by (seed, global env id, purpose, epoch): sharding-invariant;
 *   LG_RNG_TORCH   the elements torch.rand / torch.randn on this CUDA device would return for the reference's own
 *                  calls (LgTorchRng): a seeded run samples what a seeded reference run samples.  One shard only. */
enum LgRngStream { LG_RNG_PHILOX = 0, LG_RNG_TORCH = 1 };

/* slots of the statistics vector (sums over the envs of this shard; the reference's
 * `_step_info` means are sum / num_envs — trifinger_env.py:554, :1067-1068, :1076, :1098-1099) */
enum LgStat {
  LG_STAT_TERM0 = 0,            /* .. LG_STAT_TERM0 + 6: per-term reward means (6 = keypoint extension) */
  LG_STAT_POSITION_GOAL = 7,    /* count of envs within the position tolerance         */
  LG_STAT_ORIENTATION_GOAL = 8, /* count of envs within the orientation tolerance      */
  LG_STAT_SUCCESSES = 9,        /* count of set `_successes` flags                     */
  LG_STAT_REWARD = 10,          /* sum of the total reward                             */
  LG_STAT_RESETS = 11,          /* count of `_reset_buf` flags after the timeout check */
  LG_STAT_DONES = 12            /* count of dones                                      */
};

/* Extension (no reference code): slots of LgBuffers.episode_stats, the episodes that ended by a reset (any route but
 * a goal-only reset) and were first seen by this lg_post_physics call.  Sums over the envs of this shard. */
#define LG_NUM_EPISODE_STATS 4
enum LgEpisodeStat {
  LG_EPISODE_COUNT = 0,         /* finished episodes                                   */
  LG_EPISODE_RETURN_SUM = 1,    /* sum of their returns (sum of fp32 rewards)          */
  LG_EPISODE_LENGTH_SUM = 2,    /* sum of their lengths in steps                       */
  LG_EPISODE_SUCCESSES = 3      /* how many ended with `_successes` set                */
};

/* Extension (no reference code): slots of a per-term episode return row (LgBuffers.episode_term_return,
 * last_episode_term_return, episode_term_stats): slot k < 7 is reward term k (LgTerm order), then the success bonus. */
#define LG_NUM_EPISODE_TERMS 8
enum { LG_EPISODE_TERM_BONUS = 7 };

typedef struct LgRewardTerm {
  int32_t activate;    /* RewardTerm.activate (utils/mdp.py:11-33)                        */
  int32_t _pad;
  double weight;       /* RewardTerm.weight                                               */
  double sched_start;  /* thresh_sched_start | linear_schedule_start (rewards.py:46, :158) */
  double sched_end;    /* thresh_sched_end   | linear_schedule_end                         */
  double scale;        /* object_rot.scale (rewards.py:109); keypoint: lgsk scale          */
  double eps;          /* keypoint: lgsk epsilon                                          */
} LgRewardTerm;

/* Everything the kernels need from the env config (SURVEY.md §A.6). Plain data, passed by value. */
typedef struct LgParams {
  /* ---- hot block: everything the per-step kernels read on their critical path sits in the first
   * 160 bytes (two constant-cache lines), ahead of the cold tables ---- */
  int64_t num_envs;         /* envs held by this process (the shard)                            */
  int64_t env_offset;       /* global index of local env 0 (sharding; keys the RNG)             */
  int64_t global_num_envs;  /* env count of the whole job: env_steps_count = frames x this
                               (envs/env_base.py:286-289)                                       */
  int64_t episode_length;   /* config["episode_length"]; < 0 encodes None (env_base.py:393)      */
  int32_t action_dim;       /* 9, or 18 for position_impedance (trifinger_env.py:277)            */
  int32_t asymmetric_obs;   /* fill the states buffer (trifinger_env.py:1026)                    */
  int32_t normalize_obs;    /* apply scale_transform (trifinger_env.py:981-994)                  */
  int32_t normalize_action; /* unscale the action in pre_step (trifinger_env.py:449-457)         */
  int32_t command_mode;     /* LgCommandMode (trifinger_env.py:460-478)                          */
  int32_t apply_safety_damping; /* trifinger_env.py:486-494                                      */
  int32_t task_difficulty;  /* -1, 1..6 (trifinger_env.py:1211-1246)                             */
  int32_t robot_reset;      /* LgResetKind (trifinger_env.py:1119-1144)                          */
  int32_t object_reset;     /* LgResetKind (trifinger_env.py:1164-1177)                          */
  int32_t goal_rotation;    /* goal_movement.rotation.activate (trifinger_env.py:1248-1253)      */
  int32_t success_activate; /* termination_conditions.success.activate (trifinger_env.py:1088)   */
  int32_t control_decimation;
  /* simulator layout (trifinger_env.py:811-825, :881-883; SURVEY.md §A.1) */
  int32_t bodies_per_env;   /* 20 */
  int32_t actors_per_env;   /* 4  */
  int32_t fingertip_body[3];/* 6, 11, 16 */
  int32_t robot_slot, object_slot, goal_slot; /* 0, 2, 3 */
  /* wrapper clipping (wrappers/vec_task.py:146-170); used only for the *_clipped outputs */
  float clip_obs, clip_actions;
  int32_t clip_input_actions; /* clamp the incoming action to +-clip_actions (vec_task.py:162) */
  int32_t dr_activate;      /* extension: domain-randomisation noise (all sigmas zero = off)    */
  int32_t inject_draws;     /* test hook: read uniforms/normals from LgBuffers.inject_* */
  int32_t use_device_clock; /* frame count and reward coefficients come from device memory
                               (LgControl / LgBuffers.reward_coef): CUDA-graph replay           */
  int32_t fuse_bookkeeping; /* lg_post_physics also does steps += 1, timeout and dones
                               (env_base.py:391-399); 0 = _post_step semantics only              */
  int32_t term_active_mask; /* bit k = terms[k].activate                                        */
  uint64_t seed;
  int64_t stats_num_envs;   /* denominator of the statistics means; 0 = num_envs.  Lets a caller run the
                               post-physics pass over sub-ranges of a shard (chunked host pipeline)      */
  /* ---- cold block ---- */
  double dt;                /* config["sim"]["dt"]                                               */
  double success_bonus, position_tolerance, orientation_tolerance;
  double dof_pos_stddev, dof_vel_stddev, goal_rate_magnitude;
  LgRewardTerm terms[LG_NUM_TERMS];
  /* scale_transform tables (utils/torch_utils.py:18-36): centre = (lo+hi)*0.5 and
   * span = hi-lo, both evaluated in fp32 on the host; first obs_dim entries double as
   * the observation table (trifinger_env.py:663-710) */
  float scale_centre[LG_MAX_STATE_DIM];
  float scale_span[LG_MAX_STATE_DIM];
  float scale_rcp[LG_MAX_STATE_DIM];   /* fp32(1/span), correctly rounded: lets the kernel divide in 3 instructions */
  /* pre_step tables (trifinger_env.py:442-498) */
  float action_low[LG_MAX_ACTION_DIM], action_high[LG_MAX_ACTION_DIM];
  float kp[9], kd[9], safety_kd[9];
  float torque_low[9], torque_high[9];
  float dof_default_pos[9], dof_default_vel[9];
  /* cube geometry (envs/trifinger/utils.py:54-131), python doubles as the reference holds them */
  double cube_half_size, cube_radius_3d, cube_max_height, max_com_distance;
  float dr_action_sigma;
  float dr_sigma[LG_MAX_STATE_DIM];
  int32_t _pad_tail;
  int32_t rng_stream;       /* LgRngStream                                                          */
  int32_t sm_count;         /* LG_RNG_TORCH: the device's multiProcessorCount and                   */
  int32_t threads_per_sm;   /* maxThreadsPerMultiProcessor, which fix torch's launch grid           */
  int32_t _pad_tail2;
  /* extension (no reference code): per-episode domain-randomisation offsets, drawn when an env is reset (any route
   * but a goal-only reset) into LgBuffers.obs_bias / action_bias and added to the raw actor observation and to the
   * action on every step of the episode.  sigma = 0 switches a column off; all zero = off.  Nonzero sigmas need
   * dr_activate. */
  float dr_bias_sigma[64];    /* sigma of the offset of raw obs column c (c < obs_dim = 32 + action_dim)   */
  uint64_t dr_bias_mask;    /* bit c set exactly where dr_bias_sigma[c] != 0 (obs_dim <= 50 < 64)                  */
  float dr_action_bias_sigma; /* sigma of the offset of every action column                                        */
  int32_t _pad_tail3;
} LgParams;

/* Scalar coefficients of the reward terms for ONE value of env_steps_count: the Python-float
 * arithmetic of the reward modules (weights x schedule gates x dt, rewards.py:56-63, :123-139, :169-184),
 * rounded to fp32 where the reference hands the scalar to an fp32 tensor op.  Computed on the host by
 * lg_post_physics, or on the device by lg_pre_physics when P.use_device_clock is set. */
#define LG_NUM_COEF 20
typedef struct LgCoef { float v[LG_NUM_COEF]; } LgCoef;

/* Device-resident control block (one per env shard; zero-initialised by the caller). */
typedef struct LgControl {
  uint64_t rng_epoch;     /* RNG epoch of lg_reset_envs / lg_goal_reset_envs, advanced once per call       */
  int64_t frame_count;    /* simulator frames; advanced by lg_pre_physics when P.use_device_clock  */
  uint32_t scan_ticket;   /* tile ticket dispenser of the ordered compaction                        */
  uint32_t scan_epoch;    /* validity tag of the look-back status words; advances once per compaction
                             launch and doubles as the RNG epoch of the fused resets                */
  uint32_t scan_readers;  /* direct-prefix variant of lg_pre_physics: tiles that have read their predecessors' flags */
  uint32_t scan_exits;    /* ... and tiles that have finished; the last one re-arms both and advances scan_epoch   */
} LgControl;

/* State of torch's CUDA Philox generator as LG_RNG_TORCH draws from it (device-resident, one per env).  `seed` and
 * `offset` are what torch.cuda.manual_seed / Generator.get_offset() hold; every launch that draws advances `offset` as
 * the reference's calls would.  The rest is workspace of lg_pre_physics (zero-initialise it). */
typedef struct LgTorchRng {
  uint64_t seed;
  uint64_t offset;
  uint64_t launch_base;     /* offset the current lg_pre_physics launch draws from                  */
  int32_t launch_counts[2]; /* its reset / goal-reset list lengths                                  */
  uint32_t acc[2];          /* counting launch: running list lengths (re-armed to 0)                */
  uint32_t ticket;          /* counting launch: CTAs done (re-armed to 0)                           */
  uint32_t _pad;
} LgTorchRng;

/* The simulator-owned tensors (zero-copy views in the reference, trifinger_env.py:602-617). */
typedef struct LgSimState {
  float* dof_state;         /* [N, 9, 2]                 read; written by resets               */
  float* root_state;        /* [actors_per_env*N, 13]    read; written by resets               */
  const float* rigid_body;  /* [N, bodies_per_env, 13]   read                                  */
  const float* dof_force;   /* [N, 9]   asymmetric only (may be NULL otherwise)                */
  const float* ft_sensors;  /* [N, 18]  asymmetric only (may be NULL otherwise)                */
} LgSimState;

/* The env-owned buffers (envs/env_base.py:560-572, trifinger_env.py:336, :588-590). */
typedef struct LgBuffers {
  float* obs;               /* _obs_buf    [N, obs_dim]                                         */
  float* states;            /* _states_buf [N, state_dim]   (NULL when symmetric)               */
  float* obs_clipped;       /* optional: clamp(obs, +-clip_obs)     (vec_task.py:167)           */
  float* states_clipped;    /* optional: clamp(states, +-clip_obs)  (vec_task.py:147)           */
  float* action;            /* _action_buf [N, A]                                               */
  float* reward;            /* _reward_buf [N]                                                  */
  uint8_t* reset;           /* _reset_buf  [N] bool                                             */
  uint8_t* goal_reset;      /* _goal_reset_buf [N] bool                                         */
  uint8_t* successes;       /* _successes  [N] bool                                             */
  uint8_t* dones;           /* reset & goal_reset [N] bool (env_base.py:399)                    */
  int64_t* steps_count;     /* _steps_count_buf [N]                                             */
  float* goal_pose;         /* _object_goal_poses_buf [N, 7]                                    */
  float* goal_movement;     /* _object_goal_movement_buf [N, 6]                                 */
  float* history;           /* [N, 16] previous fingertip positions (9) + object pose (7): the
                               only columns of history entry 1 the path reads (SURVEY.md a24)  */
  float* applied_torque;    /* optional [N, 9]: what set_dof_actuation_force_tensor receives    */
  float* term_rewards;      /* optional [LG_NUM_TERMS, N]: every term's value (parity tests)    */
  double* step_stats;       /* [LG_NUM_STATS] this shard's `_step_info`: means of the reward terms, of the
                               total reward and of `_successes`, counts for the rest.  Zeroed by
                               lg_pre_physics, accumulated (fp64 RED) by lg_post_physics              */
  /* compaction outputs (env_base.py:374-379, trifinger_env.py:413-416, :435-436) */
  int64_t* reset_ids;       /* [N] ascending env ids with _reset_buf set                        */
  int64_t* goal_reset_ids;  /* [N] ascending env ids with _goal_reset_buf set                   */
  int32_t* counts;          /* [2] number of valid entries in reset_ids / goal_reset_ids        */
  int32_t* robot_indices;   /* [N]  int32 actor indices for set_dof_state_tensor_indexed        */
  int32_t* reset_root_indices; /* [3N] unique(cat(robot,object,goal)) for the reset envs        */
  int32_t* goal_root_indices;  /* [N]  goal actor indices for the goal-reset envs               */
  uint64_t* scan_status;    /* [lg_scan_tiles(N)] look-back status words (workspace)            */
  LgControl* control;
  float* reward_coef;       /* [LG_NUM_COEF] device copy of LgCoef, written by lg_pre_physics when
                               P.use_device_clock (optional otherwise)                              */
  const float* scale_table; /* [4, LG_MAX_STATE_DIM] device copy of P.scale_centre | scale_span | scale_rcp |
                               dr_sigma (coalesced reads; the parameter block is a constant bank)    */
  /* test hook (P.inject_draws): canonical draw arrays indexed by compaction rank */
  const float* inject_reset_u;  /* [k, 24] robot noise 0:18 | object r,theta,yaw | goal u0,u1,u2 */
  const float* inject_reset_n;  /* [k, 8]  goal quaternion 0:4 | ang-vel axis 4:7 | magnitude 7  */
  const float* inject_goal_u;   /* same layouts for the goal-reset list                          */
  const float* inject_goal_n;
  /* optional bfloat16 copies of the outputs for the policy / value networks (SURVEY.md 8 f2): round-to-nearest-even
     of the clipped values when obs_clipped / states_clipped are requested, else of obs / states */
  uint16_t* obs_bf16;       /* [N, obs_dim]   */
  uint16_t* states_bf16;    /* [N, state_dim] */
  /* optional [N] bool masks OR-ed into _reset_buf / _goal_reset_buf by lg_pre_physics before the compaction: what a
     caller does with `env._reset_buf |= mask` between steps (tests, reset-heavy workloads), without a separate pass */
  const uint8_t* force_reset;
  const uint8_t* force_goal_reset;
  /* optional episode statistics (extension, no reference code): all five or none.  lg_post_physics adds each env's
     reward to its running return; every reset of an env with steps_count > 0 (lg_pre_physics, lg_reset_envs; not a
     goal-only reset) moves the return, steps_count and _successes into the env's record and zeroes the return; the
     first lg_post_physics after the reset adds the record into episode_stats (zeroed where step_stats is) */
  float* episode_return;          /* [N] return of the running episode                                  */
  float* last_episode_return;     /* [N] record of the env's last finished episode: return              */
  int64_t* last_episode_length;   /* [N]   its length in steps (0: none finished yet)                   */
  uint8_t* last_episode_success;  /* [N]   _successes when it ended                                      */
  double* episode_stats;          /* [LG_NUM_EPISODE_STATS] LgEpisodeStat sums of the episodes reported  */
  /* optional per-term episode returns (extension, no reference code): all three or none, and only with the five
     episode buffers above; the two row arrays 16-byte aligned.  lg_post_physics adds each active term's value (and the
     success bonus when it is paid) to the env's running row; the same resets that end an episode move the row into
     the env's record and zero it; the first lg_post_physics after the reset adds the record into episode_term_stats
     (zeroed where episode_stats is) */
  float* episode_term_return;       /* [N, LG_NUM_EPISODE_TERMS] running episode, per term + success bonus     */
  float* last_episode_term_return;  /* [N, LG_NUM_EPISODE_TERMS] record of the env's last finished episode     */
  double* episode_term_stats;       /* [LG_NUM_EPISODE_TERMS] sums of the records of the episodes reported    */
  /* per-episode domain-randomisation offsets (extension, no reference code; LgParams.dr_bias_sigma /
     dr_action_bias_sigma).  Required when the matching sigmas are nonzero, otherwise ignored.  Every reset of an env
     (lg_pre_physics, lg_reset_envs; not a goal-only reset) redraws its rows: sigma x a standard normal of this build's
     Philox stream keyed by (seed, global env id, epoch of the reset's own draws), never torch's stream or injected
     draws; columns with sigma = 0 hold +0.0.  lg_post_physics / lg_fill_observations add obs_bias to the raw actor
     observation (columns with sigma != 0 only, before the white noise); lg_pre_physics adds action_bias to the
     incoming action before the white noise and the clamp; the rows of the envs it reset are drawn by a small launch
     behind it. */
  float* obs_bias;          /* [N, obs_dim] */
  float* action_bias;       /* [N, action_dim] */
  LgTorchRng* torch_rng;   /* P.rng_stream == LG_RNG_TORCH: the generator state (NULL otherwise)  */
} LgBuffers;

int lg_version(void);
const char* lg_last_error(void);
/* sizeof of the ABI structs, for binding self-checks: 0 LgParams, 1 LgSimState, 2 LgBuffers,
 * 3 LgControl, 4 LgRewardTerm, 5 LgHostStep */
size_t lg_struct_size(int which);

/* Hint for the device-wide L2 fetch granularity (cudaLimitMaxL2FetchGranularity): the path gathers 52-byte
 * simulator rows, for which 32-byte fetches cut the DRAM over-fetch.  bytes in {32, 64, 128}. */
int lg_set_l2_fetch_granularity(int bytes);


/* number of look-back status words lg_pre_physics needs for n envs */
int64_t lg_scan_tiles(int64_t num_envs);
/* Largest tile count whose pre-physics CTAs are all co-resident on the current device (occupancy of the kernel x SM
 * count).  Shards with more tiles take their tiles by ticket (dispatch order) instead of by block index; results are
 * identical, the value is exposed for tests and capacity planning.  Needs a CUDA device. */
int64_t lg_pre_resident_tiles(void);

/*
 * Everything IsaacEnvBase.step does BEFORE physics (envs/env_base.py:369-381), one launch:
 *   _action_buf = clamp?(action_in)                         env_base.py:369, vec_task.py:162
 *   env_ids = nonzero(_reset_buf), goal ids likewise          env_base.py:374-379  (ordered compaction)
 *   _reset_impl(env_ids); _goal_reset_impl(goal_env_ids)      trifinger_env.py:373-440, :1101-1265,
 *                                                             samplers envs/trifinger/sample.py:22-84
 *   _pre_step(): action -> torque                             trifinger_env.py:442-498
 * `action_in` [N, A] may alias B->action.
 */
int lg_pre_physics(const LgParams* P, const LgSimState* S, const LgBuffers* B,
                   const float* action_in, void* stream);
/*
 * The same pass for a caller whose inputs are ready early.  Contract: `action_in` and `S->dof_state` were complete
 * before the lg_post_physics call that precedes this call on `stream` started to execute, and nothing writes them
 * until this call has finished (a rollout that draws its actions from a buffer, an asynchronous policy; NOT the
 * synchronous loop obs -> policy -> action).  The launch is then chained to that lg_post_physics programmatically:
 * the grid becomes resident and fetches the action / joint-state slabs while the post-physics pass is still
 * finishing, and reads everything that pass writes only after it has completed (16 384 envs: 10.6 -> 10.3 us/step).
 * If the library call preceding this one on the calling thread was not lg_post_physics on the same stream, the call
 * is plain lg_pre_physics.  `exclusive_sm` != 0 reserves a whole SM per CTA (grids of 32..128 tiles): CTAs of a grid
 * that starts early pile up on the SMs that drain first, which slows reset-heavy steps (30 % of the envs resetting:
 * 16.7 instead of 15.5 us/step; 15.1 with the SM reserved); costs 0.25 us/step when hardly anything resets.
 */
int lg_pre_physics_chained(const LgParams* P, const LgSimState* S, const LgBuffers* B,
                           const float* action_in, int exclusive_sm, void* stream);

/*
 * Everything after physics, one launch: _post_step (trifinger_env.py:500-559) =
 * _fill_observations_and_states (:959-1051) + six reward terms (rewards.py) + accumulation and
 * per-term means (:551-554) + __check_termination (:1053-1099), then the step counter, timeout
 * and dones of IsaacEnvBase.step (env_base.py:391-399) and the step statistics (plus, with
 * LgBuffers.episode_return, the running returns and the finished-episode statistics).
 * `sched_step` is env_steps_count (env_base.py:286-289); ignored when P->use_device_clock.
 */
int lg_post_physics(const LgParams* P, const LgSimState* S, const LgBuffers* B,
                    double sched_step, void* stream);

/* _fill_observations_and_states alone (what IsaacEnvBase.reset runs, env_base.py:340):
 * history shift + obs/states, no reward, no termination, no counters. */
int lg_fill_observations(const LgParams* P, const LgSimState* S, const LgBuffers* B, void* stream);

/* history seeding of TrifingerEnv.__initialize (trifinger_env.py:619-628) */
int lg_init_history(const LgParams* P, const LgSimState* S, const LgBuffers* B, void* stream);

/* mask -> ascending int64 ids (torch.nonzero(mask).view(-1), env_base.py:374/377).
 * count_out: device int32.  status: lg_scan_tiles(n) words of workspace; control as above. */
int lg_compact(const uint8_t* mask, int64_t n, int64_t* ids_out, int32_t* count_out,
               uint64_t* status, LgControl* control, void* stream);

/* The hooks on an explicit id list (`instances` of trifinger_env.py:373 / :425).  `k_host` ids
 * are read from the device array `ids` (int64, any order, no duplicates). */
int lg_reset_envs(const LgParams* P, const LgSimState* S, const LgBuffers* B,
                  const int64_t* ids, int64_t k_host, void* stream);
int lg_goal_reset_envs(const LgParams* P, const LgSimState* S, const LgBuffers* B,
                       const int64_t* ids, int64_t k_host, void* stream);

/* torch's CUDA uniform / normal stream as a batched primitive: out[0..n) = what torch.rand(n) (normal == 0) or
 * torch.randn(n) (normal != 0) returns in fp32 on the current device for a generator with this seed and Philox
 * offset (a multiple of 4).  Advances nothing.  n < 2^31. */
int lg_torch_philox(uint64_t seed, uint64_t offset, int64_t n, int normal, float* out, void* stream);
/* Host only: how far such a call advances the generator's offset on a device with `sm_count` SMs of
 * `threads_per_sm` threads (0 for n == 0). */
uint64_t lg_torch_philox_advance(int64_t n, int32_t sm_count, int32_t threads_per_sm);

/* _pre_step alone (trifinger_env.py:442-498) on the current _action_buf */
int lg_pre_step(const LgParams* P, const LgSimState* S, const LgBuffers* B, void* stream);

/* Batched math primitives of utils/torch_utils.py and rewards.py:20-34 (n rows). */
int lg_quat_mul(const float* a, const float* b, float* out, int64_t n, void* stream);       /* :83-113  */
int lg_quat_diff_rad(const float* a, const float* b, float* out, int64_t n, void* stream);  /* :131-150 */
int lg_scale_transform(const float* x, const float* lower, const float* upper, float* out,
                       int64_t n, int32_t dims, void* stream);                              /* :18-36   */
int lg_unscale_transform(const float* x, const float* lower, const float* upper, float* out,
                         int64_t n, int32_t dims, void* stream);                            /* :39-57   */
int lg_saturate(const float* x, const float* lower, const float* upper, float* out,
                int64_t n, int32_t dims, void* stream);                                     /* :60-75   */
int lg_lgsk_kernel(const float* x, float scale, float* out, int64_t n, void* stream);       /* rewards.py:20-34 */

/* Self-test of the kernels' fast division by `span` (with `rcp` = fp32(1/span)) over all 2^32 numerators.
 * out_dev[0] = numerators with 2^-100 <= |x| < 2^100 or x = 0 whose quotient is not bit-identical to IEEE
 * x / span (expected 0); out_dev[1] = worst ulp distance for 0 < |x| < 2^-100 (expected <= 1);
 * out_dev[2] = numerators >= 2^100 / inf the range guard failed to flag (expected 0).  out_dev: 3 x uint64. */
int lg_selftest_division(float span, float rcp, unsigned long long* out_dev, void* stream);

/* Extension (no reference code): world-frame cube corners, [n,7] poses -> [n,8,3] keypoints. */
int lg_cube_keypoints(const float* pose, float cube_size, float* out, int64_t n, void* stream);

/* Extension (stand-in for PhysX integrating the moving-goal task's goal body, SURVEY.md 8 f3): advances the goal
 * actor's root rows of S->root_state by dt -- p += v dt, q <- normalize(exp(w dt / 2) (x) q), w = world-frame
 * angular velocity (cols 10:13, re-imposed each step by lg_pre_physics / lg_pre_step, trifinger_env.py:1267-1277). */
int lg_integrate_goal(const LgParams* P, const LgSimState* S, float dt, void* stream);

/*
 * Host-buffer convenience entry for callers whose simulator state lives in HOST memory
 * (the reference's default `use_gpu_pipeline: False`, env_base.py:60): copies the five
 * simulator tensors and the action host->device, runs lg_pre_physics + lg_post_physics and
 * copies obs / reward / dones (and states when asymmetric) device->host, all on `stream`.
 * Host pointers should be pinned; outputs are valid after the stream is synchronised.
 */
typedef struct LgHostStep {
  const float* dof_state_host; const float* root_state_host; const float* rigid_body_host;
  const float* dof_force_host; const float* ft_sensors_host; const float* action_host;
  float* obs_host; float* states_host; float* reward_host; uint8_t* dones_host;
  /* obs_host may be NULL when asymmetric_obs && !dr_activate: the observation is then the first obs_dim columns
     of every states_host row (same values; ref trifinger_env.py:995-1051) and is not transferred a second time */
  float* action_staging;    /* device [N, A] scratch for the uploaded action */
} LgHostStep;
/* Host -> device staging of one simulator state (pinned host pointers of H; outputs of H unused): the whole
 * dof_state / dof_force / ft_sensors tensors; of root_state only the object actor's rows and of rigid_body only
 * the three fingertip bodies (strided 2-D copies of 52-byte rows) -- the rows lg_post_physics reads. */
int lg_upload_sim_state(const LgParams* P, const LgSimState* S, const LgHostStep* H, void* stream);
int lg_step_host(const LgParams* P, const LgSimState* S, const LgBuffers* B,
                 const LgHostStep* H, double sched_step, void* stream);

/*
 * lg_step_host with the shard cut into `chunks` env ranges and pipelined over three streams: uploads on
 * `stream_up`, kernels on `stream_main`, downloads on `stream_down` (PCIe is full duplex, so the upload of range
 * c+1 overlaps the kernels of range c and the download of range c-1).  lg_pre_physics runs once over the whole
 * shard (its ordered compaction spans it); lg_post_physics runs per range on offset pointers.  All outputs are
 * valid once `stream_main` is synchronised.  Results are identical to lg_step_host.
 */
int lg_step_host_pipelined(const LgParams* P, const LgSimState* S, const LgBuffers* B, const LgHostStep* H,
                           double sched_step, int chunks, void* stream_main, void* stream_up, void* stream_down);

#ifdef __cplusplus
}
#endif
#endif /* LEIBNIZ_B200_H_ */
