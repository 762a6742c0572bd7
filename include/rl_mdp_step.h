/*
 * rl_mdp_step.h - C-ABI of the B200-native per-step MDP pipeline (observation / reward /
 * termination / command / joint-position-action terms of robot_lab's velocity-locomotion tasks).
 *
 * What each entry point replaces in the reference (paths relative to /root/reference; V/ =
 * source/robot_lab/robot_lab/tasks/manager_based/locomotion/velocity/; [IL] = IsaacLab v2.3.2 code the
 * reference calls but does not vendor, restated in SURVEY.md Appendix A):
 *
 *   rl_process_action   ActionManager.process_action + JointPositionAction.process_actions [IL]
 *                       (configured at V/velocity_env_cfg.py:124-126, GO2/rough_env_cfg.py:51-53)
 *   rl_step             TerminationManager.compute + RewardManager.compute + CommandManager.compute +
 *                       ObservationManager.compute [IL] looping over the term functions of
 *                       V/mdp/rewards.py:22-687, V/mdp/observations.py:17-35, V/mdp/commands.py:22-85 and the
 *                       upstream terms wired at V/velocity_env_cfg.py:134-254,379-664, in the order of
 *                       ManagerBasedRLEnv.step() [IL] (SURVEY.md section 3.2), plus reset_buf.nonzero()
 *   rl_reset_envs       the manager part of ManagerBasedRLEnv._reset_idx [IL]: episode-sum / metric logging
 *                       means, zeroing, command resample (V/mdp/commands.py:43-47), action reset
 *   rl_term_eval        one reward term function called on its own: func(env, **params) -> Tensor[N]
 *                       (term protocol, V/mdp/rewards.py:22 ff.)
 *   neighbours of the path (SURVEY.md 8(f)):
 *   rl_contact_sensor_update   ContactSensor._update_buffers_impl [IL] (V/velocity_env_cfg.py:86,726)
 *   rl_reset_scene_state       reset_root_state_uniform (V/mdp/events.py:205-271) + reset_joints_by_scale [IL]
 *   rl_actuator_step           Articulation._apply_actuator_model [IL] with the DCMotor / IdealPD / Implicit
 *                              actuator models the reference selects at assets/unitree.py:55-63,107-115,504-575
 *   rl_is_robot_on_terrain     is_robot_on_terrain (V/mdp/utils.py:73-127)
 *   rl_command_pit_restrict    the terrain-aware tail of UniformThresholdVelocityCommand._update_command
 *                              (V/mdp/commands.py:61-85)
 *   rl_height_scan_cast        the grid-pattern RayCaster [IL] (V/velocity_env_cfg.py:70-77) over a height-field
 *                              terrain: produces ray_hits_z / ray_sensor_pos_z for the height_scan observation
 *   rl_interval_push           EventManager.reset / apply("interval") [IL] for one non-global interval term running
 *                              push_by_setting_velocity [IL] (randomize_push_robot, V/velocity_env_cfg.py:366-371)
 *
 * Conventions: every function returns 0 on success or a negative RL_E* code; rl_last_error() gives the
 * message (thread-local). All data pointers are DEVICE pointers borrowed for the duration of the call;
 * the caller (PyTorch) owns every tensor, the library owns only the opaque context. Launches are
 * asynchronous on the given cudaStream_t and never synchronise. One context per GPU; a context is not
 * thread-safe, different contexts are independent. No torch types cross this boundary.
 */
#ifndef RL_MDP_STEP_H_
#define RL_MDP_STEP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RL_ABI_VERSION 13

#define RL_MAX_JOINTS 64
#define RL_MAX_BODIES 64        /* bodies in the contact-force history tensor                  */
#define RL_MAX_TIME_BODIES 64   /* bodies in the air/contact-time tensors                       */
#define RL_MAX_ASSET_BODIES 64  /* bodies in the body_pos_w / body_lin_vel_w tensors            */
#define RL_MAX_REWARD_TERMS 48
#define RL_MAX_OBS_TERMS 12
#define RL_MAX_DONE_TERMS 8
#define RL_MAX_IDX 32
#define RL_MAX_TASKS 112       /* entries of the static work schedule (debug interface) */
#define RL_DEBUG_STRIDE 160     /* int64 words per CTA in the debug buffer */
#define RL_NUM_OBS_GROUPS 2     /* 0 = policy, 1 = critic                                        */
#define RL_NUM_CMD_UNIFORMS 7   /* time_left, vx, vy, wz, heading, is_heading, is_standing       */
#define RL_NUM_INTERVAL_UNIFORMS 8 /* rl_interval_push: timer on reset, timer on fire, 6 velocities */

enum RlError {
  RL_OK = 0,
  RL_EINVAL = -1,   /* bad argument / inconsistent spec */
  RL_ECUDA = -2,    /* CUDA runtime error               */
  RL_ENOMEM = -3,
  RL_EUNSUPPORTED = -4
};

/* Reward term kinds. The comment names the reference function each one restates. */
enum RlRewardType {
  RL_REW_NONE = 0,
  RL_REW_IS_TERMINATED = 1,              /* [IL] mdp.is_terminated                               */
  RL_REW_LIN_VEL_Z_L2 = 2,               /* V/mdp/rewards.py:647                                  */
  RL_REW_ANG_VEL_XY_L2 = 3,              /* :656                                                  */
  RL_REW_FLAT_ORIENTATION_L2 = 4,        /* :678                                                  */
  RL_REW_BASE_HEIGHT_L2 = 5,             /* :616 (sensor_cfg=None branch only)                    */
  RL_REW_JOINT_TORQUES_L2 = 6,           /* [IL] mdp.joint_torques_l2                             */
  RL_REW_JOINT_VEL_L2 = 7,               /* [IL] mdp.joint_vel_l2                                 */
  RL_REW_JOINT_ACC_L2 = 8,               /* [IL] mdp.joint_acc_l2                                 */
  RL_REW_JOINT_DEVIATION_L1 = 9,         /* [IL] mdp.joint_deviation_l1                           */
  RL_REW_JOINT_POS_LIMITS = 10,          /* [IL] mdp.joint_pos_limits                             */
  RL_REW_JOINT_VEL_LIMITS = 11,          /* [IL] mdp.joint_vel_limits                             */
  RL_REW_JOINT_POWER = 12,               /* :81                                                   */
  RL_REW_STAND_STILL = 13,               /* :93                                                   */
  RL_REW_JOINT_POS_PENALTY = 14,         /* :107                                                  */
  RL_REW_JOINT_MIRROR = 15,              /* :259                                                  */
  RL_REW_ACTION_MIRROR = 16,             /* :281                                                  */
  RL_REW_ACTION_SYNC = 17,               /* :306                                                  */
  RL_REW_ACTION_RATE_L2 = 18,            /* [IL] mdp.action_rate_l2                               */
  RL_REW_UNDESIRED_CONTACTS = 19,        /* :665                                                  */
  RL_REW_CONTACT_FORCES = 20,            /* [IL] mdp.contact_forces                               */
  RL_REW_TRACK_LIN_VEL_XY_EXP = 21,      /* :22                                                   */
  RL_REW_TRACK_ANG_VEL_Z_EXP = 22,       /* :38                                                   */
  RL_REW_TRACK_LIN_VEL_XY_YAW_FRAME_EXP = 23, /* :51                                              */
  RL_REW_TRACK_ANG_VEL_Z_WORLD_EXP = 24, /* :69                                                   */
  RL_REW_FEET_AIR_TIME = 25,             /* :340                                                  */
  RL_REW_FEET_AIR_TIME_POSITIVE_BIPED = 26, /* :363                                               */
  RL_REW_FEET_AIR_TIME_VARIANCE = 27,    /* :386                                                  */
  RL_REW_FEET_GAIT = 28,                 /* :156-256 (GaitReward)                                 */
  RL_REW_FEET_CONTACT = 29,              /* :400                                                  */
  RL_REW_FEET_CONTACT_WITHOUT_CMD = 30,  /* :416                                                  */
  RL_REW_FEET_STUMBLE = 31,              /* :428                                                  */
  RL_REW_FEET_SLIDE = 32,                /* :557                                                  */
  RL_REW_FEET_HEIGHT = 33,               /* :507                                                  */
  RL_REW_FEET_HEIGHT_BODY = 34,          /* :527                                                  */
  RL_REW_FEET_DISTANCE_Y_EXP = 35,       /* :439                                                  */
  RL_REW_FEET_DISTANCE_XY_EXP = 36,      /* :464                                                  */
  RL_REW_UPWARD = 37,                    /* :608                                                  */
  RL_REW_WHEEL_VEL_PENALTY = 38,         /* :132                                                  */
  RL_REW_TYPE_COUNT = 39
};

/*
 * One reward term: func + weight + params of the reference's RewardTermCfg, with every name/regex
 * already resolved to indices. Parameter slots p[] per type:
 *   TRACK_*_EXP                    p0 = std**2
 *   STAND_STILL                    p0 = command_threshold
 *   JOINT_POS_PENALTY              p0 = stand_still_scale, p1 = velocity_threshold, p2 = command_threshold
 *   JOINT_MIRROR / ACTION_MIRROR   idx_a[i] <-> idx_b[i] (n_idx joint pairs), p0 = 1/len(mirror_joints)
 *   ACTION_SYNC                    idx_a = action columns, grouped: idx_b[g] = group start in idx_a,
 *                                  idx_c[g] = group size, n_idx = #groups, p0 = 1/len(joint_groups)
 *   UNDESIRED_CONTACTS             p0 = threshold, body_mask over history bodies
 *   CONTACT_FORCES                 p0 = threshold, body_mask
 *   FEET_AIR_TIME                  p0 = threshold, idx_a = feet in time-body space
 *   FEET_AIR_TIME_POSITIVE_BIPED   p0 = threshold, idx_a
 *   FEET_AIR_TIME_VARIANCE         idx_a
 *   FEET_GAIT                      p0 = std, p1 = max_err**2, p2 = velocity_threshold, p3 = command_threshold,
 *                                  idx_a[0..3] = {pair0[0], pair0[1], pair1[0], pair1[1]} in time-body space
 *   FEET_CONTACT                   p0 = expect_contact_num, idx_a
 *   FEET_CONTACT_WITHOUT_CMD       idx_a
 *   FEET_STUMBLE                   idx_c = feet in history-body space
 *   FEET_SLIDE                     idx_c = feet (history space, contact), idx_b = feet (asset-body space, velocity)
 *   FEET_HEIGHT / _BODY            p0 = target_height, p1 = tanh_mult, idx_b
 *   FEET_DISTANCE_Y_EXP            p0 = stance_width, p1 = std**2, idx_b
 *   FEET_DISTANCE_XY_EXP           p0 = stance_width, p1 = stance_length, p2 = std**2, idx_b (4 feet)
 *   BASE_HEIGHT_L2                 p0 = target_height
 *   JOINT_VEL_LIMITS               p0 = soft_ratio
 *   WHEEL_VEL_PENALTY              p0 = velocity_threshold, p1 = command_threshold, idx_a = wheel bodies in
 *                                  time-body space, idx_b = matching wheel joints (native ids)
 *   joint terms                    joint_mask = native joint ids the term sums over
 */
typedef struct RlRewardTerm {
  int32_t type;
  float weight;
  float p[6];
  uint64_t joint_mask;
  uint64_t body_mask;
  int32_t n_idx;
  int32_t reserved;
  uint8_t idx_a[RL_MAX_IDX];
  uint8_t idx_b[RL_MAX_IDX];
  uint8_t idx_c[RL_MAX_IDX];
} RlRewardTerm;

enum RlObsType {
  RL_OBS_NONE = 0,
  RL_OBS_BASE_LIN_VEL = 1,        /* [IL] root_lin_vel_b                                   */
  RL_OBS_BASE_ANG_VEL = 2,        /* [IL] root_ang_vel_b                                   */
  RL_OBS_PROJECTED_GRAVITY = 3,   /* [IL] projected_gravity_b                              */
  RL_OBS_GENERATED_COMMANDS = 4,  /* [IL] command_manager.get_command                      */
  RL_OBS_JOINT_POS_REL = 5,       /* [IL] joint_pos - default_joint_pos, ids[] order       */
  RL_OBS_JOINT_VEL_REL = 6,       /* [IL] joint_vel - default_joint_vel, ids[] order       */
  RL_OBS_LAST_ACTION = 7,         /* [IL] action_manager.action                            */
  RL_OBS_HEIGHT_SCAN = 8,         /* [IL] sensor z - ray hit z - offset (p0 = offset)      */
  RL_OBS_JOINT_POS_REL_WITHOUT_WHEEL = 9, /* V/mdp/observations.py:17, zero_mask = wheel columns */
  RL_OBS_PHASE = 10,              /* V/mdp/observations.py:30, p0 = cycle_time             */
  RL_OBS_TYPE_COUNT = 11
};

/* ObservationTermCfg: func -> clone -> (+noise) -> clip -> scale (SURVEY 8(a3)). */
typedef struct RlObsTerm {
  int32_t type;
  int32_t dim;
  int32_t has_noise;
  float noise_lo, noise_hi;
  int32_t has_clip;
  float clip_lo, clip_hi;
  int32_t has_scale;
  float scale;
  float p[2];
  uint64_t zero_mask;             /* columns forced to 0 (JOINT_POS_REL_WITHOUT_WHEEL) */
  uint8_t ids[RL_MAX_JOINTS];     /* joint terms: column c reads native joint ids[c]   */
} RlObsTerm;

typedef struct RlObsGroup {
  int32_t n_terms;
  int32_t dim;                    /* sum of term dims = row width */
  int32_t enable_corruption;
  int32_t reserved;
  RlObsTerm terms[RL_MAX_OBS_TERMS];
} RlObsGroup;

enum RlDoneType {
  RL_DONE_NONE = 0,
  RL_DONE_TIME_OUT = 1,               /* [IL] episode_length_buf >= max_episode_length        */
  RL_DONE_TERRAIN_OUT_OF_BOUNDS = 2,  /* [IL] p0 = 0.5*W - buf, p1 = 0.5*H - buf, p2 = is_generator */
  RL_DONE_ILLEGAL_CONTACT = 3,        /* [IL] p0 = threshold, body_mask                       */
  RL_DONE_TYPE_COUNT = 4
};

typedef struct RlDoneTerm {
  int32_t type;
  int32_t time_out;                   /* 1 -> truncated, 0 -> terminated */
  float p[4];
  uint64_t body_mask;
} RlDoneTerm;

/* UniformThresholdVelocityCommandCfg (V/velocity_env_cfg.py:106-117, V/mdp/commands.py:22-92). */
typedef struct RlCommandCfg {
  float resampling_time_lo, resampling_time_hi;
  float rel_standing_envs, rel_heading_envs;
  int32_t heading_command;
  float heading_control_stiffness;
  float lin_vel_x_lo, lin_vel_x_hi;
  float lin_vel_y_lo, lin_vel_y_hi;
  float ang_vel_z_lo, ang_vel_z_hi;
  float heading_lo, heading_hi;
  float small_cmd_threshold;          /* 0.2, V/mdp/commands.py:47 */
  float max_command_step;             /* resampling_time_hi / step_dt [IL] */
} RlCommandCfg;

/* The action terms of the ActionManager [IL], concatenated in declaration order into one action vector:
 * JointPositionActionCfg (V/velocity_env_cfg.py:124-126) and, for the wheeled robots, a second JointVelocityActionCfg
 * term (e.g. V/config/wheeled/unitree_go2w/rough_env_cfg.py:22-32,101-106). Column a drives native joint joint_ids[a]:
 * target = clamp(action * scale + offset, clip), written to the joint POSITION target (target_kind 0, offset =
 * default joint position) or the joint VELOCITY target (target_kind 1, offset = default joint velocity). */
enum RlActionTargetKind { RL_ACTION_JOINT_POSITION = 0, RL_ACTION_JOINT_VELOCITY = 1 };

typedef struct RlActionCfg {
  int32_t n_actions;
  int32_t has_clip;
  uint8_t joint_ids[RL_MAX_JOINTS];
  uint8_t target_kind[RL_MAX_JOINTS];
  float scale[RL_MAX_JOINTS];
  float offset[RL_MAX_JOINTS];
  float clip_lo[RL_MAX_JOINTS];
  float clip_hi[RL_MAX_JOINTS];
} RlActionCfg;

/* The flat, fully resolved description of one task's MDP step (host POD, copied at rl_ctx_create). */
typedef struct RlStepSpec {
  int32_t abi_version;                /* must be RL_ABI_VERSION */
  int32_t num_joints;                 /* J  */
  int32_t num_hist_bodies;            /* B  : bodies in net_forces_w_history                 */
  int32_t hist_len;                   /* T  */
  int32_t num_time_bodies;            /* Bt : bodies in the air/contact-time tensors         */
  int32_t num_asset_bodies;           /* Ba : bodies in body_pos_w / body_lin_vel_w          */
  int32_t num_rays;                   /* R  (0 = no height scanner)                          */
  int32_t num_reward_terms;           /* K  */
  int32_t num_done_terms;
  int32_t max_episode_length;         /* ceil(episode_length_s / step_dt)                    */
  float step_dt;
  float contact_time_abs_tol;         /* 1e-8, ContactSensor.compute_first_contact [IL]      */
  float default_joint_pos[RL_MAX_JOINTS];
  float default_joint_vel[RL_MAX_JOINTS];
  float soft_pos_limit_lo[RL_MAX_JOINTS];
  float soft_pos_limit_hi[RL_MAX_JOINTS];
  float soft_vel_limit[RL_MAX_JOINTS];
  RlRewardTerm rewards[RL_MAX_REWARD_TERMS];
  RlDoneTerm dones[RL_MAX_DONE_TERMS];
  RlObsGroup obs[RL_NUM_OBS_GROUPS];
  RlCommandCfg command;
  RlActionCfg action;
} RlStepSpec;

/*
 * A strided view of one per-env field: element (env, comp) lives at ptr[env*env_stride + comp*comp_stride]
 * (strides in ELEMENTS). SoA [C][N] is {1, N}; AoS [N][C] is {C, 1}. Multi-index fields flatten their
 * trailing dims row-major into comp (history: comp = (t*B + b)*3 + xyz; body vectors: comp = b*3 + xyz).
 */
typedef struct RlField {
  void* ptr;
  int64_t env_stride;
  int64_t comp_stride;
} RlField;

/* Read-only per-step state produced by physics + sensors (SURVEY.md Appendix C). fp32 unless noted. */
typedef struct RlStateView {
  RlField root_pos_w;            /* 3                                       */
  RlField root_quat_w;           /* 4  (w, x, y, z)                         */
  RlField root_lin_vel_w;        /* 3                                       */
  RlField root_ang_vel_w;        /* 3                                       */
  RlField joint_pos;             /* J  native joint order                   */
  RlField joint_vel;             /* J                                       */
  RlField joint_acc;             /* J                                       */
  RlField applied_torque;        /* J                                       */
  RlField net_forces_w_history;  /* T*B*3, index 0 of T = newest            */
  RlField current_air_time;      /* Bt                                      */
  RlField last_air_time;         /* Bt                                      */
  RlField current_contact_time;  /* Bt                                      */
  RlField last_contact_time;     /* Bt                                      */
  RlField body_pos_w;            /* Ba*3                                    */
  RlField body_lin_vel_w;        /* Ba*3                                    */
  RlField ray_hits_z;            /* R   (z of ray_hits_w)                   */
  RlField ray_sensor_pos_z;      /* 1   (z of the ray caster's pos_w)       */
} RlStateView;

/* Manager-owned state that the step reads AND writes. */
typedef struct RlMdpState {
  RlField action;                /* A   action_manager.action       (read by rl_step)    */
  RlField prev_action;           /* A   action_manager.prev_action  (read by rl_step)    */
  RlField command;               /* 3   vel_command_b                                      */
  RlField heading_target;        /* 1                                                      */
  RlField time_left;             /* 1                                                      */
  RlField is_heading_env;        /* 1   uint8                                              */
  RlField is_standing_env;       /* 1   uint8                                              */
  RlField metric_error_vel_xy;   /* 1                                                      */
  RlField metric_error_vel_yaw;  /* 1                                                      */
  RlField episode_length;        /* 1   int32 (int64 at the torch boundary)                */
  RlField episode_sums;          /* K   reward_manager._episode_sums                       */
} RlMdpState;

/* Logging reductions produced at reset (extras["log"] of the reference [IL]). */
typedef struct RlResetLog {
  float* episode_sum_mean;       /* [K]  mean over reset ids of episode_sums (caller divides by
                                         max_episode_length_s as RewardManager.reset does)  */
  float* done_term_count;        /* [RL_MAX_DONE_TERMS] count over reset ids                 */
  float* metric_mean;            /* [2]  error_vel_xy, error_vel_yaw means                   */
} RlResetLog;

/* Outputs of one step. Any pointer may be NULL to skip that output. */
typedef struct RlStepOut {
  float* obs[RL_NUM_OBS_GROUPS]; /* [N, obs_pitch[g]] rows                                 */
  int64_t obs_pitch[RL_NUM_OBS_GROUPS]; /* row pitch in elements (>= group dim)            */
  float* reward;                 /* [N]                                                    */
  uint8_t* terminated;           /* [N]                                                    */
  uint8_t* truncated;            /* [N]                                                    */
  uint8_t* done_bits;            /* [N] bit i = done term i fired                          */
  RlField step_reward;           /* K  reward_manager._step_reward (value / dt)            */
  int32_t* reset_ids;            /* [N] ascending ids with terminated|truncated            */
  int32_t* n_reset;              /* [1]                                                    */
  RlResetLog reset_log;          /* written by RL_PHASE_RESET launches                     */
} RlStepOut;

/* Which manager phases a launch evaluates (bit flags). */
enum RlPhase {
  RL_PHASE_DONES = 1,       /* episode_length += 1, termination terms                       */
  RL_PHASE_REWARDS = 2,     /* reward terms, episode sums, step reward                      */
  RL_PHASE_COMMAND = 4,     /* CommandTerm.compute: metrics, timer, resample, heading update*/
  RL_PHASE_OBS = 8,         /* observation groups                                           */
  RL_PHASE_COMPACT = 16,    /* reset id compaction (ascending)                              */
  RL_PHASE_SKIP_DONE_ENVS = 32, /* COMMAND/OBS only for envs that are not done this step
                                   (they are refreshed after the external reset instead)   */
  RL_PHASE_RESET = 64,      /* manager reset BEFORE the other phases of the launch - logging means
                               (RlStepOut.reset_log), zero episode sums / metrics / actions / episode length,
                               command resample. Combines with COMMAND / OBS only. Two forms:
                               - with env_ids: every env of the list is reset (gathered tiles);
                               - without: all envs are processed and those whose out->terminated |
                                 out->truncated byte is set are reset (out->n_reset = their count, as left by
                                 the DONES | COMPACT launch) - full-tile fast path.
                               RESET|COMMAND|OBS is the whole post-reset part of ManagerBasedRLEnv.step() [IL]
                               in one launch; DONES|REWARDS|COMPACT followed by it reproduces the reference's
                               order terminations -> rewards -> reset -> command -> observations exactly.  */
  RL_PHASE_ALL = 31
};

/* Random inputs. NULL pointers select the in-kernel Philox4x32-10 stream (seed, step, env). */
typedef struct RlRandom {
  uint64_t seed;
  uint64_t step;                 /* step counter: part of the Philox counter                */
  const uint64_t* step_counter;  /* optional DEVICE counter added to `step` (the env's common_step_counter
                                    [IL]); rl_process_action increments it, so a captured CUDA graph
                                    draws fresh noise on every replay                          */
  int64_t env_id_offset;         /* global id of env 0 of this shard (multi-GPU)            */
  const float* cmd_uniforms;     /* [RL_NUM_CMD_UNIFORMS][N] U[0,1) or NULL                 */
  const float* obs_uniforms[RL_NUM_OBS_GROUPS]; /* [N, group dim] U[0,1) or NULL           */
} RlRandom;


typedef struct RlCtx RlCtx;

int rl_abi_version(void);
const char* rl_last_error(void);
/* sizeof() of an ABI struct by name ("RlStepSpec", "RlRewardTerm", ...), -1 if unknown: lets a foreign-
 * language binding verify its mirror of the layouts before the first call. */
int64_t rl_struct_sizeof(const char* name);

/* Dynamic shared memory (bytes) one CTA of rl_step - a tile of 32 envs - needs for this spec; no device required.
 * An SM of the B200 holds two such CTAs when 2 * (bytes + 1024) <= 233472: from the second wave of tiles on
 * (> ~4700 envs) that second resident CTA is worth 1.5 x (profiles/r1_summary.md section 5). -1: invalid spec. */
int64_t rl_tile_record_bytes(const RlStepSpec* spec);

/* A context owns device scratch that its launches share (tickets and per-tile partials of the launch-wide reductions,
 * the status words and the epoch of the reset-id look-back): the launches of ONE context must be ordered - one stream, or
 * streams ordered by events, or one captured graph - like the manager calls of the ManagerBasedRLEnv they replace. Use one
 * context per concurrently stepping env. Copies of inputs / results may run on other streams. The scratch grows (is
 * re-allocated) when a launch brings more envs than any launch of the context before: make the first launches of a context
 * at its full env count before capturing graphs - a graph captured earlier holds the old scratch pointers. */
int rl_ctx_create(const RlStepSpec* spec, int device, RlCtx** out);
void rl_ctx_destroy(RlCtx* ctx);

/* Tuning knob of the general step kernel: warps per tile (4, 8 or 16; 0 = default 16). A tile is 32 consecutive envs
 * (one lane per env); its warps share the termination / reward / command / observation terms according to a static
 * schedule. envs_per_cta must be 0 or 32 (two tiles per CTA were measured slower in round 1 and removed; the cluster
 * kernels below are what shares code between tiles). Build-time specialised specs have their own kernel at 16 warps;
 * at 4 / 8 warps they run the generic one. Synchronous (re-uploads the schedule): not for hot loops or stream capture. */
int rl_ctx_set_launch_config(RlCtx* ctx, int envs_per_cta, int warps_per_cta);
/* The configuration of the general kernel in effect (after rl_ctx_create's defaults or the last successful set). */
int rl_ctx_get_launch_config(const RlCtx* ctx, int* envs_per_cta, int* warps_per_tile);
/* The two launches of an env step - rl_step(DONES | REWARDS | COMPACT) and rl_step(RESET | COMMAND | OBS) without an
 * env-id list - have their own kernels for the build-time specialised specs (csrc/mdp_step_v2.cu): SoA fields arrive by
 * 2-D TMA tensor-map copies issued by one thread, contact-force norms are computed once per env, results leave from
 * registers as coalesced rows. A configuration is (C, G, NW): a thread-block cluster of C CTAs shares G tiles, CTA r
 * evaluating the r-th share of the term list for all of them (C = G = 1: one tile per CTA, no cluster), NW warps per
 * CTA. A launch uses these kernels when num_envs is a multiple of 32 * G, every staged field is an SoA tensor ({1, row
 * stride}, 16-byte aligned) and the sensor rows are contiguous; anything else runs the general kernel, with bit-identical
 * results. This call reports what a launch of num_envs envs would use - *cluster_size = 0: the general kernel - and how
 * many launches these kernels have handled so far on this context (any pointer may be NULL).
 * Environment: RL_MDPSTEP_V2=0 switches them off at rl_ctx_create, RL_MDPSTEP_V2_CFG="CxG[xNW]" pins a configuration. */
int rl_ctx_get_cluster_config(const RlCtx* ctx, int64_t num_envs, int32_t* cluster_size, int32_t* tiles_per_cta,
                              int32_t* warps_per_cta, int64_t* launches);
/* Programmatic dependent launch: let each kernel's launch latency overlap the tail of its predecessor on
 * the stream (data dependencies are still honoured through cudaGridDependencySynchronize). Default off. */
int rl_ctx_set_pdl(RlCtx* ctx, int enabled);
/* Profiling aid: when set (device int64[ceil(N/32)][RL_DEBUG_STRIDE]), every CTA of rl_step records clock64():
 * words 0-7 phase boundaries (0 start, 1 loads issued, 2 tile resident, 3 stage 1 done, 4 stage 2 done, 5 stores
 * issued, 6 compaction done, 7 exit); words 8 .. 8+RL_MAX_TASKS-1 the duration of each scheduled task (index as in
 * rl_ctx_get_schedule); then one word per warp: the clock at which it entered stage 1. NULL switches it off. */
int rl_ctx_set_debug_buffer(RlCtx* ctx, void* device_i64_buffer);
/* The static work schedule of the current launch config: out[i] = {kind (0 reward, 1 observation, 2 terminations,
 * 3 command), a (reward term / obs group), b (half / obs term), owner warp, lo, hi, first column, late}. */
int rl_ctx_get_schedule(RlCtx* ctx, int32_t* out /* [RL_MAX_TASKS][8] */, int32_t* n_tasks);

/* prev_action <- action; action <- new_action; column a: target = clamp(a*scale+offset) written to
 * joint_target[:, joint_ids[a]] (position columns) or joint_vel_target[:, joint_ids[a]] (velocity columns). */
int rl_process_action(RlCtx* ctx, int64_t num_envs, const RlField* new_action, const RlMdpState* mdp,
                      const RlField* joint_target /* J, native order; columns not driven are untouched */,
                      const RlField* joint_vel_target /* J; may be NULL when no column is a velocity column */,
                      uint64_t* step_counter /* device, may be NULL: incremented by 1 */, void* stream);

/* Reset events of the reference (mode="reset", V/velocity_env_cfg.py:326-363): `reset_root_state_uniform`
 * (V/mdp/events.py:205-271, the non-pit branch; the "pits" sub-terrain is absent from the in-scope terrains) and
 * `reset_joints_by_scale` [IL]. Ranges are x, y, z, roll, pitch, yaw. */
typedef struct RlResetStateCfg {
  float default_root_state[13];   /* asset.data.default_root_state: pos 3, quat (w,x,y,z) 4, lin vel 3, ang vel 3 */
  float pose_lo[6], pose_hi[6];
  float vel_lo[6], vel_hi[6];
  float joint_pos_scale_lo, joint_pos_scale_hi;   /* reset_joints_by_scale position_range */
  float joint_vel_scale_lo, joint_vel_scale_hi;   /* reset_joints_by_scale velocity_range */
} RlResetStateCfg;

/* SURVEY.md 8(f) row 2: writes the post-reset physical state of the envs being reset, i.e. what the two events
 * above write into the simulator:
 *   root_pos_w   = default_pos + env_origin + U(pose xyz)
 *   root_quat_w  = quat_mul(default_quat, quat_from_euler_xyz(U(roll), U(pitch), U(yaw)))
 *   root_lin/ang_vel_w = default_vel + U(velocity ranges)
 *   joint_pos    = clamp(default_joint_pos * U(position_range), soft limits), joint_vel likewise (soft vel limit)
 * for env_ids[0 .. *n_env_ids) or, when env_ids is NULL, for the envs whose terminated | truncated byte is set.
 * Uniforms: Philox streams RL_STREAM_RESET_STATE (12 per env) / RL_STREAM_RESET_JOINTS (2J per env) of `rnd`, or
 * `uniforms` = [12 + 2J][N] U[0,1) when not NULL (pose 6, velocity 6, joint pos J, joint vel J). */
int rl_reset_scene_state(RlCtx* ctx, int64_t num_envs, const RlResetStateCfg* cfg, const RlField* env_origins /* [N,3] */,
                         const RlStateView* state, const uint8_t* terminated, const uint8_t* truncated,
                         const int32_t* env_ids, const int32_t* n_env_ids, const RlRandom* rnd,
                         const float* uniforms,
                         const uint8_t* assigned_to_pits /* [N] is_env_assigned_to_terrain(env, "pits")
                            (V/mdp/utils.py:44-70) or NULL: those envs get the default root state at their
                            origin with zero velocity and no perturbation (V/mdp/events.py:232-244) */,
                         void* stream);

/* ContactSensor update [IL] (isaaclab/sensors/contact_sensor/contact_sensor.py, _update_buffers_impl; the reference
 * configures it at V/velocity_env_cfg.py:86 and updates it every physics sub-step, :726): the step immediately in
 * front of the path (SURVEY.md 8(f) row 1). For every env:
 *   - history: net_forces_w_history[:, 1:] = history[:, :-1]; history[:, 0] = net_forces_w      (ring_slot < 0)
 *     or, B200-native, only history[:, ring_slot] = net_forces_w (ring_slot in [0, T)): no data is moved. Every
 *     consumer of the history takes the max over the history axis, which does not depend on the order of the samples -
 *     EXCEPT feet_stumble (V/mdp/rewards.py:428-436), which reads net_forces_w = history[:, 0], the NEWEST sample: a
 *     spec with an active feet_stumble term must use the rolling form (the Python providers check this);
 *   - air / contact timers of the tracked bodies, with is_contact = |F| > force_threshold:
 *       last_air        = first_contact ? current_air + dt     : last_air       (first_contact  = current_air > 0 & contact)
 *       current_air     = contact ? 0 : current_air + dt
 *       last_contact    = first_detach ? current_contact + dt  : last_contact   (first_detach = current_contact > 0 & !contact)
 *       current_contact = contact ? current_contact + dt : 0
 * net_forces_w is [N, B*3] in the body space of the history tensor; time_body_to_hist[i] is the history-space index
 * of timer body i (device-independent host array, num_time_bodies entries). */
int rl_contact_sensor_update(RlCtx* ctx, int64_t num_envs, const RlField* net_forces_w, const RlStateView* state,
                             const int32_t* time_body_to_hist, float dt, float force_threshold, int32_t ring_slot,
                             void* stream);

/* ---------------------------------------------------------------------------------------------------
 * SURVEY.md 8(f) row 3: the actuator models between process_action and physics. IsaacLab runs them inside
 * Articulation.write_data_to_sim() -> _apply_actuator_model() [IL], once per physics sub-step (decimation = 4,
 * V/velocity_env_cfg.py:714), on the joint position target rl_process_action wrote:
 *   error_pos = target_pos - joint_pos;  error_vel = target_vel - joint_vel
 *   computed  = stiffness * error_pos + damping * error_vel + target_effort            (IdealPDActuator.compute [IL])
 *   IDEAL_PD / IMPLICIT:  applied = clip(computed, -effort_limit, effort_limit)
 *   DC_MOTOR (DCMotor._clip_effort [IL], the four-quadrant torque-speed curve):
 *       vel       = clip(joint_vel, -vel_at_effort_lim, vel_at_effort_lim),
 *                   vel_at_effort_lim = velocity_limit * (1 + effort_limit / saturation_effort)
 *       top       = saturation_effort * ( 1 - vel / velocity_limit);  max_effort = min(top, effort_limit)
 *       bottom    = saturation_effort * (-1 - vel / velocity_limit);  min_effort = max(bottom, -effort_limit)
 *       applied   = clip(computed, min_effort, max_effort)
 * For IMPLICIT actuators PhysX integrates the PD law itself; computed / applied are the approximations IsaacLab
 * logs in data.computed_torque / data.applied_torque - exactly what joint_torques_l2 and joint_power read.
 * The reference's actuator groups: A1 / Go2 "legs" DCMotor (assets/unitree.py:55-63, 107-115), G1 ImplicitActuator
 * groups (:504-575).
 */
enum RlActuatorType { RL_ACT_NONE = 0, RL_ACT_IDEAL_PD = 1, RL_ACT_IMPLICIT = 2, RL_ACT_DC_MOTOR = 3 };

typedef struct RlActuatorCfg {
  int32_t num_joints;
  int32_t reserved;
  uint8_t type[RL_MAX_JOINTS];              /* RlActuatorType per native joint (RL_ACT_NONE: joint left untouched) */
  float stiffness[RL_MAX_JOINTS];
  float damping[RL_MAX_JOINTS];
  float effort_limit[RL_MAX_JOINTS];
  float saturation_effort[RL_MAX_JOINTS];   /* DC_MOTOR only */
  float velocity_limit[RL_MAX_JOINTS];      /* DC_MOTOR only */
} RlActuatorCfg;

/* Reads state->joint_pos / joint_vel and the targets, writes state->applied_torque and (optionally) computed_torque.
 * joint_vel_target / joint_effort_target may be NULL (zeros: the velocity tasks only set position targets). */
int rl_actuator_step(RlCtx* ctx, int64_t num_envs, const RlActuatorCfg* cfg, const RlField* joint_pos_target,
                     const RlField* joint_vel_target, const RlField* joint_effort_target, const RlStateView* state,
                     const RlField* computed_torque, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * SURVEY.md 8(f) row 4: terrain-aware command restriction.
 * Terrain grid: terrain_origins is the DEVICE tensor terrain.terrain_origins [num_rows, num_cols, 3] (contiguous);
 * [col_start, col_end) is _get_terrain_column_range(cfg, name) (V/mdp/utils.py:16-41), computed on the host.
 */
typedef struct RlTerrainGrid {
  const float* terrain_origins;   /* device, [num_rows * num_cols * 3] */
  int32_t num_rows, num_cols;
  int32_t col_start, col_end;     /* columns of the named sub-terrain; col_start >= col_end = terrain absent */
} RlTerrainGrid;

/* is_robot_on_terrain (V/mdp/utils.py:73-127): nearest terrain origin in the xy plane (first minimum in flat
 * row-major order, like torch.argmin), out[env] = col_start <= (argmin % num_cols) < col_end. */
int rl_is_robot_on_terrain(RlCtx* ctx, int64_t num_envs, const RlField* root_pos_w, const RlTerrainGrid* grid,
                           uint8_t* out /* [N] */, void* stream);

/* The tail of UniformThresholdVelocityCommand._update_command (V/mdp/commands.py:61-85), to be launched after
 * rl_step(... | RL_PHASE_COMMAND) and before the observations when the terrain has a "pits" sub-terrain:
 *   on_pits  = is_robot_on_terrain(env, "pits")
 *   left pit (was_on_pit & !on_pits): _resample_command - new vx, vy, wz, heading target, heading / standing flags,
 *            xy command zeroed below small_cmd_threshold (:43-47); time_left is NOT touched
 *   on pits: vx = clamp(|vx|, 0.3, 0.6), vy = wz = 0, heading_target = 0
 *   was_on_pit = on_pits
 * Uniforms: rnd->cmd_uniforms rows 1..6 ([RL_NUM_CMD_UNIFORMS][N], row 0 unused) or the Philox stream
 * RL_STREAM_PIT_RESAMPLE. Uses the command ranges of the context's spec. */
int rl_command_pit_restrict(RlCtx* ctx, int64_t num_envs, const RlField* root_pos_w, const RlTerrainGrid* grid,
                            const RlMdpState* mdp, uint8_t* was_on_pit /* [N] in/out */, const RlRandom* rnd,
                            void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Height scanner: RayCasterCfg(offset (0,0,20), ray_alignment "yaw", GridPatternCfg(resolution 0.1, size
 * [1.6, 1.0]), mesh_prim_paths ["/World/ground"]) at V/velocity_env_cfg.py:70-77 -> 17 x 11 = 187 vertical rays.
 * Upstream [IL] casts them against the terrain triangle mesh with Warp; the generated rough terrains are height
 * fields (isaaclab.terrains.height_field), whose mesh is the regular triangulation of a height grid, so the hit
 * point of a vertical ray is the piecewise-linear interpolation of that grid at the ray's (x, y):
 *   ray start = root_pos_w + quat_apply(yaw_quat(root_quat_w), ray_starts[r])     (quat_apply_yaw [IL])
 *   data.pos_w = root_pos_w (the 20 m offset lives in ray_starts, not in pos_w)
 *   hit z = interpolation over the cell's two triangles (diagonal from vertex (i, j) to (i+1, j+1), the
 *           triangulation of convert_height_field_to_mesh [IL]); rays that leave the grid hit nothing -> +inf
 * Output: ray_hits_z [N, R] and ray_sensor_pos_z [N] of RlStateView - what the height_scan observation reads.
 */
typedef struct RlHeightField {
  const float* heights;          /* device [num_x * num_y] vertex heights (m), x-major: h[ix * num_y + iy] */
  int32_t num_x, num_y;
  float x0, y0;                  /* world position of vertex (0, 0) */
  float horizontal_scale;        /* vertex spacing (m) */
  int32_t num_rays;              /* R = spec.num_rays */
  const float* ray_starts;       /* device [R * 3]: pattern offsets in the sensor frame INCLUDING the sensor offset
                                    (RayCaster.ray_starts [IL]); rays point along -z */
} RlHeightField;

int rl_height_scan_cast(RlCtx* ctx, int64_t num_envs, const RlHeightField* hf, const RlStateView* state /* reads
                        root_pos_w, root_quat_w; writes ray_hits_z, ray_sensor_pos_z */, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Stage 8 of ManagerBasedRLEnv.step() [IL]: event_manager.apply("interval", dt=step_dt) for one non-global interval
 * term (EventTermCfg(mode="interval", is_global_time=False)) whose function is push_by_setting_velocity [IL]; the
 * reference's randomize_push_robot (V/velocity_env_cfg.py:366-371). IsaacLab semantics (isaaclab/managers/
 * event_manager.py, isaaclab/envs/mdp/events.py), with sample_uniform(lo, hi) = u * (hi - lo) + lo, u in [0, 1):
 *   construction / EventManager.reset(ids):  time_left[ids] = sample_uniform(interval_lo, interval_hi)
 *   apply("interval", dt):                   time_left -= dt
 *                                            fire = time_left < 1e-6
 *                                            time_left[fire] = sample_uniform(interval_lo, interval_hi)
 *                                            root_vel_w[fire] += sample_uniform(vel_lo, vel_hi)   (6 components)
 * root_vel_w is (root_lin_vel_w x, y, z, root_ang_vel_w x, y, z); body velocities are not touched.
 */
typedef struct RlIntervalEventCfg {
  float interval_lo, interval_hi;     /* EventTermCfg.interval_range_s                                       */
  float vel_lo[6], vel_hi[6];         /* velocity_range x, y, z, roll, pitch, yaw; a missing key is (0, 0)   */
} RlIntervalEventCfg;

/* Two forms:
 *   reset form (env_ids != NULL): time_left[env_ids[0 .. *n_env_ids)] resampled; nothing else is read or written
 *     (pushed_ids / n_pushed may be NULL).
 *   step form (env_ids == NULL): one thread per env; an env whose terminated | truncated byte is set first gets a fresh
 *     timer (the reset of stage 6 of the step), then every env is decremented, compared and pushed. The ids of the
 *     pushed envs are written to pushed_ids[0 .. *n_pushed) in no particular order; *n_pushed is zeroed on the stream
 *     by the call itself, so it is defined after every launch without a host round trip (a CUDA graph replays it).
 *     A simulator writes the root velocities of exactly those envs back (write_root_velocity_to_sim [IL]).
 * time_left is a DEVICE float [N]; state->root_lin_vel_w / root_ang_vel_w are read and written.
 * Uniforms: Philox streams RL_STREAM_INTERVAL_RESET (timer on reset) / RL_STREAM_INTERVAL_PUSH (timer on fire, six
 * velocity components) of `rnd`, or `uniforms` = [8][N] U[0,1) when not NULL: row 0 timer on reset, row 1 timer on fire,
 * rows 2-7 velocity x, y, z, roll, pitch, yaw. */
int rl_interval_push(RlCtx* ctx, int64_t num_envs, const RlIntervalEventCfg* cfg, float dt, float* time_left,
                     const RlStateView* state, const uint8_t* terminated, const uint8_t* truncated,
                     const int32_t* env_ids, const int32_t* n_env_ids, int32_t* pushed_ids /* [N] */,
                     int32_t* n_pushed /* device [1] */, const RlRandom* rnd, const float* uniforms, void* stream);

/* The fused step over envs [0, num_envs), or over env_ids[0 .. *n_env_ids) when env_ids != NULL
 * (n_env_ids is a DEVICE pointer so that no host sync is needed after the reset compaction). */
int rl_step(RlCtx* ctx, int64_t num_envs, const RlStateView* state, const RlMdpState* mdp,
            const RlStepOut* out, const RlRandom* rnd, uint32_t phases,
            const int32_t* env_ids, const int32_t* n_env_ids, void* stream);

/* Manager-side reset of env_ids[0 .. *n_env_ids): log means, zero episode sums / metrics / actions /
 * episode length, resample the command (CommandTerm.reset [IL] -> V/mdp/commands.py:43-47). */
int rl_reset_envs(RlCtx* ctx, int64_t num_envs, const RlMdpState* mdp, const uint8_t* done_bits,
                  const RlRandom* rnd, const RlResetLog* log, const int32_t* env_ids,
                  const int32_t* n_env_ids, void* stream);

/* One reward term evaluated alone (raw value, no weight, no dt): the term-function protocol. */
int rl_term_eval(RlCtx* ctx, int64_t num_envs, const RlRewardTerm* term, const RlStateView* state,
                 const RlMdpState* mdp, const uint8_t* terminated /* may be NULL */, float* out,
                 void* stream);

/* Derived articulation views [IL] (ArticulationData properties) for Python term functions that run against the env
 * surface (SURVEY.md 8(b).2; e.g. V/mdp/rewards.py:34 reads projected_gravity_b, :226 root_com_lin_vel_b): one launch
 * writes projected_gravity_b [3], root_lin_vel_b [3] (= root_com_lin_vel_b), root_ang_vel_b [3] and heading_w [1] from
 * the root state, with the arithmetic of the step kernels. Any output may be NULL / have a NULL pointer. */
int rl_derived_views(RlCtx* ctx, int64_t num_envs, const RlStateView* state, const RlField* projected_gravity_b,
                     const RlField* root_lin_vel_b, const RlField* root_ang_vel_b, const RlField* heading_w, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RL_MDP_STEP_H_ */
