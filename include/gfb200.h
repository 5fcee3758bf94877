/*
 * gfb200.h -- C ABI of libgfb200.so: the fused genesis-forge manager step for NVIDIA B200 (sm_100a).
 *
 * The reference (jgillick/genesis-forge 0.2.1) is pure Python and has NO FFI layer for this path;
 * its only native-style call site is the Taichi launch
 *     kernel_get_contact_forces(force, position, link_a, link_b, links_quat, target_link_ids,
 *                               with_link_ids, out_forces, out_positions, position_counts, flag)
 * at genesis_forge/managers/contact/contact_manager.py:414-426 (caller allocates and zero-fills the
 * outputs, tensors contiguous, nothing returned).  The seam this library plugs into is therefore the
 * reference's MANAGER PROTOCOL: ManagedEnvironment.step / reset / get_observations
 * (genesis_forge/managed_env.py:274-398) and the manager step()/reset() methods it fans out to.  Each
 * entry point below names the reference code it replaces.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - plain C: integers, floats, raw device pointers, one opaque handle; no torch / C++ types.
 *   - every function returns 0 on success, a negative gfb_status otherwise; no exception crosses
 *     the boundary; gfb_last_error() gives the message.
 *   - all device buffers are OWNED BY THE CALLER (PyTorch tensors in the drop-in); the library
 *     borrows the pointers for the duration of the call.  The handle owns only scratch (per-slab
 *     partials, the report block, timing events).
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Kernels are enqueued
 *     and the call returns; only gfb_read_report() blocks.
 *   - rows are contiguous: an (N, W) array is N*W consecutive elements.  fp32 data, int32 counters,
 *     1-byte bool masks, int64 reset indices -- the dtypes the reference uses
 *     (genesis_env.py:75-77,84-86; gs.tc_float / gs.tc_int / gs.tc_bool).
 *   - one handle per (environment, device); not thread-safe; call from the thread that drives
 *     env.step().
 */
#ifndef GFB200_H
#define GFB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GFB_ABI_VERSION 14

/* ---- limits ------------------------------------------------------------------------------- */
#define GFB_MAX_DOFS 32
#define GFB_MAX_REWARD_TERMS 32
#define GFB_MAX_TERMINATION_TERMS 16
#define GFB_MAX_COMMANDS 4
#define GFB_MAX_COMMAND_DIMS 8
#define GFB_MAX_CONTACT_MANAGERS 4
#define GFB_MAX_CONTACT_LINKS 16
#define GFB_MAX_WITH_LINKS 32
#define GFB_MAX_OBS_GROUPS 4
#define GFB_MAX_OBS_COLS 256 /* summed over all groups, one frame each */
#define GFB_MAX_STAGED 24

typedef enum {
  GFB_OK = 0,
  GFB_ERR_INVALID = -1, /* bad argument / program            */
  GFB_ERR_CUDA = -2,    /* a CUDA runtime call failed        */
  GFB_ERR_NO_DEVICE = -3,
  GFB_ERR_UNSUPPORTED = -4
} gfb_status;

/* ---- buffer table -------------------------------------------------------------------------
 * Every device pointer a launch may touch lives in one table indexed by gfb_buf, so the packed
 * program can refer to buffers by small integers.  Unused entries are NULL.                    */
typedef enum {
  /* engine state, read only (Genesis getters; SURVEY.md appendix E) */
  GFB_B_POS = 0,      /* (N,3)  robot.get_pos()                         */
  GFB_B_QUAT,         /* (N,4)  robot.get_quat(), w first               */
  GFB_B_VEL,          /* (N,3)  robot.get_vel(), world frame            */
  GFB_B_ANG,          /* (N,3)  robot.get_ang(), world frame            */
  GFB_B_DOF_POS,      /* (N,D)  robot.get_dofs_position(dofs_idx)       */
  GFB_B_DOF_VEL,      /* (N,D)  robot.get_dofs_velocity(dofs_idx)       */
  GFB_B_DOF_FORCE,    /* (N,D)  robot.get_dofs_force(dofs_idx)          */
  GFB_B_C_FORCE,      /* (N,C,3) collider.get_contacts()["force"]       */
  GFB_B_C_POS,        /* (N,C,3) ...["position"]                        */
  GFB_B_C_LINK_A,     /* (N,C) int32                                    */
  GFB_B_C_LINK_B,     /* (N,C) int32                                    */
  GFB_B_LINKS_QUAT,   /* (N,L,4) rigid_solver.get_links_quat()          */
  GFB_B_LINKS_VEL,    /* (N,L,3) per-link linear velocity (feet_slide)  */
  /* environment state (genesis_env.py) */
  GFB_B_EPISODE_LENGTH,     /* (N,) int32  R/W                          */
  GFB_B_MAX_EPISODE_LENGTH, /* (N,) int32  R/W                          */
  GFB_B_ENV_ACTIONS,        /* (N,D) env.actions        R/W             */
  GFB_B_ENV_LAST_ACTIONS,   /* (N,D) env.last_actions   R/W             */
  GFB_B_TARGETS,            /* (N,D) action manager _actions (PD targets) */
  GFB_B_ACTION_RATE,        /* (N,)  sum((last_a - a)^2), written by gfb_action_step */
  /* managers */
  GFB_B_COMMAND0, GFB_B_COMMAND1, GFB_B_COMMAND2, GFB_B_COMMAND3,   /* (N,K_k) R/W */
  GFB_B_BASE_POS, GFB_B_BASE_QUAT, GFB_B_INV_BASE_QUAT,             /* entity cache, written */
  GFB_B_CONTACTS0, GFB_B_CONTACTS1, GFB_B_CONTACTS2, GFB_B_CONTACTS3,         /* (N,Lc,3) written */
  GFB_B_CONTACT_POS0, GFB_B_CONTACT_POS1, GFB_B_CONTACT_POS2, GFB_B_CONTACT_POS3,
  GFB_B_AIR0, GFB_B_AIR1, GFB_B_AIR2, GFB_B_AIR3, /* (4,N,Lc): last_air, cur_air, last_contact, cur_contact */
  GFB_B_TERMINATED,   /* (N,) bool written */
  GFB_B_TRUNCATED,    /* (N,) bool written */
  GFB_B_REWARD,       /* (N,) written      */
  GFB_B_EP_SECONDS,   /* (N,) R/W          */
  GFB_B_EP_SUMS,      /* (T_r, N) R/W, one row per reward term in table order */
  GFB_B_FIXED_COMMAND,/* (N,3) constant command tensor (examples/simple)      */
  GFB_B_TARGET_HEIGHT,/* (N,) per-env target height tensor for base_height    */
  GFB_B_HEIGHT_FIELD, /* (Hf,Wf) terrain height field                         */
  GFB_B_BODY_ACC_PREV,/* (N,6) previous body-frame lin/ang velocity           */
  /* observations */
  GFB_B_OBS_OUT0, GFB_B_OBS_OUT1, GFB_B_OBS_OUT2, GFB_B_OBS_OUT3,     /* (N, O_g*H_g) written     */
  GFB_B_OBS_PREV0, GFB_B_OBS_PREV1, GFB_B_OBS_PREV2, GFB_B_OBS_PREV3, /* previous step's rows     */
  GFB_B_OBS_NOISE0, GFB_B_OBS_NOISE1, GFB_B_OBS_NOISE2, GFB_B_OBS_NOISE3, /* (N,O_g) injected U(-1,1) */
  GFB_B_OBS_EXT0, GFB_B_OBS_EXT1, GFB_B_OBS_EXT2, GFB_B_OBS_EXT3,     /* (N,W) externally computed term values */
  /* reset / logging outputs */
  GFB_B_RESET_IDX,    /* (N,) int64 ascending env ids that reset this step (first n_reset valid) */
  GFB_B_LOG_OUT,      /* (T_r + T_t,) fp32: per-term episode means, per-term fire fractions       */
  GFB_B_LOG_ACC,      /* (T_r + T_t + 1,) fp64: per-term sums, fire counts, n_reset (for allreduce) */
  GFB_B_FORCE_RESET,  /* (N,) bool: envs to reset when GFB_PHASE_FORCED_RESET is requested          */
  /* injected random draws (parity mode; production mode draws Philox in-kernel) */
  GFB_B_INJ_CMD_STEP0, GFB_B_INJ_CMD_STEP1, GFB_B_INJ_CMD_STEP2, GFB_B_INJ_CMD_STEP3,     /* (N,K_k) */
  GFB_B_INJ_CMD_RESET0, GFB_B_INJ_CMD_RESET1, GFB_B_INJ_CMD_RESET2, GFB_B_INJ_CMD_RESET3, /* (N,K_k) */
  GFB_B_INJ_MAX_LEN,  /* (N,) fp32 U(-1,1) draws for max_episode_length */
  /* values of user-defined (host-evaluated) reward / termination terms: (J, N) fp32, one row per term */
  GFB_B_EXT_VALUES,
  GFB_B_DONES,        /* (N,) bool written: terminated | truncated (what wrappers/rsl_rl.py:57 computes) */
  /* per-env state of class-style user terms lowered into the specialised kernel: (N, *s) fp32 / int32 / bool,
     read and updated in place (ABI v14); a free slot may instead hold a per-launch (N, |U|, 3) fp32 gather of
     the engine's link positions / velocities that lowered terms read (read only) */
  GFB_B_USER_STATE0, GFB_B_USER_STATE1, GFB_B_USER_STATE2, GFB_B_USER_STATE3,
  GFB_B_USER_STATE4, GFB_B_USER_STATE5, GFB_B_USER_STATE6, GFB_B_USER_STATE7,
  GFB_B_COUNT
} gfb_buf;

/* ---- term opcodes --------------------------------------------------------------------------
 * One opcode per mdp function of the reference (file:line in genesis_forge/mdp/).              */
typedef enum {
  GFB_R_NONE = 0,
  GFB_R_IS_ALIVE,            /* rewards.py:31-37   */
  GFB_R_TERMINATED,          /* rewards.py:40-46   */
  GFB_R_BASE_HEIGHT,         /* rewards.py:54-90   p0=target; flags: target source, terrain */
  GFB_R_DOF_SIMILAR,         /* rewards.py:93-109  */
  GFB_R_LIN_VEL_Z,           /* rewards.py:112-135 */
  GFB_R_ANG_VEL_XY,          /* rewards.py:138-161 */
  GFB_R_FLAT_ORIENTATION,    /* rewards.py:164-193 */
  GFB_R_BODY_ACC_EXP,        /* rewards.py:196-249 p0=sensitivity */
  GFB_R_ACTION_RATE,         /* rewards.py:257-271 */
  GFB_R_TRACK_LIN_VEL,       /* rewards.py:279-317 p0=sensitivity, mgr=command or -1 (fixed) */
  GFB_R_TRACK_ANG_VEL,       /* rewards.py:320-358 */
  GFB_R_STAND_STILL,         /* rewards.py:361-385 p0=command_threshold */
  GFB_R_HAS_CONTACT,         /* rewards.py:393-410 p0=threshold, i0=min_contacts */
  GFB_R_CONTACT_FORCE,       /* rewards.py:413-428 p0=threshold */
  GFB_R_FEET_AIR_TIME,       /* rewards.py:431-469 p0=time_threshold p1=max-thr p2=dt+margin; i0=command mgr or -1 */
  GFB_R_FEET_SLIDE,          /* rewards.py:472-504 */
  GFB_R_EXTERNAL,            /* value column supplied by the host (user-defined term) */
  GFB_R_USER                 /* user-defined term lowered to device code (genesis_forge_b200/expr.py): i0 = identity
                                of its expression, p = its live scalar params.  Only a specialised kernel generated
                                for that expression evaluates it; the generic kernel refuses the launch. */
} gfb_reward_op;

typedef enum {
  GFB_T_NONE = 0,
  GFB_T_TIMEOUT,             /* terminations.py:17-23  */
  GFB_T_BAD_ORIENTATION,     /* terminations.py:26-71  p0=tilt threshold (see DESIGN.md), i0=grace */
  GFB_T_BASE_HEIGHT_MIN,     /* terminations.py:74-99  p0=minimum height */
  GFB_T_OUT_OF_BOUNDS,       /* terminations.py:102-137 p0..p3 = x_lo,x_hi,y_lo,y_hi */
  GFB_T_HAS_CONTACT,         /* terminations.py:139-155 p0=threshold, i0=min_contacts */
  GFB_T_CONTACT_FORCE,       /* terminations.py:158-172 p0=threshold */
  GFB_T_CONTACT_FORCE_GRACE, /* terminations.py:175-205 p0=threshold, i0=grace */
  GFB_T_EXTERNAL,            /* host-evaluated term: fires where row i0 of GFB_B_EXT_VALUES is non-zero */
  GFB_T_USER                 /* lowered user-defined term, as GFB_R_USER */
} gfb_termination_op;

/* observation column sources (mdp/observations.py:16-193 and the manager getters they wrap) */
typedef enum {
  GFB_O_ZERO = 0,
  GFB_O_COMMAND,       /* command manager `mgr`, column `col` (command_manager.py:172-174) */
  GFB_O_ANG_VEL_B,     /* entity_manager.get_angular_velocity()  entity_manager.py:142-146 */
  GFB_O_LIN_VEL_B,     /* entity_manager.get_linear_velocity()   entity_manager.py:136-140 */
  GFB_O_GRAVITY_B,     /* entity_manager.get_projected_gravity() entity_manager.py:130-134 */
  GFB_O_DOF_POS,       /* action_manager.get_dofs_position()                               */
  GFB_O_DOF_VEL,
  GFB_O_DOF_FORCE,
  GFB_O_TARGETS,       /* action_manager.get_actions(): processed targets                  */
  GFB_O_ENV_ACTIONS,   /* env.actions (raw)                                                */
  GFB_O_CONTACT_NORM,  /* |contacts[mgr][:, col]|  observations.py:181-193                 */
  GFB_O_EXTERNAL,      /* column `col` of GFB_B_OBS_EXT0, a (N, mgr) array of host-evaluated terms */
  GFB_O_USER           /* word `col` of the (N, mgr) values of the lowered user-defined observation terms
                          (genesis_forge_b200/expr.py): the post kernel's owner threads compute them into the
                          stash; gfb_observe has the specialised library compute them into GFB_B_OBS_EXT1.
                          Only a specialised kernel generated for them evaluates them (obs_group.user_id). */
} gfb_obs_src;

/* gfb_program_head.manager_flags */
#define GFB_MF_REWARD_DISABLED 1u /* RewardManager.enabled == False: the reset phase neither logs nor clears
                                     the episode sums (reward_manager.py:204); the host drops GFB_PHASE_REWARD */

/* reward-term flag bits */
#define GFB_RF_TARGET_FROM_COMMAND 1u /* base_height: target = command[mgr][:,0]       */
#define GFB_RF_TARGET_FROM_TENSOR 2u  /* base_height: target = GFB_B_TARGET_HEIGHT      */
#define GFB_RF_TERRAIN_HEIGHT 4u      /* base_height: subtract sampled terrain height   */
#define GFB_RF_TERRAIN_FLAT 8u        /* base_height: subtract constant p1 (flat terrain origin z) */
#define GFB_RF_HAS_MAX 16u            /* feet_air_time: clamp(max = p1)                 */
#define GFB_RF_FIXED_COMMAND 32u      /* tracking terms: command from GFB_B_FIXED_COMMAND */

typedef struct {
  int32_t op;     /* gfb_reward_op                                               */
  int32_t mgr;    /* command / contact manager index, -1 when unused             */
  uint32_t flags; /* GFB_RF_*                                                    */
  int32_t i0;
  float weight;   /* fp32(weight * dt) (reward_manager.py:184-185); 0 = skipped  */
  float p[4];
  int32_t ext_col; /* GFB_R_EXTERNAL: row of GFB_B_EXT_VALUES holding the value */
} gfb_reward_term;

typedef struct {
  int32_t op; /* gfb_termination_op */
  int32_t mgr;
  int32_t time_out; /* termination_manager.py:171-174 */
  int32_t i0;
  float p[4];
} gfb_termination_term;

typedef struct {
  int32_t n_dims;
  int32_t resample_steps; /* int(resample_time_sec / dt), command_manager.py:130 */
  int32_t enabled;        /* 0: never resampled in the kernel (external controller, user-level
                             subclass stepped on the host); such a manager may have n_dims == 0 */
  int32_t _pad;
  float lo[GFB_MAX_COMMAND_DIMS];
  float hi[GFB_MAX_COMMAND_DIMS];
} gfb_command_manager;

typedef struct {
  int32_t n_links;
  int32_t n_with;
  int32_t has_with_filter;
  int32_t track_air_time;
  float air_time_threshold; /* contact_manager.py:446-449 */
  float scene_dt;           /* contact_manager.py:441     */
  int32_t disabled;         /* manager.enabled == False: nothing is recomputed (contact_manager.py:331-336) */
  int32_t _pad;
  int32_t link_ids[GFB_MAX_CONTACT_LINKS];       /* global link idx */
  int32_t local_link_ids[GFB_MAX_CONTACT_LINKS]; /* for feet_slide  */
  int32_t with_ids[GFB_MAX_WITH_LINKS];
} gfb_contact_manager;

typedef struct {
  int32_t src; /* gfb_obs_src */
  int32_t mgr;
  int32_t col;
  float scale; /* observation_manager.py:241-244 */
  float noise; /* observation_manager.py:246-250; 0 = none */
} gfb_obs_col;

typedef struct {
  int32_t n_cols;    /* O_g: width of one frame                     */
  int32_t history;   /* H_g >= 1 (observation_manager.py:152-153)   */
  int32_t col_begin; /* first entry in gfb_program.obs_cols         */
  int32_t user_id;   /* identity of the lowered user-defined observation terms (GFB_O_USER columns) of
                        the table, nonzero in every group when it has any; 0 otherwise.  Structural: part
                        of what a specialised kernel is matched on */
} gfb_obs_group;

/* The packed term table ("program").  Re-packed by the host every step from the live Python
 * config objects (weights / params / ranges are curriculum-mutable in the reference:
 * docs/guide/managers/reward.md:132-171, command_manager.py:99-119) and passed by value to the
 * kernels as a __grid_constant__ parameter.                                                   */
typedef struct {
  int32_t num_envs;
  int32_t num_dofs;
  int32_t n_contact_slots; /* C */
  int32_t n_links_total;   /* L */
  float env_dt;            /* fp32(env.dt)                                  */
  int32_t base_max_episode_length; /* ceil(sec/dt) or 0 (no limit)          */
  float max_len_random_span;       /* fp32(base * scaling) or 0             */
  int32_t rng_mode;                /* 0 = injected draws, 1 = Philox        */
  uint64_t rng_seed;
  uint64_t step_index;

  int32_t n_reward, n_termination, n_command, n_contact, n_obs_groups;
  uint32_t manager_flags; /* GFB_MF_* */
  int32_t height_field_rows, height_field_cols;
  float terrain_bounds[4];

  /* action manager (position_action_manager.py:389-419, position_within_limits.py:113-131) */
  int32_t action_mode; /* 0 none, 1 position, 2 within-limits */
  int32_t _pad1;
  float action_scale[GFB_MAX_DOFS];
  float action_offset[GFB_MAX_DOFS];
  float action_clip_lo[GFB_MAX_DOFS];
  float action_clip_hi[GFB_MAX_DOFS];
  float default_dof_pos[GFB_MAX_DOFS];

  gfb_reward_term reward[GFB_MAX_REWARD_TERMS];
  gfb_termination_term termination[GFB_MAX_TERMINATION_TERMS];
  gfb_command_manager command[GFB_MAX_COMMANDS];
  gfb_contact_manager contact[GFB_MAX_CONTACT_MANAGERS];
  gfb_obs_group obs_group[GFB_MAX_OBS_GROUPS];
} gfb_program_head;

typedef struct {
  gfb_program_head head;
  gfb_obs_col obs_cols[GFB_MAX_OBS_COLS];
} gfb_program;

typedef struct {
  void* buf[GFB_B_COUNT];
} gfb_buffers;

/* phases of gfb_post_physics (bit mask).  GFB_PHASE_ALL is the fused step; subsets exist for the
 * initial / user-requested reset and for split execution around host-evaluated (external) terms. */
#define GFB_PHASE_ENTITY 1u       /* entity_manager.py:189-195                                */
#define GFB_PHASE_CONTACT 2u      /* contact_manager.py:331-336                               */
#define GFB_PHASE_TERMINATION 4u  /* termination_manager.py:151-190 + managed_env.py:308-310  */
#define GFB_PHASE_REWARD 8u       /* reward_manager.py:166-195                                */
#define GFB_PHASE_COMMAND 16u     /* command_manager.py:152-162                               */
#define GFB_PHASE_RESET 32u       /* genesis_env.py:233-252, contact_manager.py:316-329,
                                     reward_manager.py:197-222, command_manager.py:164-170    */
#define GFB_PHASE_OBSERVE 64u     /* observation_manager.py:218-256 for every env             */
#define GFB_PHASE_FORCED_RESET 128u /* reset set = GFB_B_FORCE_RESET (NULL: all envs)          */
#define GFB_PHASE_ALL 127u

/* status bits in gfb_report.status */
#define GFB_STATUS_NAN_ACTION 1u   /* position_action_manager.py:403-404 */
#define GFB_STATUS_INF_ACTION 2u   /* position_action_manager.py:405-406 */
#define GFB_STATUS_BAD_CONTACT 4u  /* contact_manager.py:401-403         */
#define GFB_STATUS_PEER_TIMEOUT 8u /* a peer rank did not deliver its logging partials in time */
#define GFB_STATUS_SCAN_TIMEOUT 16u /* internal: a slab waited > 2 s for its predecessors' reset counts */

#define GFB_MAX_PEERS 16           /* ranks of one NVLink domain sharing the logging exchange   */
#define GFB_IPC_HANDLE_BYTES 64    /* sizeof(cudaIpcMemHandle_t)                                */

/* The step report.  It is written by the post-physics kernel itself -- by its last block to leave,
 * once the launch-wide accumulators are final -- straight into mapped pinned host memory: every field,
 * then (behind a system-scope fence) `seq`, the word gfb_read_report() spins on.  No copy is enqueued
 * and the host does not wait for the stream.  Everything the host needs to continue is in it; the
 * logged episode means of the reward terms are device values (GFB_B_LOG_OUT, complete when the
 * launch has finished in stream order).  (A two-stage variant that delivered the reset count as soon
 * as the last slab had evaluated its terminations was measured in round 2 and not kept:
 * profiles/r2_02_post_kernel_experiments.txt.)                                                  */
typedef struct {
  int32_t n_reset;   /* number of valid entries in GFB_B_RESET_IDX */
  uint32_t status;   /* GFB_STATUS_* seen since the last report    */
  int32_t termination_count[GFB_MAX_TERMINATION_TERMS]; /* envs that fired each term this step */
  /* envs sharded over ranks (gfb_peer_connect): the same quantities over ALL ranks; on a
   * single-rank handle they repeat the local values                                            */
  int64_t global_n_reset;
  int64_t global_termination_count[GFB_MAX_TERMINATION_TERMS];
  uint64_t seq;      /* written last: number of the launch (with GFB_PHASE_RESET) this report belongs to */
  /* Sharded handles: n_reset (the rank's own count -- all the host needs to start its reset fan-out) is
   * complete as soon as the rank's kernel has finished its slabs; the global_* fields additionally
   * wait for the slowest peer's partials.  `local_seq` (same numbering as `seq`) is released right after
   * n_reset / status / termination_count, BEFORE the exchange: gfb_read_report_local() returns then, and
   * the wait for the peers overlaps the host's work instead of preceding it.                    */
  uint64_t local_seq;
} gfb_report;

typedef struct gfb_handle gfb_handle;

/* Create a handle for `num_envs` environments on CUDA device `device`.  device < 0 creates a
 * host-only handle (no CUDA calls): it accepts gfb_set_program / gfb_spec_describe only.        */
int gfb_create(int32_t num_envs, int32_t device, gfb_handle** out);
void gfb_destroy(gfb_handle* h);
const char* gfb_last_error(const gfb_handle* h);
int gfb_abi_version(void);
/* Binding self-check: size in bytes of gfb_program (0), gfb_buffers (1), gfb_report (2),
 * gfb_program_head (3); GFB_B_COUNT (4); gfb_spawn (5).  A foreign-language binding compares these
 * with its own struct layouts at load time.                                                     */
int64_t gfb_abi_sizeof(int32_t which);

/* Install the packed term table used by subsequent launches (host memcpy; cheap, call every step). */
int gfb_set_program(gfb_handle* h, const gfb_program* program);

/* Pre-physics launch.  Replaces GenesisEnv.step (genesis_env.py:193-203: episode_length += 1,
 * last_actions <- actions, actions <- raw) and the action manager's handle_actions
 * (position_action_manager.py:389-419: NaN/Inf check, a*scale+offset, clamp).
 *   raw_env:  (N,D) actions as given to env.step
 *   raw_mgr:  (N,D) actions the action manager processes (differs from raw_env only with a delay FIFO)
 * Uses GFB_B_EPISODE_LENGTH, ENV_ACTIONS, ENV_LAST_ACTIONS, TARGETS, ACTION_RATE of `b`.        */
int gfb_action_step(gfb_handle* h, const gfb_buffers* b, const float* raw_env, const float* raw_mgr,
                    void* stream);

/* The same launch for a caller that keeps its two action buffers as a RING: before the call it has
 * exchanged the roles of the buffers, so GFB_B_ENV_LAST_ACTIONS already holds the previous step's
 * actions (read only: action rate) and GFB_B_ENV_ACTIONS -- the buffer that was last_actions before --
 * is overwritten with `raw_env`.  The copy last_actions <- actions (genesis_env.py:202) becomes a pointer
 * exchange: 48 B/env (D = 12) less traffic, same values in both buffers as after gfb_action_step.  */
int gfb_action_step_ring(gfb_handle* h, const gfb_buffers* b, const float* raw_env, const float* raw_mgr,
                    void* stream);

/* Post-physics launch: one persistent kernel.  Replaces, for the phases requested, everything
 * ManagedEnvironment.step does after scene.step() (managed_env.py:294-326): entity cache, contact
 * net forces + air time, terminations, reset mask, rewards + episode sums, command resample, the
 * in-library part of reset(), the logging reductions, the step report, and the observation rows of
 * every env.  With GFB_PHASE_RESET a small second kernel is enqueued behind it that expands the
 * slabs' reset masks into GFB_B_RESET_IDX == (terminated | truncated).nonzero(), ascending; the
 * host does not wait for it (the report has the count), only later work on the stream does.    */
int gfb_post_physics(gfb_handle* h, const gfb_buffers* b, uint32_t phases, void* stream);

/* Wait for the report of the last launch that contained GFB_PHASE_RESET (the one blocking point of a
 * step; the reference blocks at the same place, managed_env.py:309,322).  The host spins on the
 * report's sequence word in mapped host memory, which the kernel's last block stores after
 * everything else: ~1 us after the store, without the driver's wake-up latency of a stream
 * synchronisation.                                                                              */
int gfb_read_report(gfb_handle* h, gfb_report* out, void* stream);
/* First stage of the report (see gfb_report.local_seq): blocks -- spinning on mapped memory -- until the
 * rank's own counts are final and returns the number of reset envs.  gfb_read_report() of the same launch
 * must still be called for the rest (status bits, global counts).                                */
int gfb_read_report_local(gfb_handle* h, int32_t* n_reset, void* stream);

/* gfb_post_physics + gfb_read_report in one call (one boundary crossing per step).              */
int gfb_post_physics_report(gfb_handle* h, const gfb_buffers* b, uint32_t phases, gfb_report* out, void* stream);

/* ---- envs sharded over the GPUs of one node (SURVEY.md 8(e)) ------------------------------------
 * The only exchange between ranks is the logging vector [sum of episode quotients per reward term,
 * fire count per termination term, n_reset].  Instead of a collective call after the kernel, the
 * finalize kernel itself does the exchange over NVLink peer memory: its last block stores the
 * rank's partials into every peer's inbox (P2P stores + a release flag), waits for the peers'
 * partials in its own inbox, sums them in rank order (bit-identical on all ranks) and writes the
 * GLOBAL logged means to GFB_B_LOG_OUT and the global counts to the report -- so the step keeps its
 * single host synchronisation.  Every rank must issue the same sequence of launches that contain
 * GFB_PHASE_RESET (step / reset calls); a missing peer raises GFB_STATUS_PEER_TIMEOUT after ~2 s.
 *   gfb_peer_export:  allocate this rank's inbox and return its CUDA IPC handle (64 bytes)
 *   gfb_peer_connect: open all `world` inboxes (handles = world x 64 bytes, in rank order)
 *   gfb_peer_disconnect: back to single-rank behaviour                                          */
int gfb_peer_export(gfb_handle* h, void* ipc_handle_out);
int gfb_peer_connect(gfb_handle* h, int32_t rank, int32_t world, const void* ipc_handles,
                     int64_t global_num_envs);
int gfb_peer_disconnect(gfb_handle* h);

/* Observation rows for a list of envs (idx == NULL: all envs) from the CURRENT engine state and
 * the cached inverse base quaternion.  Used after the engine-side reset writes for the envs in
 * GFB_B_RESET_IDX (observations are taken after reset, managed_env.py:322-326) and for the
 * initial get_observations().  Only frame 0 of each group is written.  A program with GFB_O_USER
 * columns first has the attached specialised library whose structure matches the program compute
 * the lowered user terms of those envs into GFB_B_OBS_EXT1 ((N, w) rows, from global memory only);
 * without one the call is refused (GFB_ERR_UNSUPPORTED) before anything runs.                     */
int gfb_observe(gfb_handle* h, const gfb_buffers* b, const int64_t* idx, int32_t n, void* stream);

/* Contact net-force scatter alone, with the reference kernel's own argument list
 * (contact_manager.py:414-426 / kernel.py:5-90).  link_a / link_b are int32.  Ordered
 * accumulation (contact slot index order) instead of the reference's float atomics.            */
int gfb_contact_forces(gfb_handle* h, const float* force, const float* position, const int32_t* link_a,
                       const int32_t* link_b, const float* links_quat, const int32_t* target_link_ids,
                       const int32_t* with_link_ids, float* out_forces, float* out_positions,
                       float* position_counts, int32_t n_envs, int32_t n_slots, int32_t n_links_total,
                       int32_t n_targets, int32_t n_with, int32_t has_with_filter, void* stream);

/* out[i] = rotate(vec[i], quat[i]) for i < n, optionally with the conjugate of quat[i]
 * (genesis.utils.geom.transform_by_quat(vec, inv_quat(q)); call sites entity_manager.py:130-146,
 * utils.py:13-55).  vec == NULL means the constant vector (0, 0, -1) (projected gravity).
 * vec (n,3), quat (n,4) w-first, out (n,3).                                                     */
int gfb_rotate(gfb_handle* h, const float* vec, const float* quat, float* out, int32_t n, int32_t conjugate,
               void* stream);

/* ---- reset-side writer: spawn pose of the reset envs (SURVEY.md 8(f) rank 1) ---------------------
 * One launch for what the reference does with ~35 indexed torch ops per reset:
 *   TerrainManager.generate_random_positions / generate_random_env_pos (terrain_manager.py:168-279):
 *     x = u_x * x_span + x_lo, y = u_y * y_span + y_lo (u in [0,1)), z = terrain height(x, y) +
 *     height_offset (bilinear height-field lookup of terrain_manager.py:100-166, or flat_height);
 *     written to row idx[i] of the manager's (n_rows,3) position buffer and to row i of pos_out.
 *   randomize_terrain_position.define_quat (mdp/reset.py:172-195): axes with rot_mode DRAW get
 *     rot_buffer[idx[i], axis] = U(rot_lo, rot_hi); the quaternion of the WHOLE buffer row
 *     (extrinsic x-y-z Euler -> w-first quaternion) goes to quat_buffer[idx[i]] and quat_out[i].     */
#define GFB_SPAWN_ROT_KEEP 0 /* leave the buffer column as it is (fixed / absent axis)            */
#define GFB_SPAWN_ROT_DRAW 1 /* draw U(rot_lo, rot_hi) for the reset envs                         */

typedef struct gfb_spawn {
  float x_lo, x_span, y_lo, y_span;
  float height_offset;
  float flat_height;              /* terrain height when there is no height field                */
  float terrain_bounds[4];        /* x_min, x_max, y_min, y_max of the height field              */
  int32_t height_field_rows, height_field_cols;
  int32_t with_rotation;          /* 0: positions only                                           */
  int32_t rot_mode[3];
  float rot_lo[3], rot_hi[3];
  uint64_t rng_seed, rng_counter; /* Philox key / counter for draws not supplied by the caller   */
} gfb_spawn;

/* idx: n int64 row indices (NULL = rows 0..n-1).  height_field: (rows, cols) fp32 or NULL (flat).
 * u_x, u_y: n draws in [0,1) each, or NULL = drawn in the kernel (Philox).  u_rot_{x,y,z}: n FINAL
 * angles for DRAW axes (already in [rot_lo, rot_hi)), or NULL = drawn in the kernel.
 * position_buffer (n_rows,3) in/out; rot_buffer (n_rows,3) in/out and quat_buffer (n_rows,4) out are
 * required when with_rotation; pos_out (n,3) and quat_out (n,4) are optional compact copies.        */
int gfb_spawn_pose(gfb_handle* h, const gfb_spawn* cfg, const int64_t* idx, int32_t n, int32_t n_rows,
                   const float* height_field, const float* u_x, const float* u_y, const float* u_rot_x,
                   const float* u_rot_y, const float* u_rot_z, float* position_buffer, float* rot_buffer,
                   float* quat_buffer, float* pos_out, float* quat_out, void* stream);

/* ---- reset-side writer: value rows for the engine setters of the reset envs (SURVEY.md 8(f) rank 1) ----
 * One launch for what the reference does with a few indexed torch ops per setter:
 *   GFB_ROWS_NOISE    out[i, j] = base[j] + u * a,  u ~ U(-1, 1)   PositionActionManager._add_random_noise
 *                     (position_action_manager.py:516-525) for the gains (n = 1, idx = NULL) and the
 *                     default joint positions of the reset envs (:432-464)
 *   GFB_ROWS_UNIFORM  out[i, j] = U(a, b)                           mdp.reset.randomize_link_mass_shift
 *                     (mdp/reset.py:229-284)
 * idx: n int64 env ids (NULL = rows 0..n-1); base: (width) or NULL (UNIFORM); draws: (n, width) injected
 * draws -- U(-1, 1) for NOISE, the final values for UNIFORM -- or NULL = Philox in the kernel keyed by
 * (seed, env id, counter, column); out (n, width) compact rows; scatter (rows, width) optional per-env
 * buffer that receives row idx[i].                                                              */
#define GFB_ROWS_NOISE 0
#define GFB_ROWS_UNIFORM 1
int gfb_reset_rows(gfb_handle* h, const int64_t* idx, int32_t n, int32_t width, int32_t mode, const float* base,
                   float a, float b, const float* draws, uint64_t seed, uint64_t counter, float* out, float* scatter,
                   void* stream);

/* ---- compile-time specialisation of the fused kernel -------------------------------------------
 * The fused post-physics kernel is an interpreter over the packed term table.  For a given table
 * STRUCTURE (opcodes, manager indices, flags, widths, link ids, observation layout -- everything
 * except live values such as weights, thresholds, ranges, dt) and slab plan, the same source can be
 * compiled with the structure as compile-time constants (genesis_forge_b200/spec.py generates the
 * header and runs nvcc; results are cached as genesis_forge_b200/_spec/spec_<hash>.so).
 *   gfb_spec_describe  structure of the CURRENT program for `phases`: the program head with every
 *                      live value zeroed (sizeof(gfb_program_head) bytes), the slab plan as int32
 *                      words (returns their count via *plan_words; capacity in plan_cap), the slab
 *                      size.  Works on a host-only handle (gfb_create with device < 0).
 *   gfb_spec_attach    load a specialised kernel library; it is used by gfb_post_physics whenever
 *                      its structure, plan, slab size and phases match the launch, otherwise the
 *                      generic kernel runs.  path == NULL detaches everything.                  */
int gfb_spec_describe(gfb_handle* h, const gfb_buffers* b, uint32_t phases, void* canonical_head,
                      int32_t* plan_out, int32_t plan_cap, int32_t* plan_words, int32_t* tile);
int gfb_spec_attach(gfb_handle* h, const char* path);
/* number of gfb_post_physics launches so far that ran a specialised / the generic kernel, and of
 * gfb_observe calls that ran a specialised library's lowered user-defined observation terms */
int gfb_spec_stats(const gfb_handle* h, int64_t* specialised, int64_t* generic, int64_t* user_observe);

/* Timing instrumentation: when enabled, each launch of gfb_post_physics' fused kernel is bracketed
 * by CUDA events on its stream; gfb_profile_read returns the accumulated device time.          */
int gfb_profile_enable(gfb_handle* h, int32_t enabled);
int gfb_profile_read(gfb_handle* h, float* post_ms_total, int32_t* post_launches, float* action_ms_total,
                     int32_t* action_launches);
/* Same for the small kernels; ms_total / launches are arrays of 4: [0] index compaction (behind
 * the post kernel), [1] observe (gfb_observe), [2] spawn (gfb_spawn_pose), [3] the lowered user-
 * defined observation terms of gfb_observe (specialised library).                                */
int gfb_profile_read_aux(gfb_handle* h, float* ms_total, int32_t* launches);
/* kernels launched by this handle since creation (gfb_action_step: 1, gfb_post_physics: 1-2, ...) */
int64_t gfb_launch_count(const gfb_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* GFB200_H */
