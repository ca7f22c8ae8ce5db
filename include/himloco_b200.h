/* himloco_b200.h -- C ABI of libhimloco_b200.so (hand-written sm_100a CUDA kernels for the
 * post-physics + GAE + AMP hot path of the HIMLoco legged_gym / rsl_rl stack).
 *
 * The reference (xyyandhtl/IsaacgymLoco) has no FFI layer for this path: the boundary is Python
 * bound methods mutating `self.*` tensors (SURVEY.md §8b).  Each entry point below names the
 * reference method it replaces; paths are relative to the reference root, LR =
 * legged_gym/legged_gym/envs/base/legged_robot.py.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *  - the library never allocates or frees caller-visible memory and never synchronises;
 *  - all work is enqueued on the `stream` argument (a cudaStream_t passed as void*);
 *    every call is CUDA-graph capturable;
 *  - return value 0 = success, otherwise an HL_E_* code; hl_last_error() gives the message
 *    (thread-local).  No exceptions cross the ABI.
 *  - tensors are consumed in Isaac Gym's own AoS layouts (LR:929-944).
 */
#ifndef HIMLOCO_B200_H_
#define HIMLOCO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HL_VERSION 102

#define HL_OK 0
#define HL_E_INVALID 1   /* bad argument / inconsistent config */
#define HL_E_CUDA 2      /* a CUDA runtime call or launch failed */
#define HL_E_UNSUPPORTED 3

#define HL_MAX_TERMS 64
#define HL_MAX_PTS 32
#define HL_MAX_BODIES_IDX 16
#define HL_NUM_DOF 12
#define HL_NUM_FEET 4
#define HL_OBS_STEP 45        /* one-step observation (LR:385-391)            */
#define HL_OBS_HISTORY 6      /* obs_buf = 6 x 45, newest first (LR:403)       */
#define HL_PRIV_OBS 238       /* 45 + 3 + 3 + 187 (LR:397-404)                 */
#define HL_AMP_OBS 30         /* LR:416                                        */
#define HL_AMP_FRAME 49       /* rsl_rl/rsl_rl/datasets/motion_loader.py:17-48 */

/* index-path arithmetic flavour (see DESIGN.md "bit-exact indices") */
#define HL_INDEX_MATH_TORCH_CUDA 0
#define HL_INDEX_MATH_TORCH_CPU 1

/* stages of hl_post_physics_stages (bit mask) -- one per reference method */
#define HL_ST_COUNTERS 0x001u    /* episode_length_buf += 1                     LR:193        */
#define HL_ST_FRAME 0x002u       /* base_lin_vel/base_ang_vel/projected_gravity LR:197-200    */
#define HL_ST_CONTACTS 0x004u    /* contact, contact_filt, last_contacts, feet  LR:203-209    */
#define HL_ST_HEADING 0x008u     /* commands[:,2] from heading error            LR:616-620    */
#define HL_ST_HEIGHTS 0x010u     /* measured_heights = _get_heights()           LR:1318-1355  */
#define HL_ST_TERMINATION 0x020u /* check_termination()                         LR:249-286    */
#define HL_ST_REWARD 0x040u      /* compute_reward() + all _reward_* terms      LR:363-380    */
#define HL_ST_OBS 0x080u         /* compute_observations()                      LR:382-404    */
#define HL_ST_OBS_NOSHIFT 0x100u /* with HL_ST_OBS: overwrite slot 0 only, keep the history   */
#define HL_ST_OBS_CLIP 0x200u    /* clip +-clip_observations (end of step())    LR:167-171    */
#define HL_ST_ROLL 0x400u        /* disturbance=0, last_* <- current            LR:235-241    */
#define HL_ST_BASE_HEIGHT 0x800u /* base_height_out = _get_base_heights()       LR:1357-1398  */
#define HL_ST_RESET_ZERO 0x1000u /* the RNG-free buffer resets of reset_idx     LR:323-329,350,361 */
#define HL_ST_RESET_DRAW 0x2000u /* the state re-draws of reset_idx (needs HlReset) LR:301-320,336-341 */
#define HL_ST_ALL_STEP (HL_ST_COUNTERS | HL_ST_FRAME | HL_ST_CONTACTS | HL_ST_HEADING | HL_ST_HEIGHTS | \
                        HL_ST_TERMINATION | HL_ST_REWARD | HL_ST_OBS | HL_ST_OBS_CLIP | HL_ST_ROLL)

/* Plain-old-data config; built once from the reference's cfg object (scales already x dt,
 * LR:1041-1046).  Field order is mirrored by isaacgymloco_b200/config.py::HlCfg. */
typedef struct HlCfg {
  int32_t struct_bytes;          /* = sizeof(HlCfg): ABI guard */
  int32_t num_bodies;            /* 17 for aliengo */
  int32_t control_type;          /* 0 = "P", 1 = "V", 2 = "T"   (LR:676-687) */
  int32_t only_positive_rewards; /* LR:374 */
  int32_t n_terms;               /* active reward terms, excluding `termination` */
  int32_t has_termination_term;  /* LR:377 */
  int32_t add_noise;             /* LR:393 */
  int32_t mesh_type;             /* 0 plane, 1 heightfield/trimesh (LR:1331) */
  int32_t measure_heights;
  int32_t terrain_rows, terrain_cols; /* height_samples.shape */
  int32_t term_base_vel_violate, term_out_of_border, term_fall_down; /* LR:266,275,282 */
  int32_t heading_command;       /* LR:616 */
  int32_t index_math;            /* HL_INDEX_MATH_* */
  int32_t n_px, n_py;            /* measured_points_x / _y counts (17, 11) */
  int32_t n_bx, n_by;            /* base height grid (7, 9; LR:1308-1309) */
  int32_t n_penalised, n_term_contact;
  int32_t feet_idx[HL_NUM_FEET];
  int32_t penalised_idx[HL_MAX_BODIES_IDX];
  int32_t term_contact_idx[HL_MAX_BODIES_IDX];
  int32_t term_id[HL_MAX_TERMS]; /* HlTerm ids in accumulation (alphabetical) order */
  int64_t max_episode_length;
  int64_t env_id_offset;         /* global id of local env 0 (env-sharded multi-GPU) */
  int64_t stairsup_start, stairsup_end, pit_start, gap_end; /* global slices, LR:71-90 */
  float dt, action_scale, hip_reduction, sim_dt;
  float soft_dof_vel_limit, soft_torque_limit, tracking_sigma, base_height_target;
  float foot_height_target_base, foot_height_target_terrain, max_contact_force;
  float termination_scale;
  float obs_lin_vel, obs_ang_vel, obs_dof_pos, obs_dof_vel, obs_height, clip_obs;
  float noise_height;            /* noise_scale_vec[45:232] (uniform) */
  float horizontal_scale, inv_horizontal_scale, vertical_scale, border_size;
  float x_limit, y_limit;        /* terrain.py:226 */
  float commands_scale[3];
  float p_gains[HL_NUM_DOF], d_gains[HL_NUM_DOF], torque_limits[HL_NUM_DOF];
  float default_dof_pos[HL_NUM_DOF], dof_pos_lo[HL_NUM_DOF], dof_pos_hi[HL_NUM_DOF];
  float dof_vel_limits[HL_NUM_DOF];
  float noise45[HL_OBS_STEP];    /* noise_scale_vec[0:45], LR:901-906 */
  float term_scale[HL_MAX_TERMS];
  float px[HL_MAX_PTS], py[HL_MAX_PTS], bx[HL_MAX_PTS], by[HL_MAX_PTS];
} HlCfg;

/* Device buffers of one env shard, named after the LeggedRobot attributes they are. */
#define HL_BUF_HISTORY_CLIPPED 1u /* obs_buf_in already lies within +-clip_observations (true after any step) */

struct HlReset;
typedef struct HlEnvBuffers {
  int32_t struct_bytes;
  uint32_t flags;                 /* HL_BUF_* */
  /* PhysX state (read-only), LR:929-944 */
  const float* root_states;       /* (N,13)  pos3 quat_xyzw4 lin3 ang3 */
  const float* dof_state;         /* (N,12,2) interleaved pos,vel      */
  const float* contact_forces;    /* (N,B,3)                            */
  const float* rigid_body_states; /* (N,B,13)                           */
  /* terrain */
  const int16_t* height_samples;  /* (rows,cols) int16, x -> rows       */
  const int16_t* height_min3;     /* (rows-1,cols-1) from hl_terrain_prepare; may be NULL */
  /* policy-side state */
  const float* actions;           /* (N,12) */
  float* last_actions;            /* (N,12) */
  float* last_last_actions;       /* (N,12) */
  float* last_dof_pos;            /* (N,12) */
  float* last_dof_vel;            /* (N,12) */
  const float* torques;           /* (N,12) */
  float* last_torques;            /* (N,12) */
  float* last_root_vel;           /* (N,6)  */
  float* commands;                /* (N,4)  */
  int64_t* episode_length_buf;    /* (N,)   */
  uint8_t* last_contacts;         /* (N,4) bool */
  uint8_t* contact_filt;          /* (N,4) bool */
  float* feet_air_time;           /* (N,4)  */
  float* disturbance;             /* (N,B,3); only [:,0,:] is read/zeroed */
  const int64_t* terrain_levels;  /* (N,)   */
  float* episode_sums;            /* (R,N): rows follow cfg term order, `termination` last */
  /* derived state */
  float* base_lin_vel;            /* (N,3) */
  float* base_ang_vel;            /* (N,3) */
  float* projected_gravity;       /* (N,3) */
  float* measured_heights;        /* (N,n_px*n_py) */
  float* feet_pos;                /* (N,4,3) optional (NULL = not materialised) */
  float* feet_vel;                /* (N,4,3) optional */
  uint8_t* reset_buf;             /* (N,) bool */
  uint8_t* time_out_buf;          /* (N,) bool */
  float* rew_buf;                 /* (N,)  */
  const float* obs_buf_in;        /* (N,270) previous history            */
  float* obs_buf_out;             /* (N,270) may alias obs_buf_in        */
  float* privileged_obs_buf;      /* (N,238) */
  /* observation noise: pre-drawn U[0,1) tensors (parity mode) or NULL => in-kernel Philox */
  const float* noise_u45;         /* (N,45)  */
  const float* noise_u187;        /* (N,187) */
  uint64_t philox_seed;
  uint64_t philox_offset;         /* advance by 1 per step (relative to *step_base when that is set) */
  int32_t* height_idx_out;        /* optional debug: (N,n_px*n_py,2) clipped (px,py) */
  float* base_height_out;         /* (N,) written by HL_ST_BASE_HEIGHT */
  /* Optional single-launch mode of hl_post_physics_fused: when reset_ids_out is non-NULL the fused
   * kernel itself emits what hl_select_reset_ids + hl_terminal_rows would (ascending ids by a
   * decoupled look-back over the CTAs; terminal rows from the data the CTA already holds). */
  int64_t* reset_ids_out;         /* (N,) capacity */
  int32_t* n_reset_out;           /* (1,) */
  float* term_priv_out;           /* (N, 51+P) capacity: compute_termination_observations rows */
  float* term_amp_out;            /* (N, 30) capacity or NULL */
  const float* term_noise_u45;    /* pre-drawn U[0,1) for the terminal rows, or NULL => Philox stream 1 */
  const float* term_noise_u187;
  uint64_t* fused_ws;             /* hl_fused_workspace_bytes(N) bytes, zeroed ONCE at allocation; also the tile
                                   * ticket of the persistent fused kernel (NULL => the tiled fallback kernel runs) */
  const float* foot_records;      /* optional (N,4,13): the four foot body-state records packed (what a host that ships PhysX
                                   * state over PCIe should send: 208 B/env instead of the 884 B of rigid_body_states);
                                   * when non-NULL it replaces rigid_body_states[:, feet_idx] */
  const struct HlReset* resample_host; /* HOST pointer or NULL: when set (with resample_interval > 0) the fused step itself resamples
                                   * the commands of the envs whose incremented episode length is a multiple of the interval
                                   * (_post_physics_step_callback, LR:612-613) before the heading command: ranges / uniforms
                                   * are read from this struct at launch time (Philox stream 2 when uniforms is NULL) */
  int64_t resample_interval;
  const float* height_min3f;      /* (rows-1,cols-1) fp32 = min3 * vertical_scale from hl_terrain_prepare_f32; may be
                                   * NULL (then the fused step uses the tiled fallback kernel and height_min3) */
  const int64_t* step_base;       /* (1,) device step counter or NULL.  Set: every Philox key uses *step_base + philox_offset
                                   * in place of philox_offset, read by each CTA after griddepcontrol.wait -- a captured CUDA
                                   * graph then draws fresh noise on every replay once something on the stream advances the
                                   * counter.  NULL = the step index arrives by value in philox_offset. */
} HlEnvBuffers;

int hl_version(void);
const char* hl_last_error(void);
/* sizeof() of the structs as compiled into the library (binding self-check) */
int hl_sizeof_cfg(void);
int hl_sizeof_env_buffers(void);

/* LeggedRobot._compute_torques(actions) -- LR:658-688.
 * `actions` is row-strided (a column slice of delayed_actions (N,4,12), LR:146). */
int hl_pd_torque(const HlCfg* cfg, const float* actions, int64_t actions_row_stride,
                 const float* dof_state, const float* motor_strength, const float* kp_factors,
                 const float* kd_factors, const float* last_dof_vel, float* torques_out,
                 float* joint_pos_target_out /* may be NULL */, int64_t n_envs, void* stream);

/* One-off per terrain: min3[px,py] = min(h[px,py], h[px+1,py], h[px,py+1]) (LR:1349-1353),
 * shape (rows-1, cols-1); turns the three gathers of every height sample into one. */
int hl_terrain_prepare(const int16_t* height_samples, int32_t rows, int32_t cols,
                       int16_t* height_min3_out, void* stream);
/* Same table already in metres: out[px,py] = fp32(min3) * vertical_scale (the product `heights *
 * vertical_scale` of LR:1355, rounded once like torch does), so a scan point is one fp32 gather. */
int hl_terrain_prepare_f32(const int16_t* height_samples, int32_t rows, int32_t cols, float vertical_scale,
                           float* height_min3f_out, void* stream);

/* The fused post-physics step: every HL_ST_* stage for all envs in ONE kernel
 * (LeggedRobot.post_physics_step LR:178-247 minus the RNG/PhysX-driven calls, plus the obs clip
 * of step() LR:167-171).  Observations are written speculatively for every env; envs that reset
 * are patched afterwards by hl_post_reset_fixup. */
int hl_post_physics_fused(const HlCfg* cfg, const HlEnvBuffers* bufs, int64_t n_envs, void* stream);
int64_t hl_fused_workspace_bytes(int64_t n_envs);
/* Which form the calling thread's last hl_post_physics_fused launch took: 0 = tiled (the default), 1 = persistent
 * role-pipelined (environment HL_FUSED_IMPL=persist, when the shard qualifies), -1 = none yet.  For tests / tools. */
int hl_fused_last_impl(void);

/* Any subset of stages, for the individual drop-in methods (check_termination(),
 * compute_reward(), compute_observations(), _get_heights(), ...).  If `env_ids` is non-NULL the
 * stages run only for ids[0 .. *n_ids_dev). */
int hl_post_physics_stages(const HlCfg* cfg, const HlEnvBuffers* bufs, uint32_t stages,
                           const int64_t* env_ids, const int32_t* n_ids_dev, int64_t n_envs,
                           void* stream);

/* env_ids = reset_buf.nonzero().flatten() -- LR:225.  Ascending int64 ids + count, on device.
 * workspace: hl_select_workspace_bytes(n) bytes. */
int64_t hl_select_workspace_bytes(int64_t n_envs);
int hl_select_reset_ids(const uint8_t* reset_buf, int64_t n_envs, int64_t* ids_out,
                        int32_t* count_out, void* workspace, void* stream);

/* compute_termination_observations(env_ids) (LR:439-460) and get_amp_observations()[env_ids]
 * (LR:228,406-416) for the compacted reset set, from the PRE-reset state.
 * noise: pre-drawn (N,45)/(N,187) U[0,1) indexed by env id, or NULL => Philox stream 1. */
int hl_terminal_rows(const HlCfg* cfg, const HlEnvBuffers* bufs, const int64_t* env_ids,
                     const int32_t* n_ids_dev, const float* term_noise_u45,
                     const float* term_noise_u187, float* term_priv_obs_out /* (cap,238) */,
                     float* term_amp_out /* (cap,30) or NULL */, int64_t n_envs, void* stream);

/* hl_select_reset_ids + hl_terminal_rows in ONE multi-CTA launch (ordered by summing the counts of
 * the lower-numbered CTAs).  workspace: hl_select_terminal_workspace_bytes(n) bytes, zeroed ONCE at
 * allocation (the kernel re-arms it itself: CUDA-graph safe).  out_priv may be NULL (ids only). */
int64_t hl_select_terminal_workspace_bytes(int64_t n_envs);
int hl_select_and_terminal(const HlCfg* cfg, const HlEnvBuffers* bufs, const float* term_noise_u45,
                           const float* term_noise_u187, int64_t* ids_out, int32_t* count_out,
                           float* term_priv_obs_out, float* term_amp_out, void* workspace, int64_t n_envs,
                           void* stream);

/* hl_select_and_terminal + hl_reset_and_fixup in ONE launch (LR:225-241 for the envs that reset): ids, count and terminal
 * rows as above; the warp that wrote an env's terminal rows then re-draws its state, zeroes its buffers, accumulates the
 * episode-logging means (reset->means_out / means_ws) and redoes its scan, observation slot 0 and roll. */
int hl_select_terminal_reset(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const float* term_noise_u45,
                             const float* term_noise_u187, int64_t* ids_out, int32_t* count_out, float* term_priv_obs_out,
                             float* term_amp_out, void* workspace, int64_t n_envs, void* stream);

/* After reset_idx mutated the reset envs: re-scan their heights (LR:332-333), rewrite slot 0 of
 * obs_buf and privileged_obs_buf from the post-reset state (stale base velocities, LR:232) and
 * redo the end-of-step roll for them (LR:235-241).  with_reset_zero != 0 first applies the
 * RNG-free part of reset_idx itself (last_* / feet_air_time / episode_sums / episode_length_buf
 * = 0, LR:323-329,350,361) for callers whose reset_idx does not (synthetic replay, bench). */
int hl_post_reset_fixup(const HlCfg* cfg, const HlEnvBuffers* bufs, const int64_t* env_ids,
                        const int32_t* n_ids_dev, int32_t with_reset_zero, int64_t n_envs, void* stream);

/* reset_idx's state re-draws in the kernel chain (SURVEY.md §8f rank 2): _update_terrain_curriculum
 * (LR:845-866), _reset_dofs (LR:690-716), _reset_root_states (LR:718-820), _resample_commands (LR:634-656) and
 * the Kp / Kd / motor-strength factor re-draws (LR:336-341), one warp per reset env.  Every `torch_rand_float(lo, hi)`
 * of the reference is `lo + (hi - lo) * u` with u from a per-env vector of HL_RESET_NU uniforms: pre-drawn
 * (`uniforms`, parity mode: rows indexed by env id) or Philox4x32-10 stream 3 keyed by (seed, offset, global env id)
 * -- statistically, not bitwise, the reference's torch stream.  The PhysX setters the reference calls afterwards
 * (set_dof_state_tensor_indexed, set_actor_root_state_tensor_indexed) stay with the caller: the kernel writes the
 * same rows of the same tensors.  Column map of the uniforms:
 *   0-11 dof_pos ratio | 12-23 dof_vel | 24-26 base x,y,z | 27-29 roll,pitch,yaw | 30-35 base lin/ang vel |
 *   36 cmd vx | 37 cmd vy | 38 cmd heading (or yaw rate) | 39 cmd vx of a high-speed env | 40 Kp | 41 Kd |
 *   42 motor strength | 43 random terrain level */
#define HL_RESET_NU 44
#define HL_RESET_DOFS 1u
#define HL_RESET_ROOT 2u
#define HL_RESET_COMMANDS 4u
#define HL_RESET_FACTORS 8u
#define HL_RESET_CURRICULUM 16u
typedef struct HlReset {
  int32_t struct_bytes;            /* sizeof(HlReset): ABI guard */
  int32_t custom_origins;          /* LR:726 */
  int32_t has_pos_range;           /* domain_rand.base_init_pos_range given (else xy in +-1 m, LR:746) */
  int32_t has_rot_range;           /* domain_rand.base_init_rot_range given (LR:753) */
  int32_t vel_range_is_dict;       /* base_init_vel_range: 0 = (lo, hi) for all six, 1 = per axis (LR:779-816) */
  int32_t randomize_dof_pos;       /* dof_init_pos_ratio_range given (LR:698) */
  int32_t randomize_dof_vel;       /* LR:707 */
  int32_t randomize_kp, randomize_kd, randomize_motor_strength;   /* LR:336-341 */
  int32_t heading_command;         /* LR:645 */
  int32_t terrain_curriculum;      /* cfg.terrain.curriculum and init_done (LR:301,853) */
  int32_t max_terrain_level;       /* LR:1235 */
  int32_t n_terrain_types;         /* columns of terrain_origins */
  int32_t parts;                   /* 0 = everything; else HL_RESET_* bits: only those parts (the individual reset hooks) */
  int32_t pad_;
  int64_t num_envs_global;         /* all shards together */
  int64_t high_vel_envs;           /* size of the high-speed command slice: global env ids < high_vel_envs take it (LR:649,
                                      `env_ids < num_envs * 0.2`, counted on the host with the reference's own expression) */
  float base_init_state[13];       /* LR:1160-1161 */
  float pos_range[6];              /* x lo,hi, y lo,hi, z lo,hi */
  float rot_range[6];              /* roll, pitch, yaw lo,hi */
  float vel_range[12];             /* tuple: [0],[1]; dict: x,y,z,roll,pitch,yaw lo,hi */
  float dof_pos_ratio[2], dof_vel_range[2];
  float kp_range[2], kd_range[2], motor_strength_range[2];
  float cmd_lin_vel_x[2], cmd_lin_vel_y[2], cmd_ang_vel_yaw[2], cmd_heading[2];   /* self.command_ranges (they move with the curriculum) */
  float env_length, max_episode_length_s;   /* LR:858,860 */
  /* device buffers the re-draws write (the env's own tensors) */
  float* root_states;              /* (N,13) */
  float* dof_state;                /* (N,12,2) */
  float* commands;                 /* (N,4) */
  float* env_origins;              /* (N,3) */
  const float* terrain_origins;    /* (levels, types, 3) or NULL */
  int64_t* terrain_levels;         /* (N,) */
  const int64_t* terrain_types;    /* (N,) or NULL */
  float* kp_factors;               /* (N,1) or NULL */
  float* kd_factors;               /* (N,1) or NULL */
  float* motor_strength_factors;   /* (N,1) or NULL */
  const float* uniforms;           /* (N, HL_RESET_NU) pre-drawn U[0,1) or NULL => Philox stream 3 */
  /* optional episode logging of reset_idx (LR:346-350) folded into the reset launch: means_out[k] = mean over the reset
   * envs of episode_sums[k] / clip(episode_length, 1) / dt, unchanged when no env resets.  means_ws: (n_rows + 1)
   * doubles, zeroed ONCE at allocation (the kernel re-arms it). */
  float* means_out;                /* (n_rows,) or NULL */
  double* means_ws;
  /* (8,) device float64 command ranges in the order of the by-value fields (lin_vel_x lo,hi | lin_vel_y lo,hi |
   * ang_vel_yaw lo,hi | heading lo,hi) or NULL = the by-value cmd_* fields.  Set: every command draw (hl_resample_commands,
   * the re-draws of the reset launches, the fused step's pre-step resampling through resample_host) reads the ranges
   * here, after griddepcontrol.wait, and converts each with (float) -- the round-to-nearest a c_float assignment of the
   * same Python float does, so both forms draw bit-identical commands from equal values.  A captured graph then follows
   * range changes made on the device (hl_command_curriculum) or copied there between replays. */
  const double* cmd_ranges;
} HlReset;
int hl_sizeof_reset(void);
/* reset_idx(env_ids) without the fix-up: curriculum, state re-draws, the RNG-free buffer resets (LR:323-329,361). */
int hl_reset_idx(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                 const int32_t* n_ids_dev, int64_t n_envs, void* stream);
/* Only the re-draws selected by reset->parts, no buffer zeroing: the individual hooks _reset_dofs(env_ids) /
 * _reset_root_states(env_ids) called on their own. */
int hl_reset_draw(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                  const int32_t* n_ids_dev, int64_t n_envs, void* stream);
/* The same followed by hl_post_reset_fixup's work for the same env, in ONE launch (what post_physics_step runs). */
int hl_reset_and_fixup(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                       const int32_t* n_ids_dev, int64_t n_envs, void* stream);
/* _resample_commands(env_ids) (LR:634-656).  env_ids NULL: the envs whose episode_length_buf + 1 is a multiple of
 * `interval` -- the pre-step resampling of _post_physics_step_callback (LR:612-613), evaluated before the fused step
 * increments the counter.  Uniform columns 36-39 (Philox stream 2 for the pre-step form). */
int hl_resample_commands(const HlCfg* cfg, const HlEnvBuffers* bufs, const HlReset* reset, const int64_t* env_ids,
                         const int32_t* n_ids_dev, int64_t interval, int64_t n_envs, void* stream);
/* update_command_curriculum(env_ids) (LR:868-880) on device-resident ranges, as one capturable launch (one CTA, no host
 * sync, no allocation).  n = *n_ids_dev; n == 0 leaves the ranges alone.  Otherwise s = float64 sum of
 * tracking_sums[env_ids[i]], v = fp32(fp32(s / n) / fp32(max_episode_length)), and when (double)v > threshold the
 * lin_vel_x / lin_vel_y bounds move by -+0.1 and are clipped in float64 as np.clip does: x lo to [-max_backward, 0],
 * x hi to [0, max_forward], y lo to [-max_lat, 0], y hi to [0, max_lat].  ranges: (8,) in/out, HlReset.cmd_ranges order;
 * ranges_log: (8,) or NULL, receives the ranges after the decision.  The host's fp32 torch.mean sums in another order, so
 * the two decisions can differ when the mean lies within a few ulp of the threshold. */
int hl_command_curriculum(const float* tracking_sums, const int64_t* env_ids, const int32_t* n_ids_dev, double threshold,
                          int64_t max_episode_length, double max_backward, double max_forward, double max_lat,
                          double* ranges, double* ranges_log, int64_t n_envs, void* stream);

/* ReplayBuffer.insert(states, next_states) -- rsl_rl/rsl_rl/storage/replay_buffer.py:52-68: row r of
 * both (n_rows, width) inputs is written to ring row (step + r) mod buffer_rows; when more than
 * buffer_rows rows arrive only the last buffer_rows survive (the reference's second slice
 * overwrites the first).  One launch for both tensors. */
int hl_ring_insert(const float* states, const float* next_states, float* ring_states, float* ring_next,
                   int64_t n_rows, int32_t width, int64_t buffer_rows, int64_t step, void* stream);

/* The runners' episode statistics of one env-step (him_on_policy_runner.py / hybrid_runner.py), as one launch without a
 * host sync or allocation:
 *   cur_reward_sum += rewards; cur_episode_length += 1
 *   new_ids = (dones > 0).nonzero(); rewbuffer.extend(cur_reward_sum[new_ids]); lenbuffer.extend(cur_episode_length[new_ids])
 *   cur_reward_sum[new_ids] = 0; cur_episode_length[new_ids] = 0
 * The deques are a device ring of ring_size entries per buffer: entry i of the run goes to slot i mod ring_size, in
 * ascending env id within a step.  ids: the step's done envs, ascending, count *n_ids_dev on the device (the capacity-N
 * buffer of post_physics_step_device() will do); only envs with dones set search them.  cursor: int64 {total, ticket},
 * the ticket zero between launches; total = the entries written so far, advanced by *n_ids_dev.  Of a step with more
 * done envs than ring_size only the last ring_size are written. */
int hl_episode_stats(const float* rewards, const uint8_t* dones, const int64_t* ids, const int32_t* n_ids_dev,
                     float* cur_reward_sum, float* cur_episode_length, float* ring_reward, float* ring_length,
                     int64_t ring_size, int64_t* cursor, int64_t n_envs, void* stream);

/* reset_idx's episode logging -- LR:346-350: for every reward row k,
 *   means_out[k] = mean_{e in env_ids}( episode_sums[k][e] / clip(episode_length_buf[e], min=1) / dt )
 * (one launch instead of 21 masked-mean chains; the id count stays on the device).  With
 * zero_rows != 0 the rows of the listed envs are zeroed afterwards (`episode_sums[key][env_ids] = 0`). */
int hl_episode_means(float* episode_sums, const int64_t* episode_length_buf, const int64_t* env_ids,
                     const int32_t* n_ids_dev, int32_t n_rows, int64_t n_envs, float dt, int32_t zero_rows,
                     float* means_out, void* stream);

/* get_amp_observations() for all envs -- LR:406-416: (N,30) = dof_pos, base_lin_vel,
 * base_ang_vel, dof_vel. */
int hl_amp_observations(const float* dof_state, const float* base_lin_vel, const float* base_ang_vel,
                        float* amp_obs_out, int64_t n_envs, void* stream);

/* HIMRolloutStorage.compute_returns(last_values, gamma, lam) --
 * rsl_rl/rsl_rl/storage/him_rollout_storage.py:113-127 (== amp_rollout_storage.py:141-155).
 * Step 1: reverse-time GAE scan; writes returns and raw advantages (T,N,1) and accumulates
 * moments[0..2] = (sum adv, sum adv^2, count) in float64 (caller zeroes `moments` first; when
 * env-sharded, all-reduce them before step 2).  Step 2: (adv - mean) / (std_unbiased + 1e-8). */
int hl_gae_scan(const float* rewards, const float* values, const uint8_t* dones,
                const float* last_values, float* returns, float* advantages, double* moments,
                int32_t t_len, int64_t n_envs, float gamma, float lam, void* stream);
int hl_adv_normalize(float* advantages, const double* moments, int64_t n_elems, void* stream);

/* One rollout step recorded into the time-major storage slots, fused:
 *   runner terminal-observation patch   rsl_rl/rsl_rl/runners/him_on_policy_runner.py:122-123
 *       next_critic_obs = critic_obs.clone(); next_critic_obs[termination_ids] = termination_privileged_obs
 *   HIMPPO.process_env_step             rsl_rl/rsl_rl/algorithms/him_ppo.py:104-115
 *       rewards += gamma * squeeze(values * time_outs.unsqueeze(1), 1)      (each op rounded on its own)
 *   HIMRolloutStorage.add_transitions   rsl_rl/rsl_rl/storage/him_rollout_storage.py:92-108
 *       the ten slot copies at `step` (dones stored as uint8)
 * Sources are env-major device rows; `*_out` point at slot `step` of the (T,N,.) tensors.  A
 * source/destination pair with either pointer NULL is skipped (e.g. the env already wrote that
 * slot in place).  term_ids: ascending unique env ids (reset_buf.nonzero()), count on the device;
 * NULL = no patch.  time_outs NULL = no bootstrap. */
typedef struct HlTransition {
  int32_t struct_bytes;            /* sizeof(HlTransition): ABI guard */
  int32_t obs_dim, priv_dim, act_dim;
  float gamma;
  int32_t pad_;
  const float* obs;                /* (N, obs_dim)  transition.observations            */
  const float* critic_obs;         /* (N, priv_dim) transition.critic_observations     */
  const float* next_critic_obs;    /* (N, priv_dim) privileged obs after the env step  */
  const int64_t* term_ids;         /* (n_term,) or NULL                                */
  const int32_t* n_term_dev;       /* device scalar                                    */
  const float* term_rows;          /* (n_term, priv_dim) termination_privileged_obs    */
  const float* actions;            /* (N, act_dim) */
  const float* rewards;            /* (N,)         */
  const uint8_t* dones;            /* (N,) bool/uint8 */
  const float* values;             /* (N,1)        */
  const uint8_t* time_outs;        /* (N,) bool/uint8 or NULL */
  const float* log_prob;           /* (N,)         */
  const float* mu;                 /* (N, act_dim) */
  const float* sigma;              /* (N, act_dim) */
  float* obs_out;
  float* critic_out;
  float* next_critic_out;
  float* actions_out;
  float* rewards_out;
  uint8_t* dones_out;
  float* values_out;
  float* log_prob_out;
  float* mu_out;
  float* sigma_out;
} HlTransition;
int hl_sizeof_transition(void);
int hl_record_transition(const HlTransition* t, int64_t n_envs, void* stream);

/* HIMRolloutStorage.mini_batch_generator's row gathers --
 * rsl_rl/rsl_rl/storage/him_rollout_storage.py:137-177: for one minibatch, `x.flatten(0,1)[batch_idx]`
 * of all ten rollout fields (observations, critic observations, actions, next critic observations,
 * values, advantages, returns, log-probs, mu, sigma), as ONE launch: each index is read once and
 * every field's row is copied to dst[row].  Fields: src (n_src_rows, width) row-major, dst
 * (n_rows, width).  Out-of-range indices are an error the caller must not make (rows are skipped). */
#define HL_MAX_GATHER_FIELDS 12
typedef struct HlGatherFields {
  int32_t struct_bytes;            /* sizeof(HlGatherFields): ABI guard */
  int32_t n_fields;
  const float* src[HL_MAX_GATHER_FIELDS];
  float* dst[HL_MAX_GATHER_FIELDS];
  int32_t width[HL_MAX_GATHER_FIELDS];
} HlGatherFields;
int hl_sizeof_gather_fields(void);
int hl_minibatch_gather(const HlGatherFields* f, const int64_t* indices, int64_t n_rows, int64_t n_src_rows,
                        void* stream);

/* AMPLoader.get_full_frame_at_time_batch(traj_idxs, times) --
 * rsl_rl/rsl_rl/datasets/motion_loader.py:231-255 with quaternion_slerp
 * rsl_rl/rsl_rl/utils/utils.py:153-186.  `frames` = all clips stacked (sum n_i, 49);
 * clip i starts at row clip_offset[i]; lens/num_frames are the float64 arrays of the loader. */
int hl_amp_frame_blend(const float* frames, const int32_t* clip_offset, const double* clip_len,
                       const double* clip_num_frames, int32_t n_clips, const int64_t* traj_idxs,
                       const double* times, float* out /* (B,49) */,
                       int32_t* idx_low_out /* optional (B,) */, int32_t* idx_high_out, int64_t batch,
                       void* stream);

/* AMPLoader.feed_forward_generator preload branch -- motion_loader.py:321-330: for each idx, the
 * 30 AMP columns [7:19] + [31:49] of preloaded_s and preloaded_s_next. */
int hl_amp_gather_pairs(const float* preloaded_s, const float* preloaded_s_next, int64_t n_preloaded,
                        const int64_t* idxs, float* s_out, float* s_next_out, int64_t batch,
                        void* stream);

/* AMPDiscriminator.predict_amp_reward input assembly -- amp_discriminator.py:59-63 with
 * Normalizer.normalize_torch utils.py:124-130 and the runner's terminal patch
 * hybrid_runner.py:191-192 fused in: row i of next_state is taken from terminal_states[j] when
 * env i == reset_ids[j].  mean/std are (30,) fp32 (std = sqrt(fp32(var + eps))).
 * Any of mean/std may be NULL (normalizer=None). */
int hl_amp_disc_input(const float* state, const float* next_state, const float* mean, const float* std_,
                      float clip, const int64_t* reset_ids, const int32_t* n_reset_dev,
                      const float* terminal_states, float* next_state_patched_out /* optional */,
                      float* x_out /* (N,60) */, int64_t n_envs, void* stream);

/* One AMP env-step of HybridPolicyRunner.learn (hybrid_runner.py:184-195 without the discriminator MLP), as one
 * launch without a host sync or allocation, issued after post_physics_step_device():
 *   next = get_amp_observations() (LR:406-416); next_with_term = next; next_with_term[reset_ids[:*n_reset]] = terminal_amp
 *   x_out = cat(normalise(amp_obs), normalise(next_with_term))   (N,60), as hl_amp_disc_input computes it
 *   ReplayBuffer.insert(amp_obs, next_with_term) (replay_buffer.py:52-68) at the device cursor
 *   amp_obs = next                                               (in place: (N,30) in/out)
 * reset_ids ascending with the count on the device; only envs with reset_buf set search them.  norm_stats: (2,30)
 * float64 [mean; var] of the Normalizer, mean = fp32(mean), std = sqrt(fp32(var + eps)), clamp to +-clip; NULL = no
 * normaliser.  Row e goes to ring row (cursor[0] + e) mod ring_rows.  cursor: int64 {step, num_samples, ticket}, the
 * ticket zero between launches; the launch advances num_samples = min(ring_rows, max(step + N, num_samples)) and
 * step = (step + N) mod ring_rows.  n_envs <= ring_rows. */
int hl_amp_transition(const float* dof_state, const float* base_lin_vel, const float* base_ang_vel,
                      const uint8_t* reset_buf, const int64_t* reset_ids, const int32_t* n_reset_dev,
                      const float* terminal_amp, const double* norm_stats, double eps, float clip, float* amp_obs,
                      float* x_out, float* ring_states, float* ring_next, int64_t ring_rows, int64_t* cursor,
                      int64_t n_envs, void* stream);

/* ... and its epilogue -- amp_discriminator.py:64-68,70-72:
 * r = coef * clamp(1 - (d-1)^2/4, min 0); if lerp > 0: r = (1-lerp) r + lerp task_r. */
int hl_amp_reward(const float* d_logits, const float* task_reward, float coef, float lerp,
                  float* reward_out, int64_t n_envs, void* stream);

/* RunningMeanStd.update moments of one batch -- utils.py:90-94: per-column mean and (biased)
 * variance of x (M,D) in float64; out = [mean(D), var(D)].  Scratch: 2*D*grid doubles provided by
 * the caller via hl_moments_workspace_bytes. */
int64_t hl_moments_workspace_bytes(int32_t dim);
int hl_column_moments(const float* x, int64_t rows, int32_t dim, double* mean_var_out,
                      void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HIMLOCO_B200_H_ */
