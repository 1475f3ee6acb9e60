/*
 * om_b200.h -- C ABI of the B200-native env-step hot path for olympics-mujoco.
 *
 * The reference (pigBond/olympics-mujoco) is pure Python; its "FFI" for this path is the set of Python
 * calls into MuJoCo / mushroom_rl / NumPy listed beside each entry point below (paths relative to the
 * reference root).  A maintainer binds these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - Every `float* / uint8_t* / int32_t*` argument is a DEVICE pointer unless its name ends in `_host`.
 *  - Per-env arrays are structure-of-arrays with the env index fastest: element (c, env) of an array
 *    with C components lives at  a[c*ld + env],  ld >= n (number of envs).  A MuJoCo field that is
 *    [nbody,3] per env therefore has C = nbody*3 components, component index body*3+axis.
 *    Rollout buffers are time-major: (t, c, env) at a[(t*C + c)*ld + env].
 *  - Quaternions are [w,x,y,z]; spatial velocities are [rot(3); lin(3)] (MuJoCo conventions).
 *  - `stream` is a cudaStream_t passed as void*; every call only ENQUEUES work on it (no host sync)
 *    unless documented otherwise.  Inputs are not retained after the call returns (tables are copied).
 *  - Return value: 0 on success, non-zero on error; om_last_error() returns a thread-local message.
 *    There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef OM_B200_H
#define OM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OM_ABI_VERSION 2

/* mjtJoint values (mujoco==2.3.6) */
#define OM_JNT_FREE 0
#define OM_JNT_BALL 1
#define OM_JNT_SLIDE 2
#define OM_JNT_HINGE 3

#define OM_MAX_BODY 48
#define OM_MAX_JNT 48
#define OM_MAX_SITE 8

const char* om_last_error(void);
int om_abi_version(void);
/* number of kernels launched by this library since load / since om_reset_launch_count() */
long long om_launch_count(void);
void om_reset_launch_count(void);
/* Tuning / test hook: force a kernel variant ("play_chunk", "h1_split", "a3_split", "a3_feat_minb", "serial_scan",
 * "disc_vail2", "disc_pg2"; -1 / 0 = automatic).  The same knobs are initialised ONCE, when the library is loaded, from the
 * OM_PLAY_CHUNK, OM_H1_SPLIT, ... environment variables; no launch path calls getenv.
 * "disc_vail2" selects the VAIL discriminator kernel: -1 / 4 disc_vail4_kernel (one CTA per SM, A operand in tensor
 * memory: the default), 6 / 5 / 7 its variants (layer-1 blocks released head by head / rotating accumulator blocks /
 * alternating producer warpgroups), 1 disc_vail2_kernel (two CTAs per SM, shared-memory operands), 3 disc_vail3_kernel
 * (two CTAs per SM, A in tensor memory), 0 the kernels that also serve GAIL ("disc_pg2" 0: one producer warpgroup). */
int om_debug_set(const char* knob, int value);

/* ------------------------------------------------------------------------------------------------
 * Model constants.  Replaces the mjModel produced by MuJoCo's MJCF compiler
 * (loco_env_base.py:143-155 MultiMuJoCo.__init__; UnitreeH1.py:70-111).  All pointers are HOST.
 * Doubles are converted to float on upload. */
typedef struct OmModelDesc {
  const char* name;            /* "UnitreeH1" / "StickFigureA3" select a specialised kernel when the
                                  tables match the ones it was generated from; anything else runs the
                                  table-driven kernel */
  int nbody, njnt, nsite, nq, nv;
  const int32_t* body_parentid;  /* [nbody] */
  const int32_t* body_rootid;    /* [nbody] */
  const int32_t* body_jntadr;    /* [nbody], -1 if none */
  const int32_t* body_jntnum;    /* [nbody] */
  const double* body_pos;        /* [nbody,3] */
  const double* body_quat;       /* [nbody,4] normalised */
  const double* body_ipos;       /* [nbody,3] */
  const double* body_mass;       /* [nbody] */
  const int32_t* jnt_type;       /* [njnt] */
  const int32_t* jnt_qposadr;    /* [njnt] */
  const int32_t* jnt_dofadr;     /* [njnt] */
  const double* jnt_axis;        /* [njnt,3] */
  const double* jnt_pos;         /* [njnt,3] */
  const double* qpos0;           /* [nq] */
  const int32_t* site_bodyid;    /* [nsite] */
  const double* site_pos;        /* [nsite,3] */
  const double* site_quat;       /* [nsite,4] */
} OmModelDesc;

typedef struct OmModel OmModel;
int om_model_create(const OmModelDesc* desc, OmModel** out);
void om_model_destroy(OmModel* m);
/* 1 when the model is served by a generated (topology-specialised) kernel, 0 for the table-driven one */
int om_model_is_specialised(const OmModel* m);
/* Which UnitreeH1 model the tables are, for the fused playback / live-step kernels (recognised by exact table match):
 * 1 the default (arms disabled), 2 no back joint, 3 arms, 4 arms without the back joint, 5 / 6 / 7 / 8 carrying a
 * 0.1 / 1 / 5 / 10 kg weight; 0 for any other model.  Only the default model is also `specialised`. */
int om_model_h1_variant(const OmModel* m);
/* Per-env mass of one body: afterwards om_fk, om_h1_step, om_h1_play_from_velocity, om_h1_play_trajectory and
 * om_h1_live_step on this model read body `body`'s mass of env i from mass[i] (DEVICE, [ld] float32, n <= ld at every
 * call) instead of the tables.  Accepted for the UnitreeH1 carry models (om_model_h1_variant 5-8) and their "weight" body
 * (the only body whose mass differs between them), for which it selects kernels with that mass as a runtime argument; any
 * other model or body is an error.  The binding lasts for the model's life (the pointer is read at every call, so a CUDA
 * graph captured afterwards stays valid); rebinding to another buffer is an error. */
int om_model_bind_env_body_mass(OmModel* m, int body, const float* mass, int ld);

/* ------------------------------------------------------------------------------------------------
 * K1: forward kinematics + COM + COM velocity = the subset of mujoco.mj_forward the path consumes
 * (mj_kinematics + mj_comPos + mj_comVel; call sites loco_env_base.py:410,525,1160 and
 * mujoco_robot_interface.py:468).  Any output pointer may be NULL.
 *   qpos [nq][ld], qvel [nv][ld] -> xpos [nbody*3][ld], xquat [nbody*4][ld], site_xpos [nsite*3][ld],
 *   site_xmat [nsite*9][ld], cvel [nbody*6][ld], subtree_com [3][ld] (COM of the tree of body 1).
 * force_generic != 0 runs the table-driven kernel even when a specialised one exists. */
int om_fk(const OmModel* m, const float* qpos, const float* qvel, int n, int ld,
          float* xpos, float* xquat, float* site_xpos, float* site_xmat, float* cvel, float* subtree_com,
          int force_generic, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2 (H1 flavour): the tail of mushroom_rl MuJoCo.step for UnitreeH1 after the physics:
 *   ObservationHelper._build_obs + LocoEnvBase._create_observation (loco_env_base.py:737-767),
 *   UnitreeH1._has_fallen (UnitreeH1.py:162-203) through is_absorbing (base_humanoid_robot.py:246-260),
 *   TargetVelocityReward on the PREVIOUS observation (utils/reward.py:66-74), fused with K1.
 * obs_perm[k] (HOST, length n_obs_q) = qpos/qvel address of observation-spec entry k; the emitted
 * observation drops the first two position entries: obs has 2*n_obs_q-2 components.
 * prev_x_vel [ld] = row x_vel_idx of the previous observation.  FK outputs may be NULL. */
typedef struct OmH1Spec {
  int n_obs_q;                 /* 17 */
  int32_t obs_perm[32];
  int x_vel_idx;               /* index of dq_pelvis_tx in the emitted observation (15) */
  float target_velocity;       /* 1.25 walk / 2.5 run (base_humanoid_robot.py:149-154) */
  int use_absorbing_states;    /* base_humanoid_robot.py:260 */
} OmH1Spec;

int om_h1_step(const OmModel* m, const OmH1Spec* spec, const float* qpos, const float* qvel,
               const float* prev_x_vel, int n, int ld,
               float* xpos, float* xquat, float* site_xpos, float* cvel,
               float* obs, float* reward, uint8_t* absorbing, void* stream);

/* LocoEnvBase.set_sim_state (loco_env_base.py:659-684) for joint-only specs: sample [2*n_obs_q][ld] in observation-spec
 * order (positions then velocities) -> qpos [nq][ld], qvel [nv][ld] in MJCF order (the inverse of the gather above). */
int om_set_sim_state(const OmModel* m, const OmH1Spec* spec, const float* sample, int n, int ld, float* qpos, float* qvel,
                     void* stream);

/* has_fallen over a batch of observations (create_dataset check, loco_env_base.py:950-957) */
int om_h1_has_fallen(const float* obs, int n, int ld, uint8_t* fallen, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K3: reference-trajectory table and per-env integer state.  Replaces utils/trajectory.py
 * reset_trajectory :289-323, get_current_sample :381-387, get_next_sample :389-401 and the wrap ->
 * reset policy of loco_env_base.py:534-537, :639-657.
 * table_host: float64 [K][n_traj][T] (the layout of Trajectory.trajectories after resampling).
 * Channels 0 and 1 (root x, y) are kept in float64 on the device because every reset re-centres them. */
typedef struct OmTraj OmTraj;
int om_traj_create(const double* table_host, int K, int n_traj, int T, OmTraj** out);
void om_traj_destroy(OmTraj* t);

/* Reset envs.  mask (may be NULL = all): reset env i iff mask[i] != 0.  forced_traj / forced_step (may be
 * NULL) >= 0 override the random draw (reset_trajectory(substep_no, traj_no)).  Random draws follow the
 * Philox contract (oracle/philox.py): key = seed, counter = (env_id0 + i, reset_count[i], 0, 0).
 * State: traj_no, step_no [n] int32, reset_count [n] uint32 (incremented), xy_off [2][ld] float64.
 * sample (may be NULL) [K][ld] = the current sample after the reset. */
int om_traj_reset(const OmTraj* t, uint64_t seed, uint32_t env_id0, const uint8_t* mask,
                  const int32_t* forced_traj, const int32_t* forced_step,
                  int32_t* traj_no, int32_t* step_no, uint32_t* reset_count, double* xy_off,
                  float* sample, int n, int ld, void* stream);
/* get_current_sample for every env */
int om_traj_current(const OmTraj* t, const int32_t* traj_no, const int32_t* step_no, const double* xy_off,
                    float* sample, int n, int ld, void* stream);
/* get_next_sample.  auto_reset != 0: an env that reaches the end of its trajectory is reset
 * (wrapped[i] = 1) exactly as loco_env_base.py:534-537 does.  auto_reset == 0: such an env keeps
 * step_no == T and its sample row is left untouched (the reference returns None), wrapped[i] = 1. */
int om_traj_next(const OmTraj* t, uint64_t seed, uint32_t env_id0, int auto_reset,
                 int32_t* traj_no, int32_t* step_no, uint32_t* reset_count, double* xy_off,
                 float* sample, uint8_t* wrapped, int n, int ld, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused playback: LocoEnvBase.play_trajectory_from_velocity (loco_env_base.py:444-560) for n envs,
 * one episode of n_steps steps per call (call once per episode).  end_episode_reset is a bit set: OM_PLAY_END_RESET
 * performs the end-of-episode reset (:555-557), OM_PLAY_START_RESET the reset() with which every call of the reference
 * begins (:481; sample = get_current_sample(), curr_qpos = sample[:len_qpos]) -- inside the same launches.  Per step: Euler step of the NQ coordinates (:515-519),
 * set_sim_state (:659-684), K1, next sample / wrap reset (:532-537), observation from the next sample
 * (:539), has_fallen (:541), TargetVelocityReward on the previous observation.
 * State in/out: traj_no, step_no, reset_count, xy_off, curr_qpos [n_obs_q][ld] (spec order, float64),
 * pending [K][ld] (the `sample` variable of the loop), prev_x_vel [ld].
 * Outputs (any may be NULL), time-major [n_steps][C][ld]: xpos, xquat, site_xpos, cvel, obs, reward,
 * fallen (uint8), traj_no_t / step_no_t (int32 state after each step).
 * Any model with om_model_h1_variant() != 0; spec->n_obs_q must be its NQ (17 default and carry, 16 no back joint, 25 arms,
 * 24 arms without the back joint), t->K = 2 NQ and obs_perm the model's own spec order.  Per-step sizes: obs [2 NQ - 2],
 * xpos [3 nbody], xquat [4 nbody], cvel [6 nbody], site_xpos [3 nsite] (nbody 21, 22 with a carried weight; nsite 1). */
#define OM_PLAY_END_RESET 1
#define OM_PLAY_START_RESET 2
typedef struct OmPlayState {
  int32_t* traj_no; int32_t* step_no; uint32_t* reset_count; double* xy_off;
  double* curr_qpos; float* pending; float* prev_x_vel;
} OmPlayState;
typedef struct OmPlayOut {
  float* xpos; float* xquat; float* site_xpos; float* cvel; float* obs; float* reward;
  uint8_t* fallen; int32_t* traj_no_t; int32_t* step_no_t;
  double* obs_moments;   /* [2 nobs + 1] float64 or NULL (nobs = 2 NQ - 2: 65 values for the default model, 97 with arms):
                            S1 fused into the playback -- sum[nobs], sumsq[nobs] and count of the emitted observations are
                            ADDED (om_moments layout and semantics: zero it first, all-reduce it after) */
} OmPlayOut;
int om_h1_play_from_velocity(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed,
                             uint32_t env_id0, double dt, int n_steps, int end_episode_reset,
                             const OmPlayState* state, const OmPlayOut* out, int n, int ld, void* stream);

/* Fused LocoEnvBase.play_trajectory (loco_env_base.py:338-442): like the call above, but every step FORCES the model to the
 * current trajectory sample (:408) instead of integrating its velocities; state->curr_qpos is not used (may be NULL). */
int om_h1_play_trajectory(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed, uint32_t env_id0,
                          int n_steps, int end_episode_reset, const OmPlayState* state, const OmPlayOut* out, int n, int ld,
                          void* stream);

/* Fused LIVE step: one env step of a trajectory-driven rollout in one kernel -- get_next_sample with the wrap -> reset
 * policy (trajectory.py:389-401, loco_env_base.py:534-537), set_sim_state (:659-684), K1, _create_observation
 * (:737-767), has_fallen (UnitreeH1.py:162-203) and TargetVelocityReward on the PREVIOUS observation (mushroom_rl
 * MuJoCo.step: reward(self._obs, action, cur_obs, absorbing), then self._obs = cur_obs).  Replaces the three launches
 * om_traj_next -> om_set_sim_state -> om_h1_step, whose sample and qpos / qvel round-tripped through HBM.
 * State in/out: traj_no, step_no [n], reset_count [n], xy_off [2][ld] float64, prev_x_vel [ld] (row x_vel_idx of the
 * previous observation in, of this step's observation out).  Outputs, single step, any may be NULL: qpos / qvel [NQ][ld]
 * (the MjData mirrors), xpos [3 nbody][ld], xquat [4 nbody][ld], site_xpos [3 nsite][ld], cvel [6 nbody][ld],
 * obs [2 NQ - 2][ld], reward [ld], absorbing [ld] uint8, wrapped [ld] uint8 (1 where the trajectory wrapped and the env was
 * reset); the default model: NQ 17, nbody 21, nsite 1.  Same models and spec rules as om_h1_play_from_velocity, and
 * x_vel_idx = NQ - 2.  Safe to capture in a CUDA graph (no host synchronisation, no allocation). */
typedef struct OmLiveState {
  int32_t* traj_no; int32_t* step_no; uint32_t* reset_count; double* xy_off; float* prev_x_vel;
} OmLiveState;
typedef struct OmLiveOut {
  float* qpos; float* qvel; float* xpos; float* xquat; float* site_xpos; float* cvel;
  float* obs; float* reward; uint8_t* absorbing; uint8_t* wrapped;
} OmLiveOut;
int om_h1_live_step(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed, uint32_t env_id0,
                    const OmLiveState* state, const OmLiveOut* out, int n, int ld, void* stream);

/* The model switch of a MultiMuJoCo reset() (loco_env_base.py:586-599) drawn per env, for n envs whose global ids start
 * at env_id0; count = the env object's number of model resets before this one.  Env i takes model
 *   random != 0:  Philox(key seed; counter env_id0 + i, count, 32, 0) word 0, times n_models, high 32 bits
 *                 (the om_traj_reset contract on stream 32 = utils/philox.py philox_randint)
 *   random == 0:  (env_id0 + i + count + 1) mod n_models  (round robin from model 0)
 * idx [n] int32 <- the model index, mass [n] float32 <- body_mass_host[idx] (HOST, [n_models] <= 16).  Feeds the buffer
 * bound with om_model_bind_env_body_mass; a plain stream-ordered launch. */
int om_h1_draw_models(uint64_t seed, uint32_t env_id0, uint32_t count, int n_models, int random,
                      const double* body_mass_host, int32_t* idx, float* mass, int n, void* stream);

/* Per-env reset of a UnitreeH1 batch: LocoEnvBase.reset (loco_env_base.py:568-604, setup :606-657) for a subset of the envs,
 * and mushroom_rl Core's reset on `last` (Core._step / _reset: last = absorbing or episode_steps >= horizon, then reset that
 * env alone).  For every env that resets:
 *   qpos = qpos0 of the model, qvel = 0 (mj_resetData); grf rows = 0 (mean_grf.reset(), :584);
 *   trajectory reset under the om_traj_reset contract (key seed, counter (env_id0 + i, reset_count[i], 0, 0); reset_count[i]
 *   += 1; forced_traj / forced_step >= 0 override the draw, as reset_trajectory(substep_no, traj_no) does);
 *   set_sim_state of the drawn sample (root x, y re-centred to 0); obs = its observation (sample keys 2..K-1, then grf = 0);
 *   prev_x_vel[i] = obs row spec->x_vel_idx; episode_step[i] = 0;
 *   with model_index: the env draws its own model (see below).
 * Modes:
 *   mask != NULL  (explicit): env i resets iff mask[i] != 0; nothing of another env is written except its obs row (below).
 *   mask == NULL  (auto-reset, after a step): episode_step[i] += 1, last[i] = absorbing[i] || episode_step[i] >= horizon,
 *                 env i resets iff last[i]; prev_x_vel[i] = obs row x_vel_idx for EVERY env.  absorbing, episode_step, last,
 *                 obs_in, obs and prev_x_vel are required.
 * obs (may be NULL in explicit mode) [obs_dim][ld] = the observation after the call: the new one for envs that reset, row i of
 * obs_in for the others (obs_in NULL: those rows are left alone; obs_in may equal obs).  obs_dim = 2 n_obs_q - 2 + n_grf.
 * Model draw (model_index != NULL; the per-env carried weight): env i's j-th partial reset, j = partial_resets[i] (then
 * incremented), takes model  random != 0: Philox(key seed; counter env_id0 + i, j, 33, 0) word 0 times n_models, high
 * 32 bits;  random == 0: (model_index[i] + 1) mod n_models;  and mass[i] = masses_host[model_index[i]].
 * qpos [nq][ld], qvel [nv][ld] of the model; the trajectory must have 2 n_obs_q keys.  No FK: the MjData mirrors (xpos ...)
 * are not written.  Every call only enqueues one kernel (no allocation, no host synchronisation): capturable in a CUDA graph
 * behind om_h1_step. */
typedef struct OmH1ResetArgs {
  const uint8_t* mask;                       /* [ld] explicit mode, or NULL = auto-reset mode */
  const uint8_t* absorbing; int horizon;     /* auto-reset mode: the step's absorbing flags [ld], info.horizon */
  int forced_traj, forced_step;              /* -1 = draw */
  int32_t* traj_no; int32_t* step_no; uint32_t* reset_count; double* xy_off;   /* the OmTraj state ([ld], xy_off [2][ld]) */
  float* qpos; float* qvel;
  const float* obs_in; float* obs; int obs_dim;
  float* prev_x_vel; int32_t* episode_step; uint8_t* last;   /* [ld]; episode_step may be NULL in explicit mode */
  float* grf; int n_grf;                     /* [n_grf][ld] or NULL */
  int32_t* partial_resets; int32_t* model_index; float* mass;   /* [ld] or all NULL */
  int n_models, random;
  const double* masses_host;                 /* [n_models] <= 16 */
} OmH1ResetArgs;
int om_h1_reset_envs(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed, uint32_t env_id0,
                     const OmH1ResetArgs* args, int n, int ld, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2 (A3 flavour): the tail of StickFigureA3.step (real_humanoid_robots/StickFigureA3.py:187-202) after
 * robot.step (= mj_step, which stays the reference's): WalkingTask.step (tasks/walking_task.py:246-293),
 * calc_reward (:74-110; terms tasks/rewards.py:27-40,65-83,85-102,121-126), done (:298-319) and get_obs
 * (StickFigureA3.py:144-178), with K1 fused in (the MjData fields are only written when asked for).
 * What the task reads from the contact solver enters as contact [4][ld]: left-foot GRF, right-foot GRF
 * (mujoco_robot_interface.py:275-297), min z of the foot-floor contact points (rewards.py:29-31), flags
 * (float-coded bits: 1 = any foot-floor contact, 2 = check_bad_collisions :393-399). */
typedef struct OmA3TaskDesc {
  int period;                    /* floor(2 * total_duration / control_dt) = 88 (walking_task.py:351) */
  int delay_frames;              /* floor(swing_duration / control_dt) = 30 (:336) */
  double target_radius;          /* 0.20 (:333) */
  double goal_height_ref;        /* 0.80 (StickFigureA3.py:110) */
  double goal_speed_ref;         /* 0 (walking_task.py:30) */
  double total_mass;             /* mj_getTotalmass */
  const double* clock_lut_host;  /* [period][4]: right/left foot force and velocity clocks evaluated at the integer
                                    phases (rewards.py:270-366), columns r_frc, r_vel, l_frc, l_vel */
  const double* init_qpos_host;  /* [25] nominal pose (environments/robot.py:61-80) */
} OmA3TaskDesc;
typedef struct OmA3Task OmA3Task;
int om_a3_task_create(const OmA3TaskDesc* desc, OmA3Task** out);
void om_a3_task_destroy(OmA3Task* t);

/* Per-env WalkingTask state.  ints [7][ld]: phase, t1, t2, target_reached_frames, mode (0 STANDING, 1 FORWARD),
 * len(sequence), target_reached.  sequence [20*4][ld]: footstep plan rows (x, y, z, theta), component
 * step*4 + c. */
typedef struct OmA3State { int32_t* ints; float* sequence; } OmA3State;
/* Outputs (any may be NULL), time-major over the n_steps of the call: obs [41], terms [6] (the weighted reward
 * terms in the reference's dict order), reward (their sum), done (uint8); MjData fields xpos [17*3],
 * xquat [17*4], site_xpos [2*3], site_xmat [2*9], cvel [17*6]. */
typedef struct OmA3Out {
  float* obs; float* terms; float* reward; uint8_t* done;
  float* xpos; float* xquat; float* site_xpos; float* site_xmat; float* cvel;
} OmA3Out;
/* n_steps == 1: one StickFigureA3.step tail on the post-physics state qpos [25][ld], qvel [24][ld].
 * n_steps > 1: replay of n_steps recorded post-physics states (qpos [n_steps][25][ld], ...), the task state
 * carried from step to step in registers. */
int om_a3_task_step(const OmModel* m, const OmA3Task* task, const float* qpos, const float* qvel, const float* contact,
                    int n_steps, const OmA3State* state, const OmA3Out* out, int n, int ld, void* stream);
/* The same step tail for a ROLLOUT BUFFER, finished with the discounted returns of PPOBuffer.finish_path
 * (rl/algos/ppo.py:68-84, bootstrap :195-196, advantage :335) -- BASELINE configs[2]: obs / reward / done + returns.  Same
 * results as om_a3_task_step followed by om_ppo_returns(out->reward, values, path_end, v_next, v_last, gamma, ...), enqueued
 * by ONE call (the scan kernel follows the task kernels on the same stream).  path_end NULL = the done flags of this call
 * (1 = terminated, bootstrap 0); out->reward and returns->ret are required. */
typedef struct OmA3Returns {
  const float* values; const float* v_next; const float* v_last; const uint8_t* path_end;
  float gamma;
  float* ret; float* adv;
} OmA3Returns;
int om_a3_task_rollout(const OmModel* m, const OmA3Task* task, const float* qpos, const float* qvel, const float* contact,
                       int n_steps, const OmA3State* state, const OmA3Out* out, const OmA3Returns* returns, int n, int ld,
                       void* stream);
/* StickFigureA3.reset_model (StickFigureA3.py:205-235) + WalkingTask.reset (walking_task.py:321-397) for the envs
 * selected by mask (NULL = all).  Draws follow the Philox contract: key = seed, counter = (env_id0 + i,
 * reset_count[i], 16 + block, 0), 15 blocks = 60 uniforms in the order documented in oracle/a3.py.
 * Writes qpos, qvel, the task state and (optionally) the first observation; reset_count[i] += 1. */
int om_a3_reset(const OmModel* m, const OmA3Task* task, uint64_t seed, uint32_t env_id0, const uint8_t* mask,
                uint32_t* reset_count, double iteration_count, float* qpos, float* qvel, const OmA3State* state,
                float* obs, int n, int ld, void* stream);
/* Auto-reset after a one-step om_a3_task_step: the path bookkeeping of the PPO sampler (rl/algos/ppo.py:150-198: a path
 * runs until done or max_traj_len steps, then the worker resets its env).  For every env i:
 *   traj_len[i] += 1;  trunc = max_traj_len > 0 && traj_len[i] >= max_traj_len;  last[i] = done[i] || trunc;
 *   path_end[i] = 1 if done[i] (bootstrap 0; wins over a truncation on the same step), 2 if trunc (bootstrap V(obs_in
 *   row i), the step's own observation), else 0 -- the codes om_ppo_returns reads;
 *   if last[i]: the reset of om_a3_reset (same draw contract: counter (env_id0 + i, reset_count[i], 16 + block, 0), then
 *   reset_count[i] += 1; step height from iteration_count) writes qpos, qvel, the task state and obs row i; traj_len[i] = 0;
 *   otherwise obs row i = obs_in row i (obs_in may equal obs).
 * Nothing of an env that does not reset is written except its obs row, traj_len, last and path_end.  obs_in / obs [41][ld];
 * done, last, path_end [ld] uint8; traj_len [ld] int32.  Every pointer is required.  The call only enqueues one kernel (no
 * allocation, no host synchronisation): capturable in a CUDA graph behind om_a3_task_step. */
typedef struct OmA3AutoResetArgs {
  const uint8_t* done;          /* [ld] the step's done flags (OmA3Out.done) */
  int max_traj_len;             /* 0 = no limit: only done ends a path */
  double iteration_count;       /* env.robot.iteration_count (reset step heights, walking_task.py:378) */
  uint32_t* reset_count; int32_t* traj_len;
  float* qpos; float* qvel;     /* [25][ld], [24][ld] */
  OmA3State state;
  const float* obs_in; float* obs;
  uint8_t* last; uint8_t* path_end;
} OmA3AutoResetArgs;
int om_a3_autoreset(const OmModel* m, const OmA3Task* task, uint64_t seed, uint32_t env_id0, const OmA3AutoResetArgs* args,
                    int n, int ld, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K4: discriminator reward  r = -log(1 - sigmoid(D(s)) + 1e-8)  (GAIL.make_discrim_reward,
 * imitation_lib/imitation/gail_TRPO.py:320-327; VAIL discrim_output vail_TRPO.py:18-21) for the two networks
 * the reference configures for UnitreeH1 (examples/imitation_learning/utils.py:151-179, confs.yaml:113-130):
 *   kind 0 VAIL  VariationalNet (networks.py:258-284): n_in -relu-> 256 -relu-> 128 -> mu[128], logvar[128],
 *                z = mu + exp(logvar/2) * eps (:21-24), d = wd . z + bd
 *   kind 1 GAIL  DiscriminatorNetwork (:208-234): n_in -tanh-> 512 -tanh-> 256 -> 1
 * n_in = 1..64: the kinematic observation of the env's UnitreeH1 variant (env.get_kinematic_obs_mask(): 32 for the
 * default model and the carry task, 30 without the back joint, 48 with arms, 46 with arms and without the back joint);
 * other values are refused.  The kernel variants forced through the "disc_vail2" / "disc_pg2" knobs (om_debug_set)
 * take n_in = 32 only: with another width om_disc_reward / om_disc_forward fail (om_last_error) and launch nothing.
 * Weights are HOST pointers, row-major [out][in] float32 (torch.nn.Linear.weight), copied at create time.
 * The contraction runs on tcgen05 tensor cores as 3xTF32 with fp32 accumulation (fp32-level results). */
typedef struct OmDiscDesc {
  int kind, n_in, n_h1, n_h2, z_size;
  const float* w1; const float* b1;      /* [n_h1][n_in], [n_h1] */
  const float* w2; const float* b2;      /* [n_h2][n_h1], [n_h2] */
  const float* wmu; const float* bmu;    /* VAIL: [z][n_h2], [z] */
  const float* wlv; const float* blv;    /* VAIL: [z][n_h2], [z] */
  const float* wd; const float* bd;      /* VAIL decoder [1][z] / GAIL output layer [1][n_h2]; [1] */
} OmDiscDesc;
typedef struct OmDisc OmDisc;
int om_disc_create(const OmDiscDesc* desc, OmDisc** out);
void om_disc_destroy(OmDisc* d);
/* s [n_in][ld] observations (SoA); mean / std [n_in] = the Standardizer snapshot to apply (networks.py:73-74; the
 * running sums are updated by the caller with om_moments); eps [z][ld] = the reparameterisation noise (VAIL; NULL
 * means z = mu); reward [ld]; d_out [ld] (may be NULL) = the raw discriminator logit. */
int om_disc_reward(const OmDisc* d, const float* s, const float* mean, const float* std, const float* eps, int n, int ld,
                   float* reward, float* d_out, void* stream);
/* The same forward pass for the discriminator FIT (N2; GAIL._fit_discriminator gail_TRPO.py:167-220 calls the network
 * on [policy batch; expert batch]): any of reward / d_out (logit) / kl_out may be NULL.  kl_out [ld] (VAIL only) =
 * VDBLoss.kl_divergence (imitation_lib/utils/math.py:83-86): 0.5 * sum_j (mu_j^2 + exp(logvar_j) - logvar_j - 1). */
int om_disc_forward(const OmDisc* d, const float* s, const float* mean, const float* std, const float* eps, int n, int ld,
                    float* reward, float* d_out, float* kl_out, void* stream);
/* Loss statistics of one discriminator fit batch: logit [n_plcy + n_demo] (policy samples first, like the reference's
 * np.concatenate([plcy, demo])), target [n] or NULL (= 0 for policy, 1 for expert samples), kl [n] or NULL.
 * ACCUMULATES into sums[9] (float64, zero it first; all-reduce it across ranks before reading):
 *   0 sum bce = max(x,0) - x t + log(1 + exp(-|x|))      GailDiscriminatorLoss.forward math.py:22-31
 *   1 sum logit_bernoulli_entropy = (1 - sigmoid x) x - logsigmoid x                      math.py:33-38
 *   2 sum kl                                                  3 policy samples with sigmoid < 0.5
 *   4 expert samples with sigmoid > 0.5                       5 / 6 sum sigmoid over policy / expert samples
 *   7 / 8 number of policy / expert samples
 * dlogit [n] (may be NULL): d/dx of  sum(bce) - entcoeff * sum(entropy)  per sample, i.e. (sigmoid x - t) +
 * entcoeff x sigmoid x (1 - sigmoid x); divide by the global n for the gradient of the mean loss. */
int om_disc_loss_stats(const float* logit, const float* target, const float* kl, int n_plcy, int n_demo, float entcoeff,
                       double* sums, float* dlogit, void* stream);
/* Expert minibatch (N2; minibatch_generator(batch, demonstrations["states"], ["next_states"]) at
 * gail_TRPO.py:175-206 = the first `batch` rows of a fresh random permutation): sample b of draw `draw` reads dataset row
 * pi_e(b mod n_src) with e = b / n_src, pi_e a keyed 4-round Feistel permutation of [0, n_src) with cycle walking,
 * round keys = Philox(seed; e, draw, stream 48) -- every epoch e is a sample WITHOUT replacement (contract:
 * oracle/learner.py expert_indices).  src [D][ld_src] holds n_src + next rows (next_states = rows shifted by one,
 * trajectory.py:170-171); out / out_next [D][ld_out] (out_next and idx_out may be NULL). */
int om_expert_minibatch(const float* src, int n_src, int ld_src, int D, uint64_t seed, uint32_t draw, int batch, float* out,
                        float* out_next, int32_t* idx_out, int ld_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K5: returns / advantages over a time-major rollout buffer [T][ld].
 * om_ppo_returns: PPOBuffer.finish_path (rl/algos/ppo.py:68-84) with the bootstrap of :195-196.
 *   path_end[t][i] (may be NULL): 0 = the path continues, 1 = it terminated at step t (bootstrap 0),
 *   2 = it was truncated at step t (max_traj_len, ppo.py:180) and bootstraps with v_next[t][i].
 *   The buffer end (t == T-1) always closes the path: bootstrap 0 if path_end == 1, else v_next (flag 2)
 *   or v_last[i] (= (not done) * V(s_T)).  ret = discounted return, adv = ret - values (:335).
 * om_gae: mushroom_rl.utils.value_functions.compute_gae (called gail_TRPO.py:126): per env,
 *   adv_t = r_t + gamma*v_next_t*(1-absorbing_t) - v_t            if last_t or t == T-1
 *         = r_t + gamma*v_next_t - v_t + gamma*lam*adv_{t+1}      otherwise;  v_target = adv + v. */
int om_ppo_returns(const float* rewards, const float* values, const uint8_t* path_end, const float* v_next,
                   const float* v_last, float gamma, int T, int n, int ld, float* ret, float* adv, void* stream);
int om_gae(const float* rewards, const float* v, const float* v_next, const uint8_t* absorbing,
           const uint8_t* last, float gamma, float lam, int T, int n, int ld,
           float* adv, float* v_target, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K6: moment partial sums (Standardizer.update_mean_std networks.py:76-81; get_normalization_params
 * rl/envs/normalize.py:48; advantage mean/std ppo.py:336, gail_TRPO.py:128).
 * x is [rows][C][ld] (rows = T or 1); sums over rows and envs.  out [2*C+1] float64 on the DEVICE:
 * sum[C], sumsq[C], count -- ADDED to the existing contents (zero it first), so that a multi-GPU caller
 * can all-reduce the same buffer with ncclAllReduce(sum). */
int om_moments(const float* x, int rows, int C, int n, int ld, double* out, void* stream);
/* stats[0] = mean, stats[1] = std + eps from a one-component moment buffer [sum, sumsq, count] (device);
 * unbiased != 0 -> torch.std (ppo.py:336, eps 1e-5), 0 -> np.std (gail_TRPO.py:128, eps 1e-8). */
int om_adv_stats(const double* moments, int unbiased, double eps, double* stats, void* stream);
/* mean[C] and denominator[C] (float64, and / or float32 copies; any output may be NULL) from a moment buffer
 * [sum[C], sumsq[C], count] on the device -- one small kernel instead of a chain of host-framework ops:
 *   kind 0 "standardizer"  sqrt(max(E[x^2] - mean^2, 1e-2))                 networks.py:76-81
 *   kind 1 "ppo_obs"       sqrt(max(var, 0) + 1e-8)                         rl/envs/normalize.py:48
 *   kind 2 "adv_ppo"       sqrt(max(var, 0) * n / (n - 1)) + 1e-5           rl/algos/ppo.py:336 (torch.std, unbiased)
 *   kind 3 "adv_gail"      sqrt(max(var, 0)) + 1e-8                         gail_TRPO.py:128 (np.std) */
int om_moment_stats(const double* moments, int C, int kind, double* mean, double* denom, float* mean32, float* denom32,
                    void* stream);
/* y = (x - mean) / denom element-wise for a [rows][ld] array with device scalars stats[0]=mean,
 * stats[1]=denom (advantage normalisation); in place allowed. */
int om_normalize(const float* x, const double* stats, int rows, int n, int ld, float* y, void* stream);

/* ------------------------------------------------------------------------------------------------
 * N1 (next row: the step immediately before the path): what feeds mj_step.
 * om_action_affine: LocoEnvBase._preprocess_action (loco_env_base.py:1050-1069): ctrl = action * delta + mean
 *   (delta, mean = half range / mid point of the actuator ctrlrange, loco_env_base.py:165-175).
 * om_pd_torque: JVRC.step + do_simulation (environments/robot.py:88-115) around MujocoRobotInterface.step_pd
 *   (interfaces/mujoco_robot_interface.py:425-443):  p = target (+ motor_offset when add_offset != 0),
 *   tau = kp (p - q_act) + kd (v - dq_act),  ctrl = tau / gear.  vel_target NULL = zeros (robot.py:111).
 * action / target / ctrl are [nu][ld]; qpos [nq][ld], qvel [nv][ld]. */
typedef struct OmActionSpec { int nu; float delta[32], mean[32]; } OmActionSpec;
typedef struct OmPdSpec {
  int nu;
  int32_t qposadr[32], dofadr[32];   /* qpos / qvel address of each actuated joint */
  float kp[32], kd[32], gear[32], offset[32];
} OmPdSpec;
int om_action_affine(const OmActionSpec* spec, const float* action, int n, int ld, float* ctrl, void* stream);
int om_pd_torque(const OmPdSpec* spec, const float* target, const float* vel_target, const float* qpos, const float* qvel,
                 int add_offset, int n, int ld, float* ctrl, void* stream);

/* ------------------------------------------------------------------------------------------------
 * N3 (next row, consumer side): the mirror-symmetry transforms of the PPO mirror loss (rl/algos/ppo.py:232-282 through
 * rl/envs/wrappers.py:51-72 SymmetricEnv.mirror_observation / mirror_action / mirror_clock_observation).
 * `mirrored` lists (StickFigureA3.py:118-129) encode a signed permutation: y[|m_i|] = sign(m_i) * x[i]
 * (wrappers.py:75-82; index 0 is written 0.1 / -0.1 there).  negate[j] != 0 marks clock rows, whose mirrored value is
 * sin(arcsin(y_j) + pi) = -y_j (wrappers.py:67-69).  x, y are [numel][ld]; y must not alias x. */
typedef struct OmMirrorSpec { int numel; int32_t index[64]; float sign[64]; uint8_t negate[64]; } OmMirrorSpec;
int om_mirror(const OmMirrorSpec* spec, const float* x, int n, int ld, float* y, void* stream);
/* The minibatch losses of PPO.update_policy (rl/algos/ppo.py:231-282) from the quantities the actor / critic produced,
 * one pass: logp, old_logp, adv, mask (NULL = 1), values / returns (NULL: no value loss) are [n]; entropy [nu][ld] (NULL:
 * none) = pdf.entropy(); act = policy(obs), act_mirror = policy(mirror(obs)) [nu][ld] (NULL: no mirror loss), with
 * action_mirror = the signed permutation of mirror_action (NULL: act_mirror is already mirrored).
 * ACCUMULATES into sums[7] (float64; zero it, all-reduce it across ranks, then):
 *   actor_loss = -sums[0]/n          entropy_penalty = -sums[1]/(n nu)     critic_loss = vf_coeff sums[2]/n
 *   approx_kl = sums[3]/n            mirror_loss = sums[4]/(n nu)           clip_fraction = sums[5]/n        n = sums[6]
 * dlogp / dvalues [n] (may be NULL) = d actor_loss / d log_probs and d critic_loss / d values with the LOCAL n as the
 * mean's denominator (rescale by n_local / n_global under data parallelism). */
int om_ppo_loss_stats(const float* logp, const float* old_logp, const float* adv, const float* mask, const float* values,
                      const float* returns, const float* entropy, const float* act, const float* act_mirror,
                      const OmMirrorSpec* action_mirror, int nu, int n, int ld, float clip, float vf_coeff, double* sums,
                      float* dlogp, float* dvalues, void* stream);

/* ------------------------------------------------------------------------------------------------
 * S1 exchange over NVLink peer memory (one process per GPU): sum of <= 128 float64 values over the ranks, the path's only
 * collective (where the reference reduces its moment sums: rl/envs/normalize.py:48, rl/algos/ppo.py:336,
 * gail_TRPO.py:128, networks.py:76-81).  create: allocates this rank's mailbox and returns its CUDA IPC handle
 * (OM_MAILBOX_HANDLE_BYTES bytes) for the caller to all-gather by any means; connect: maps every peer's mailbox;
 * allreduce: one kernel on `stream` (stores to every mailbox, system-scope flags, rank-ordered sum: identical bits on
 * every rank; in and out are device pointers, may alias).  Every rank must issue the same sequence of calls.  A round in
 * which a peer does not show up within the timeout (default 30 s; env OM_MAILBOX_TIMEOUT_MS at create time or
 * om_mailbox_set_timeout_ms; 0 = wait for ever) is given up on that rank: its whole output vector is NaN (never a
 * partial sum) and the word read by om_mailbox_timed_out is set.  om_mailbox_timed_out synchronises with the device,
 * reports whether a round gave up since the last call and clears the word. */
#define OM_MAILBOX_HANDLE_BYTES 64
typedef struct OmMailbox OmMailbox;
int om_mailbox_create(int world, int rank, OmMailbox** out, unsigned char* handle_out);
int om_mailbox_connect(OmMailbox* mb, const unsigned char* all_handles);
int om_mailbox_allreduce(OmMailbox* mb, const double* in, double* out, int n, void* stream);
int om_mailbox_set_timeout_ms(OmMailbox* mb, double ms);
int om_mailbox_timed_out(OmMailbox* mb, int* flag);
void om_mailbox_destroy(OmMailbox* mb);

#ifdef __cplusplus
}
#endif
#endif /* OM_B200_H */
