/*
 * usim.h — C ABI of the B200-native batched Ultrasound environment.
 *
 * This is the drop-in boundary for ONE hot path of
 * hermanjakobsen/robotic-ultrasound-imaging: one control step of the
 * robosuite-style `Ultrasound` env (OSC_POSE -> arm dynamics -> probe /
 * soft-torso contact -> constraint solve -> integrate -> reward / obs).
 *
 * The reference has no FFI of its own for this path: it reaches the physics
 * through mujoco-py (`sim.forward()`, `sim.step()`, `sim.data.*`) and robosuite
 * (`MujocoEnv.step`, OSC controller), see SURVEY.md §8(b).  Each entry point
 * below names the reference call site it replaces (paths relative to the
 * reference checkout).
 *
 * Conventions
 *   - plain C, no torch types; every `*_dev` pointer is DEVICE memory owned by
 *     the caller, every other pointer is HOST memory.
 *   - return 0 = OK, negative = error (message via usim_last_error()).
 *   - one handle per (process, GPU); calls are stream-ordered on the given
 *     stream, not thread-safe, and never synchronise the device unless stated.
 *     Use ONE stream for the stream-taking calls of a handle (or order your
 *     streams yourself).  usim_step_host works on a private stream: it waits
 *     (cudaStreamWaitEvent) for the last usim_reset / usim_step /
 *     usim_forward / usim_set_state issued on a caller's stream and synchronises its own
 *     stream before returning, so the two kinds of call may be mixed freely.
 *   - no CPU fallback: usim_create fails if no sm_100-class device is present.
 *   - quaternions are (w,x,y,z) in qpos (MuJoCo), (x,y,z,w) where robosuite
 *     hands them to the task code (obs[15:19]).
 */
#ifndef USIM_H_
#define USIM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define USIM_ABI_VERSION 2
#define USIM_OBS_DIM 19      /* robot0_proprio-state, ultrasound.py:363-401 */
#define USIM_TASK_DIM 48     /* per-env task-state record, layout below */
#define USIM_MAX_ACTION 7
#define USIM_NV_ARM 7
#define USIM_MAX_CONTACTS 128 /* per env (reference: nconmax 5000 for the whole scene) */

/* impedance modes of the OSC_POSE controller (rl_config.yaml:41, main.py:33) */
enum { USIM_MODE_FIXED = 0, USIM_MODE_TRACKING = 1, USIM_MODE_VARIABLE_Z = 2, USIM_MODE_WRENCH = 3 };

/* task-state record (float), one per env; see DESIGN.md §3 */
enum {
  USIM_TS_TRAJ_START = 0,  /* 3 */
  USIM_TS_TRAJ_END = 3,    /* 3 */
  USIM_TS_U0 = 6,          /* initial_traj_step, ultrasound.py:443 */
  USIM_TS_STIFFNESS = 7,   /* solrefsmooth[0] magnitude, ultrasound.py:293 */
  USIM_TS_DAMPING = 8,     /* solrefsmooth[1] magnitude, ultrasound.py:294 */
  USIM_TS_VEL_MEAN = 9,    /* ultrasound.py:474,538 */
  USIM_TS_FZ_MEAN = 10,    /* ultrasound.py:477,546 */
  USIM_TS_FZ_PREV = 11,    /* ultrasound.py:468,543 */
  USIM_TS_DFZ = 12,        /* ultrasound.py:471,542 */
  USIM_TS_TOUCHED = 13,    /* has_touched_torso, ultrasound.py:434,733 */
  USIM_TS_TIMESTEP = 14,   /* MujocoEnv.timestep */
  USIM_TS_TRAJ_PT = 15,    /* 3, ultrasound.py:447,532 */
  USIM_TS_INIT_JOINT = 18, /* 7, controller.initial_joint, ultrasound.py:465 */
  USIM_TS_EPISODE = 25,    /* episode counter (RNG key) */
  USIM_TS_DONE = 26,       /* 1 after a terminal step until reset */
  USIM_TS_POS_ERR = 27,    /* 2, cached by reward(), ultrasound.py:247 */
  USIM_TS_ORI_ERR = 29,    /* cached by reward(), ultrasound.py:251 */
  USIM_TS_IN_CONTACT = 30, /* probe∩torso contact at last forward */
  USIM_TS_SPARE = 31,
  USIM_TS_GOAL_ORI = 32,   /* 9, OSC goal_ori (row-major); persists when the ori delta is 0 [robosuite osc.set_goal] */
  USIM_TS_GOAL_POS = 41    /* 3, OSC goal_pos of the current policy step */
};

/* Scene description: flat float64/int32 arrays produced by
 * robotic-ultrasound-imaging_b200/model.py (the "MJCF compiler" of this path;
 * replaces robosuite's XML merge + MuJoCo's compiler, ultrasound.py:272-321). */
typedef struct usim_model {
  int32_t nbody, nq, nv, npart, npair, soft;
  int32_t narm, reserved0; /* real arm joints: 7 (Panda) or 6 (UR5e: the seventh arm slot is an inert, decoupled degree of freedom) */
  int32_t table_body, link1_body, hand_body, probe_body, torso_body, part_body0;
  /* generic kinematic tree (oracle / invweight computation) */
  const int32_t *body_parent, *body_jnt_type, *body_qposadr, *body_dofadr; /* [nbody] */
  const double *body_pos, *body_quat, *body_mass, *body_ipos, *body_inertia, *body_jnt_axis;
  const double *dof_damping; /* [nv] */
  const double *jnt_range;   /* [7][2] arm */
  const double *ctrl_range;  /* [7] symmetric */
  const double *qpos0;       /* [nq] */
  /* collision geometry */
  const double *probe_seg;   /* [2][3] in probe-body frame */
  const double *part_pos;    /* [npart][3] in torso frame */
  const double *part_axis;   /* [npart][3] */
  const double *part_seg_outer, *part_seg_inner; /* [npart][3] in particle-body frame */
  const int32_t *eq_pairs;   /* [npair][2] "smooth" equalities */
  const int32_t *part_nbr;   /* [npart][6] neighbour particle or -1 */
  /* constraint regularisation constants at qpos0 */
  const double *dof_invweight0;  /* [nv] */
  const double *body_invweight0; /* [nbody][2] */
  /* specialised arm tables (CUDA kernels) */
  const double *arm_link; /* [7][22] */
  const double *arm_tool; /* [34] */
  double probe_radius, cap_radius, tendon_invweight0;
  double timestep, gravity[3], impratio, solref[2], solimp[5], solref_smooth[2];
  double table_top_z, table_half_xy, table_friction, probe_friction, particle_friction;
  double init_qpos[7];
  /* trajectory grid on the torso top (ultrasound.py:184-186,787-788,807): box 0.039/0.15/0.09, cylinder 0.041/0.15/0.05 */
  double top_torso_offset, traj_x_range, traj_y_range;
} usim_model;

/* Env + controller options: the kwargs of `suite.make("Ultrasound", ...)`
 * (rl_config.yaml:18-57, ultrasound.py:99-133) that affect the hot path. */
typedef struct usim_config {
  int32_t abi_version;
  int32_t num_envs;
  int32_t env_id_offset; /* global id of local env 0 (multi-GPU sharding) */
  int32_t impedance_mode;
  int32_t horizon;
  int32_t early_termination;
  int32_t solref_randomization;
  int32_t probe_pos_randomization;
  int32_t deterministic_trajectory;
  int32_t uncouple_pos_ori;
  int32_t solver_iterations; /* CG iteration cap per step (device) */
  int32_t precond_rebuilds;   /* preconditioner rebuilds allowed per solve when contact zones change (0: default 8) */
  int32_t ignore_done;        /* robosuite `ignore_done`: the horizon does not end the episode (early termination still does) */
  int32_t reserved0;
  uint64_t seed;
  double control_freq;
  double kp[6], damping_ratio[6];      /* fixed mode (rl_config.yaml:39-40) */
  double input_max, input_min;         /* rl_config.yaml:35-36 */
  double output_max[6], output_min[6]; /* rl_config.yaml:37-38 */
  double kp_limits[2], kp_input_max, kp_input_min; /* rl_config.yaml:42-44 */
  double solver_tolerance;
  double reset_eef_bias[3]; /* systematic IK offset seen in the shipped artifacts (SURVEY App. A.6) */
} usim_config;

typedef struct usim_handle usim_handle;

/* Build the batched env on CUDA device `device`: allocate per-env state in HBM
 * and upload the model tables.  Replaces `suite.make("Ultrasound", **opts)`
 * (rl.py:38) -> `Ultrasound.__init__` / `_load_model` (ultrasound.py:99-321). */
int usim_create(const usim_model* model, const usim_config* cfg, int device, usim_handle** out);
int usim_destroy(usim_handle* h);

/* Reset the envs whose mask byte is non-zero (mask_dev == NULL: all).  Draws
 * stiffness/damping, waypoints, u0 and probe noise from per-env Philox
 * streams keyed by (seed, global env id, episode), solves the initial arm
 * pose by damped-least-squares IK, runs one forward pass and writes the
 * observation.  Replaces `MujocoEnv.reset()` -> `Ultrasound._reset_internal`
 * (ultrasound.py:416-477) incl. `_get_initial_qpos` (:812-844).
 * obs_dev: [num_envs][19] float, may be NULL. */
int usim_reset(usim_handle* h, const uint8_t* mask_dev, float* obs_dev, void* stream);

/* One control step for every env.  Replaces `MujocoEnv.step(action)` [robosuite]
 * = int(control_timestep / timestep) physics substeps of
 *   { sim.forward(); Robot.control (OSC_POSE; the goal is set on the first
 *     substep only); sim.step() }   (1 substep at rl_config.yaml's 500 Hz, 25 at
 *   the env default of 20 Hz, ultrasound.py:119); then
 * `Ultrasound._post_action` (ultrasound.py:512-550), `reward` (:230-269),
 * `_check_terminated` (:635-670) and the observables (:363-401).
 * The observation is the one robosuite returns: sampled after the last
 * sim.step() and BEFORE _post_action updates the task state, so obs[9..14]
 * (force / velocity statistics, trajectory point) are those reward() used.
 *   act_dev   [num_envs][action_dim] float
 *   obs_dev   [num_envs][19] float        rew_dev [num_envs] float
 *   done_dev  [num_envs] uint8
 *   auto_reset != 0: envs that finished are reset in the same call (SB3 VecEnv
 *   semantics); obs_dev then holds the post-reset observation and
 *   term_obs_dev [num_envs][19] (may be NULL) the terminal one. */
int usim_step(usim_handle* h, const float* act_dev, float* obs_dev, float* rew_dev,
              uint8_t* done_dev, float* term_obs_dev, int auto_reset, void* stream);

/* Forward pass without stepping: MuJoCo's mj_forward at each selected env's
 * live (qpos, qvel).  Replaces `sim.forward()` (ultrasound.py:431, and
 * robosuite's `set_robot_joint_positions` after it writes qpos).
 *   mask_dev  [num_envs] uint8, envs to evaluate (NULL: all)
 *   ctrl_dev  [num_envs][7] float joint torques, clipped to ctrl_range as MuJoCo
 *             clips a limited ctrl (NULL: zero, `data.ctrl` after mj_resetData;
 *             UR5e: the seventh column is ignored)
 *   obs_dev   [num_envs][19] float (may be NULL): the observation robosuite's
 *             _get_observations(force_update=True) gives after sim.forward():
 *             channels 0-8 and 12-18 from this pass (current kinematics, not
 *             the site pose a step's observation carries), 9-11 from the task
 *             record as it stands
 *   qacc_dev  [num_envs][nv] float (may be NULL): the solved accelerations
 * The constraint solve is warm-started from the env's qacc_warmstart row, with
 * the reset forward pass's iteration cap (2 x solver_iterations) and the
 * configured tolerance.  For the selected envs it refreshes usim_get_diag
 * (torques = the clipped ctrl), usim_get_contacts and the contact record; every
 * row of the other envs is left as it was.  It leaves the state (qpos, qvel,
 * warm start, task record), the arm record (whose qfrc_smooth feeds the next
 * step's warm-start shift: usim_get_arm_record keeps describing the last step
 * or reset), the prepared reset states, the divergence / overflow counters and
 * the done flags bit for bit as they were, so that the steps that follow run
 * exactly as without the call.  Terminated envs are evaluated too and stay
 * done.  A diverged pass reports zero forces and a finite observation, as a
 * step does, and counts nothing.  Fails before the first usim_reset. */
int usim_forward(usim_handle* h, const uint8_t* mask_dev, const float* ctrl_dev, float* obs_dev, float* qacc_dev, void* stream);

/* Convenience for host callers (the end-to-end path of bench.py and of the
 * single-env robosuite-style API): HOST buffers; the H2D/D2H copies are done
 * inside the call, which synchronises the library's stream.  A buffer that is
 * page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) is the
 * transfer end point itself; a pageable one is staged through the library's
 * pinned memory (one extra host memcpy).  Actions travel by cudaMemcpyAsync;
 * observation, reward, done and terminal-observation rows are written by the
 * step kernel straight into the page-locked result buffers (mapped host
 * memory, one coalesced 76-byte row per env: posted PCIe writes that overlap
 * the launch), so no device->host copy follows the kernel.  tobs_host rows are
 * written only for the envs whose done flag is set in this step; the other rows
 * are left untouched. */
int usim_step_host(usim_handle* h, const float* act_host, float* obs_host, float* rew_host,
                   uint8_t* done_host, float* term_obs_host, int auto_reset);

/* State access, parity hooks.  Replace `sim.data.qpos/qvel/qacc_warmstart`
 * views and `sim.data.set_joint_qpos` (ultrasound.py:430).  Layout
 * [num_envs][nq|nv|USIM_TASK_DIM] float, device memory.
 * usim_set_state with a task record, once usim_reset has run, also prepares
 * again (on `stream`, the next call on it waits for this) the reset states the
 * next two auto-resets of every env take over: episodes E and E + 1, E being
 * the restored USIM_TS_EPISODE.  So an auto-reset after a restore draws what the
 * (seed, global env id, episode) streams give for the restored counter, as
 * usim_reset does.  The arm record is not part of the state, and the solver's
 * warm start is shifted by the change of the arm's qfrc_smooth since the
 * previous step, which it holds: until its next reset a restored env agrees
 * with the run it was saved from to solver tolerance, from then on bit for bit
 * (a reset state starts from a zero warm start, without shift). */
int usim_get_state(usim_handle* h, float* qpos_dev, float* qvel_dev, float* warm_dev, float* task_dev, void* stream);
int usim_set_state(usim_handle* h, const float* qpos_dev, const float* qvel_dev, const float* warm_dev,
                   const float* task_dev, void* stream);

/* Contact list of the last forward pass, in MuJoCo order (body pair, then
 * geom).  Replaces `sim.data.contact[:ncon].geom1/geom2` + `sim.data.ncon`
 * (ultrasound.py:691-693).  geom ids: 0 floor, 1 table_collision,
 * 2 probe_collision, 3 torso centre, 4+k particle k.
 * ncon_dev [num_envs] int32; geom1/geom2_dev [num_envs][USIM_MAX_CONTACTS] int32;
 * dist_dev same shape float (may be NULL). */
int usim_get_contacts(usim_handle* h, int32_t* ncon_dev, int32_t* geom1_dev, int32_t* geom2_dev,
                      float* dist_dev, void* stream);

/* Contact record, opt-in.  enable != 0 turns it on for the launches issued after
 * this call (the record is allocated on the first enable: USIM_MAX_CONTACTS * 36
 * bytes per env); with it off every launch runs exactly as without it. */
int usim_set_contact_record(usim_handle* h, int enable);

/* Position, frame and constraint force of every contact of the last forward
 * pass -- the same pass usim_get_contacts and usim_get_diag describe, contact c
 * being row c of their list.  Replaces `sim.data.contact[:ncon].pos / .frame`
 * and `mujoco_py.functions.mj_contactForce(model, data, c, f)` (its first three
 * components: condim 3).  Device memory:
 *   pos_dev   [num_envs][USIM_MAX_CONTACTS][3] float, world contact point
 *   frame_dev [num_envs][USIM_MAX_CONTACTS][9] float, rows: the normal (geom1 ->
 *             geom2), then two tangents (MuJoCo's rule)
 *   force_dev [num_envs][USIM_MAX_CONTACTS][3] float, (normal, tangent 1,
 *             tangent 2) force on geom2 in that frame; frame^T force is the
 *             world force, and the forces on the probe add up to diag[0..2]
 * Rows at or beyond ncon are zero; any pointer may be NULL.  Fails unless
 * recording is on and every env has been stepped (or reset without mask) since
 * it was last enabled.  A diverged env reports zero forces. */
int usim_get_contact_forces(usim_handle* h, float* pos_dev, float* frame_dev, float* force_dev, void* stream);

/* Per-env diagnostics of the last forward pass (step, reset or usim_forward), [num_envs][USIM_DIAG_DIM] float:
 * 0-2 cfrc_ext[probe][-3:] (ultrasound.py:365), 3-5 ee torque (:369),
 * 6-8 eef pos, 9-12 eef quat xyzw, 13-19 joint torques, 20 solver iterations,
 * 21 solver gradient norm, 22 ncon (uncapped), 23 nefc, 24 preconditioner rebuilds, 25 line-search evaluations,
 * 26-27 spare */
#define USIM_DIAG_DIM 28
int usim_get_diag(usim_handle* h, float* diag_dev, void* stream);

/* Arm record of the last physics step, [num_envs][USIM_ARM_RECORD_DIM] float: what robosuite's controller reads through
 * mujoco-py every substep (osc.py update(): `sim.data.qM` / `cymj._mj_fullM`, `get_site_jacp/jacr`, site pose) plus the
 * controller output.  0-48 joint-space inertia M (7x7 row major), 49-55 qfrc_smooth of the arm, 56-62 clipped joint torques,
 * 63-104 grip-site Jacobian (rows 0-2 linear, 3-5 angular; 6x7), 105-125 hand-body linear Jacobian (3x7), 126-128 site position,
 * 129-137 site orientation (row major), 138-143 probe capsule end points, 144-146 / 147-167 F/T torque sensor: bias part and
 * linear map from the arm accelerations (3x7), 168-171 eef quaternion xyzw, 172-178 warm-start shift of the solver.
 * usim_forward does not write it: it keeps describing the last step or reset. */
#define USIM_ARM_RECORD_DIM 180
int usim_get_arm_record(usim_handle* h, float* rec_dev, void* stream);

/* Sizes the caller needs to allocate buffers. */
int usim_num_envs(const usim_handle* h);
int usim_nq(const usim_handle* h);
int usim_nv(const usim_handle* h);
int usim_action_dim(const usim_handle* h);
/* number of kernels launched by this handle so far (bench.py "gpu_launches") */
int64_t usim_launch_count(const usim_handle* h);
/* number of env steps whose constraint solve produced a non-finite result; such an env reports done = 1 with finite outputs
 * and is wiped by the next reset (MuJoCo: "bad qacc" auto-reset).  Synchronises the device. */
int usim_divergence_count(usim_handle* h, int64_t* count);
/* number of env steps (physics substeps) in which more than USIM_MAX_CONTACTS contacts were found and the surplus was
 * dropped (diag[22] holds the uncapped count of the last step).  Synchronises the device. */
int usim_contact_overflow_count(usim_handle* h, int64_t* count);
/* physics substeps per control step = int((1 / control_freq) / timestep) */
int usim_substeps(const usim_handle* h);
/* Kernel timing is opt-in (off by default: no event traffic in the hot path).  When enabled every launch of the dominant
 * kernel in usim_step is bracketed by CUDA events on the launch stream (at most 4096 pending pairs are kept). */
int usim_set_timing(usim_handle* h, int enable);
/* elapsed device time (ms) of the dominant kernel over its timed launches since the
 * last call with reset != 0 */
int usim_kernel_time(usim_handle* h, int reset, double* total_ms, int64_t* launches);

const char* usim_last_error(void);
int usim_abi_version(void);
/* sizeof(usim_model) / sizeof(usim_config) as compiled, so that bindings can validate their struct mirrors */
size_t usim_sizeof_model(void);
size_t usim_sizeof_config(void);

#ifdef __cplusplus
}
#endif
#endif /* USIM_H_ */
