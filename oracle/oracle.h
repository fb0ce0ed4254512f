/*
 * oracle.h — float64 CPU restatement of the Ultrasound env step.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path
 * (robotic-ultrasound-imaging_b200/, include/) may link, import or call this.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs use it, as the checker / the timed CPU baseline.
 *
 * PARITY UNPINNED at the physics boundary: the reference's arithmetic for this
 * path lives in un-vendored third-party code (MuJoCo 2.0 binary, closed
 * source; hermanjakobsen/mujoco-py and hermanjakobsen/robosuite at unpinned
 * git HEAD, requirements.txt:77-79) and the reference ships no tests.  The
 * oracle restates the published algorithms (SURVEY.md App. C) with a generic,
 * dense formulation (tree kinematics, Jacobian-sum inertia, world-frame
 * Newton-Euler, dense Newton solver) that shares no code or structure with the
 * CUDA kernels.  What IS pinned: the task layer (reward, bookkeeping,
 * termination, observation, trajectory, quaternion utilities) is checked
 * against golden vectors produced by executing the reference's own
 * ultrasound.py / utils/quaternion.py (tests/golden/make_golden.py).
 */
#ifndef ORACLE_H_
#define ORACLE_H_
#include "../include/usim.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct oracle_env oracle_env;

oracle_env* oracle_create(const usim_model* m, const usim_config* cfg, int global_env_id);
void oracle_destroy(oracle_env* e);

/* reset (ultrasound.py:416-477); writes obs[19] */
void oracle_reset(oracle_env* e, double* obs);
/* one env step (robosuite MujocoEnv.step + ultrasound.py:512-550); returns 0, or -1 if the env is done */
int oracle_step(oracle_env* e, const double* action, double* obs, double* reward, int* done);
/* number of redundant mj_forward passes per step the reference performs (3 = faithful cost; results identical) */
void oracle_set_forward_repeats(oracle_env* e, int n);

void oracle_get_state(const oracle_env* e, double* qpos, double* qvel, double* warm, double* task);
void oracle_set_state(oracle_env* e, const double* qpos, const double* qvel, const double* warm, const double* task);

/* forward pass at the current state with the given joint torques (no integration) */
void oracle_forward(oracle_env* e, const double* ctrl7);

/* The problem of the last oracle_forward evaluated at `qacc` (nv), the env left unchanged; any output may be NULL.
 * grad [nv] = M (qacc - a0) - J^T f, cost = the primal cost, efc_force [nefc] = f of every row, contact_force [3 ncon] as
 * oracle_contacts, cfrc [3] / ft_torque [3] as diag[0:6], norms [3] = |grad|, |rhs|, |Hx| of the device solver's stopping rule
 * (its quadratic part H is M plus the equality rows; rhs = qfrc_smooth + the equality
 * rows' J^T D aref, Hx = H qacc - rhs).  Returns nefc. */
int oracle_evaluate(oracle_env* e, const double* qacc, double* grad, double* cost, double* efc_force, double* contact_force,
                    double* cfrc, double* ft_torque, double* norms);
/* row type of every row of the last forward pass: 0 equality, 1 joint limit, 2 contact normal, 100 contact friction */
void oracle_efc_type(const oracle_env* e, int* type);

/* introspection of the last forward pass */
int oracle_ncon(const oracle_env* e);
void oracle_contacts(const oracle_env* e, int* geom1, int* geom2, double* dist, double* pos, double* frame, double* force);
int oracle_nefc(const oracle_env* e);
int oracle_solver_iter(const oracle_env* e);
const double* oracle_qacc(const oracle_env* e);
const double* oracle_qacc_smooth(const oracle_env* e);
const double* oracle_M(const oracle_env* e);    /* dense nv x nv */
const double* oracle_bias(const oracle_env* e); /* nv */
const double* oracle_tau(const oracle_env* e);  /* 7 */
/* diag[24], same layout as usim_get_diag */
void oracle_diag(const oracle_env* e, double* diag);
/* grip-site Jacobian 6x7 (rows: Jp then Jr), eef pos(3), eef mat(9) at the last kinematics */
void oracle_eef(const oracle_env* e, double* J6x7, double* pos, double* mat);
/* OSC torque for an action at the current state (runs kinematics) */
void oracle_controller(oracle_env* e, const double* action, double* tau7);
/* IK used by reset */
void oracle_ik(oracle_env* e, const double* target_pos, double* q7);

/* task-layer functions, pure (golden-vector checked) */
double oracle_distance_quat(const double* q1_wxyz, const double* q2_wxyz);
void oracle_difference_quat(const double* q1, const double* q2, double* out);
void oracle_mat2quat_xyzw(const double* mat9, double* q);
double oracle_reward(const double* eef_pos, const double* eef_quat_xyzw, const double* traj_pt, double vel_mean,
                     double fz_mean, double dfz, int in_contact, double* pos_err2, double* ori_err);
void oracle_post_action(double* ts, int horizon, double control_freq, int early_termination, const double* jnt_range,
                        const double* eef_pos, const double* eef_quat_xyzw, const double* hand_vel, double fz, int in_contact,
                        const double* qpos7, double* reward, int* done);
void oracle_grid_point(double tx, double ty, double tz, int ix, int iy, double* pt);
void oracle_philox(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t* out4);

/* batched rollouts for the CPU baseline: n envs, OpenMP over envs.
 * actions [steps][n][adim]; returns total env-steps executed */
long oracle_rollout(oracle_env** envs, int n, const double* actions, int steps, int adim, int auto_reset, int threads,
                    double* reward_sum);

/* one env step of n envs over host threads, per-env outputs: obs [n][19], rew [n], done [n], rc [n] (-1: env already done) */
void oracle_step_batch(oracle_env** envs, int n, const double* actions, int adim, int threads, double* obs, double* rew, int* done,
                       int* rc);

#ifdef __cplusplus
}
#endif
#endif
