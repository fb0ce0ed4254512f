// arm.cuh — K1/K2: Panda forward kinematics, site Jacobians, CRBA, RNE bias and the
// OSC_POSE torque law, one THREAD per env (7-DoF chain, everything in registers /
// local arrays).  Also the per-episode reset kernel (Philox draws + DLS inverse
// kinematics).  Replaces mj_kinematics/mj_crb/mj_rne for the arm, get_site_jacp/jacr,
// cymj._mj_fullM and robosuite's osc.py / control_utils.py (SURVEY §2.4 K1, K2).
#pragma once
#include "common.cuh"

// NJ = number of real arm joints: 7 (Panda) or 6 (UR5e).  Every per-env array keeps 7 slots; with NJ = 6 the seventh is an inert,
// decoupled degree of freedom (unit inertia, no Jacobian column, no torque), so the solve kernel and the state layout do not change.
// The per-link loops of the arm kernel can be ROLLED (ARM_ROLL=1): the kernel runs one thread per env, one warp per SM, and is
// bound by instruction fetch (fully unrolled: ~5 500 straight-line instructions executed once at ~8 cycles each); rolled, the loop bodies
// are fetched once and reused, at the price of link arrays in local memory (L1 resident).
#ifndef ARM_ROLL
#define ARM_ROLL 0 // measured at 4096 envs: rolled 3184 instead of ~5500 SASS instructions, arm launch 2 us shorter (29.4 vs 31.5 us step minus solve kernel), the step as a whole unchanged (0.528 ms): not kept
#endif
#if ARM_ROLL
#define ARM_LOOP _Pragma("unroll 1")
#else
#define ARM_LOOP _Pragma("unroll")
#endif
struct ArmKin {
  float R[7][9];  // link frames
  v3 p[7];        // link origins == joint anchors
  v3 z[7];        // joint axes (world)
  v3 site, hand;  // grip_site (== ft_frame == probe body origin), right_hand origin
  float Rs[9];    // site orientation
};

template <int NJ>
__device__ __forceinline__ void arm_fk(const float* q, ArmKin& k) {
  float Rp[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  v3 pp = mk(0, 0, 0);
ARM_LOOP
  for (int j = 0; j < NJ; j++) {
    k.p[j] = pp + mv(Rp, ld3(dm.link_pos[j]));
    float T[9], Rz[9];
    mm3(Rp, dm.link_R[j], T);
    float s, c;
    sincosf(q[j], &s, &c);
    Rz[0] = c; Rz[1] = -s; Rz[2] = 0; Rz[3] = s; Rz[4] = c; Rz[5] = 0; Rz[6] = 0; Rz[7] = 0; Rz[8] = 1;
    mm3(T, Rz, k.R[j]);
    k.z[j] = mk(k.R[j][2], k.R[j][5], k.R[j][8]);
#pragma unroll
    for (int i = 0; i < 9; i++) Rp[i] = k.R[j][i];
    pp = k.p[j];
  }
  k.site = k.p[NJ - 1] + mv(k.R[NJ - 1], ld3(dm.tool + 0));
  mm3(k.R[NJ - 1], dm.tool + 3, k.Rs);
  k.hand = k.p[NJ - 1] + mv(k.R[NJ - 1], ld3(dm.tool + 12));
}

// J[6][7]: rows 0-2 linear, 3-5 angular, of world point x on the last link (columns of absent joints are zero)
template <int NJ>
__device__ __forceinline__ void arm_jac(const ArmKin& k, v3 x, float* J) {
#pragma unroll
  for (int j = 0; j < 7; j++) {
    if (j < NJ) {
      v3 jp = cross(k.z[j], x - k.p[j]);
      J[0 * 7 + j] = jp.x; J[1 * 7 + j] = jp.y; J[2 * 7 + j] = jp.z;
      J[3 * 7 + j] = k.z[j].x; J[4 * 7 + j] = k.z[j].y; J[5 * 7 + j] = k.z[j].z;
    } else {
#pragma unroll
      for (int r = 0; r < 6; r++) J[r * 7 + j] = 0.f;
    }
  }
}

// world inertia R I R^T of a symmetric (xx,yy,zz,xy,xz,yz) local inertia
__device__ __forceinline__ void world_inertia(const float* R, const float* I6, float* W /*9*/) {
  float I[9] = {I6[0], I6[3], I6[4], I6[3], I6[1], I6[5], I6[4], I6[5], I6[2]}, T[9];
  mm3(R, I, T);
  float Rt[9] = {R[0], R[3], R[6], R[1], R[4], R[7], R[2], R[5], R[8]};
  mm3(T, Rt, W);
}

// OSC goal update on the policy step (robosuite osc.set_goal), writes the task record; site / Rs: current grip-site pose
__device__ __forceinline__ void osc_set_goal(const float* act, v3 site, const float* Rs, float* ts) {
  if (dm.mode == USIM_MODE_FIXED) {
    float d[6];
#pragma unroll
    for (int i = 0; i < 6; i++) d[i] = scale1(act[i], dm.in_min, dm.in_max, dm.out_min[i], dm.out_max[i]);
    ts[USIM_TS_GOAL_POS + 0] = site.x + d[0];
    ts[USIM_TS_GOAL_POS + 1] = site.y + d[1];
    ts[USIM_TS_GOAL_POS + 2] = site.z + d[2];
    if (d[3] != 0.f || d[4] != 0.f || d[5] != 0.f) {
      float ang = sqrtf(d[3] * d[3] + d[4] * d[4] + d[5] * d[5]);
      float s = sinf(0.5f * ang) / ang, q[4] = {cosf(0.5f * ang), s * d[3], s * d[4], s * d[5]}, Rd[9], G[9];
      quat2mat(q, Rd);
      mm3(Rd, Rs, G);
#pragma unroll
      for (int i = 0; i < 9; i++) ts[USIM_TS_GOAL_ORI + i] = G[i];
    }
  } else if (dm.mode != USIM_MODE_WRENCH) {
    ts[USIM_TS_GOAL_POS + 0] = ts[USIM_TS_TRAJ_PT + 0];
    ts[USIM_TS_GOAL_POS + 1] = ts[USIM_TS_TRAJ_PT + 1];
    ts[USIM_TS_GOAL_POS + 2] = ts[USIM_TS_TRAJ_PT + 2] + (dm.mode == USIM_MODE_VARIABLE_Z ? scale1(act[6], -1.f, 1.f, -0.05f, 0.05f) : 0.f);
    float G[9];
    goal_mat(G);
#pragma unroll
    for (int i = 0; i < 9; i++) ts[USIM_TS_GOAL_ORI + i] = G[i];
  }
}

// mode 0: env step (OSC torques from the action); mode 1: forward pass without a controller (after a reset, or usim_forward):
// torques = the row `act` clipped to ctrl_range (nullptr: ctrl = 0), no warm-start shift
// (q, qd: the arm joint positions / velocities of this env, in registers: the caller may have just written them to HBM itself)
// policy_step: first physics substep of a control step -- the only one on which the OSC goal is set (robosuite Robot.control)
// ts / ab: the env's task record and arm record; act: the env's action row (mode 0) or joint torque row [7] (mode 1)
template <int NJ>
__device__ __forceinline__ void arm_forward(int mode, bool policy_step, const float (&q)[7], const float (&qd)[7],
                                            const float* __restrict__ act, float* __restrict__ ts, float* __restrict__ ab) {
  if (mode == 0 && ts[USIM_TS_DONE] != 0.f) return; // terminated env: frozen until reset

  ArmKin k;
  arm_fk<NJ>(q, k);

  // ---------------- velocities, velocity-product accelerations (gravity folded in: a_base = -g), world frame
  v3 w[7], al[7], ac[7]; // angular vel, angular acc (vp), linear acc of the link origin (vp, with -g)
  {
    v3 wp = mk(0, 0, 0), alp = mk(0, 0, 0), acp = mk(-dm.g[0], -dm.g[1], -dm.g[2]), pp = mk(0, 0, 0);
ARM_LOOP
    for (int j = 0; j < NJ; j++) {
      v3 r = k.p[j] - pp;
      v3 zq = qd[j] * k.z[j];
      ac[j] = acp + cross(alp, r) + cross(wp, cross(wp, r));
      w[j] = wp + zq;
      al[j] = alp + cross(wp, zq);
      wp = w[j]; alp = al[j]; acp = ac[j]; pp = k.p[j];
    }
  }
  // ---------------- RNE backward pass -> bias; CRBA composites -> M
  float bias[7], M[49];
#pragma unroll
  for (int i = 0; i < 49; i++) M[i] = (i % 8 == 0) ? 1.f : 0.f; // identity in the slots of absent joints
#pragma unroll
  for (int j = 0; j < 7; j++) bias[j] = 0.f;
  {
    v3 F = mk(0, 0, 0), N = mk(0, 0, 0); // accumulated force / moment about p[j+1]
    v3 pn = k.p[NJ - 1];
    float cm = 0.f; v3 cc = mk(0, 0, 0); float Ic[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; // composite mass, com, inertia about com
ARM_LOOP
    for (int j = NJ - 1; j >= 0; j--) {
      v3 cl = mv(k.R[j], ld3(dm.link_com[j]));
      v3 com = k.p[j] + cl;
      float Iw[9];
      world_inertia(k.R[j], dm.link_I[j], Iw);
      float m = dm.link_mass[j];
      v3 acom = ac[j] + cross(al[j], cl) + cross(w[j], cross(w[j], cl));
      v3 f = m * acom;
      v3 nn = mv(Iw, al[j]) + cross(w[j], mv(Iw, w[j]));
      // moment about p[j]: own + child's moved from p[j+1]
      N = nn + cross(cl, f) + N + cross(pn - k.p[j], F);
      F = F + f;
      bias[j] = dot(k.z[j], N);
      pn = k.p[j];
      // composite inertia: merge (m, com, Iw) into (cm, cc, Ic)
      float mt = cm + m;
      v3 cn = (1.f / mt) * (cm * cc + m * com);
      v3 d1 = cc - cn, d2 = com - cn;
      float a1 = cm * dot(d1, d1), a2 = m * dot(d2, d2);
      float dv1[3] = {d1.x, d1.y, d1.z}, dv2[3] = {d2.x, d2.y, d2.z};
#pragma unroll
      for (int a = 0; a < 3; a++)
#pragma unroll
        for (int b = 0; b < 3; b++)
          Ic[3 * a + b] = Ic[3 * a + b] + Iw[3 * a + b] + (a == b ? a1 + a2 : 0.f) - cm * dv1[a] * dv1[b] - m * dv2[a] * dv2[b];
      cm = mt; cc = cn;
      // column j of M: unit acceleration of joint j moves composite j
      v3 lin = cross(k.z[j], cc - k.p[j]);
      v3 fj = cm * lin;
      v3 nj = mv(Ic, k.z[j]);
#pragma unroll
      for (int i = 0; i <= j; i++) {
        float v = dot(k.z[i], nj + cross(cc - k.p[i], fj));
        M[i * 7 + j] = v;
        M[j * 7 + i] = v;
      }
    }
  }
  // ---------------- Jacobians
  float J[42], Jh[42];
  arm_jac<NJ>(k, k.site, J);
  arm_jac<NJ>(k, k.hand, Jh);

  // ---------------- OSC_POSE torques [SURVEY App. C.2/C.3]
  float tau[7], dx[7];
#pragma unroll
  for (int j = 0; j < 7; j++) dx[j] = 0.f;
  if (mode == 1) {
#pragma unroll
    for (int j = 0; j < 7; j++) tau[j] = act && j < NJ ? fminf(fmaxf(act[j], -dm.ctrl[j]), dm.ctrl[j]) : 0.f; // (UR5e: slot 6 is inert)
  } else {
    float av[7];
    for (int i = 0; i < dm.adim; i++) av[i] = act[i];
    if (policy_step) osc_set_goal(av, k.site, k.Rs, ts);
    float kp[6], kd[6];
#pragma unroll
    for (int i = 0; i < 6; i++) {
      if (dm.mode == USIM_MODE_FIXED) { kp[i] = dm.kp[i]; kd[i] = 2.f * sqrtf(kp[i]) * dm.dr[i]; }
      else { kp[i] = scale1(av[i], dm.kp_in_min, dm.kp_in_max, dm.kp_lim[0], dm.kp_lim[1]); kd[i] = 2.f * sqrtf(kp[i]); }
    }
    float vel[6];
#pragma unroll
    for (int r = 0; r < 6; r++) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 7; j++) s += J[r * 7 + j] * qd[j];
      vel[r] = s;
    }
    float Fd[6];
    if (dm.mode == USIM_MODE_WRENCH) {
#pragma unroll
      for (int i = 0; i < 6; i++) Fd[i] = fminf(fmaxf(av[i], -10.f), 10.f);
    } else {
      v3 eo = ori_error(ts + USIM_TS_GOAL_ORI, k.Rs);
      Fd[0] = kp[0] * (ts[USIM_TS_GOAL_POS + 0] - k.site.x) - kd[0] * vel[0];
      Fd[1] = kp[1] * (ts[USIM_TS_GOAL_POS + 1] - k.site.y) - kd[1] * vel[1];
      Fd[2] = kp[2] * (ts[USIM_TS_GOAL_POS + 2] - k.site.z) - kd[2] * vel[2];
      Fd[3] = kp[3] * eo.x - kd[3] * vel[3];
      Fd[4] = kp[4] * eo.y - kd[4] * vel[4];
      Fd[5] = kp[5] * eo.z - kd[5] * vel[5];
    }
    // M^-1 J^T through one Cholesky of M (7 solves with 6 right-hand sides)
    float L[49];
#pragma unroll
    for (int i = 0; i < 49; i++) L[i] = M[i];
    chol<7>(L);
    float MiJt[42]; // [7][6]
ARM_LOOP
    for (int r = 0; r < 6; r++) {
      float col[7];
#pragma unroll
      for (int j = 0; j < 7; j++) col[j] = J[r * 7 + j];
      chol_solve<7>(L, col);
#pragma unroll
      for (int j = 0; j < 7; j++) MiJt[j * 6 + r] = col[j];
    }
    float Lf[36]; // J M^-1 J^T
#pragma unroll
    for (int r = 0; r < 6; r++)
#pragma unroll
      for (int s2 = 0; s2 < 6; s2++) {
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 7; j++) s += J[r * 7 + j] * MiJt[j * 6 + s2];
        Lf[r * 6 + s2] = s;
      }
    float W[6];
    if (dm.mode == USIM_MODE_WRENCH) {
#pragma unroll
      for (int i = 0; i < 6; i++) W[i] = Fd[i];
    } else if (dm.uncouple) {
      float Lp[9], Lo[9];
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int s2 = 0; s2 < 3; s2++) { Lp[r * 3 + s2] = Lf[r * 6 + s2]; Lo[r * 3 + s2] = Lf[(3 + r) * 6 + 3 + s2]; }
      chol<3>(Lp); chol<3>(Lo);
      float a3[3] = {Fd[0], Fd[1], Fd[2]}, b3[3] = {Fd[3], Fd[4], Fd[5]};
      chol_solve<3>(Lp, a3); chol_solve<3>(Lo, b3);
      W[0] = a3[0]; W[1] = a3[1]; W[2] = a3[2]; W[3] = b3[0]; W[4] = b3[1]; W[5] = b3[2];
    }
    float Lfc[36];
#pragma unroll
    for (int i = 0; i < 36; i++) Lfc[i] = Lf[i];
    chol<6>(Lfc);
    if (dm.mode != USIM_MODE_WRENCH && !dm.uncouple) {
#pragma unroll
      for (int i = 0; i < 6; i++) W[i] = Fd[i];
      chol_solve<6>(Lfc, W);
    }
    // null-space term: N^T M pose, N = I - Jbar J, Jbar = M^-1 J^T Lambda_full
    float pose[7], Mp[7];
#pragma unroll
    for (int j = 0; j < 7; j++) pose[j] = 10.f * (ts[USIM_TS_INIT_JOINT + j] - q[j]) - 6.3245553203f * qd[j];
#pragma unroll
    for (int i = 0; i < 7; i++) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 7; j++) s += M[i * 7 + j] * pose[j];
      Mp[i] = s;
    }
    // N^T Mp = Mp - J^T Lambda (J M^-1 Mp) ... with Jbar^T Mp = Lambda J M^-1 Mp = Lambda (MiJt^T Mp)
    float t6[6];
#pragma unroll
    for (int r = 0; r < 6; r++) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 7; j++) s += MiJt[j * 6 + r] * Mp[j];
      t6[r] = s;
    }
    chol_solve<6>(Lfc, t6);
#pragma unroll
    for (int j = 0; j < 7; j++) {
      float s = bias[j] + Mp[j];
#pragma unroll
      for (int r = 0; r < 6; r++) s += J[r * 7 + j] * (W[r] - t6[r]);
      tau[j] = fminf(fmaxf(s, -dm.ctrl[j]), dm.ctrl[j]);
    }
    // warm-start shift for the solve kernel: M^-1 (qfrc_smooth - qfrc_smooth of the previous physics step).  The arm record still
    // holds the previous step's values here; on the first step of an episode it is stale (the warm start is zero then anyway).
    if (!(policy_step && ts[USIM_TS_TIMESTEP] == 0.f)) {
#pragma unroll
      for (int j = 0; j < 7; j++) dx[j] = tau[j] - bias[j] - dm.arm_damp * qd[j] - ab[AB_QS + j];
      chol_solve<7>(L, dx);
    }
  }

  // ---------------- F/T sensor pieces for the probe body (welded to link 7)
  float tau0[3], Jft[21];
  {
    float Iw[9];
    constexpr int LL = NJ - 1; // the link the hand and the probe are welded to
    world_inertia(k.R[LL], dm.tool + 26, Iw);
    float mp = dm.tool[22];
    v3 cl = mv(k.R[LL], ld3(dm.tool + 23)); // probe COM relative to p[LL]
    v3 rc = k.p[LL] + cl - k.site;          // COM relative to the site
    v3 acom = ac[LL] + cross(al[LL], cl) + cross(w[LL], cross(w[LL], cl));
    v3 t0 = mv(Iw, al[LL]) + cross(w[LL], mv(Iw, w[LL])) + cross(rc, mp * acom);
    tau0[0] = t0.x; tau0[1] = t0.y; tau0[2] = t0.z;
ARM_LOOP
    for (int j = 0; j < 7; j++) {
      if (j < NJ) {
        v3 jr = k.z[j];
        v3 jp = mk(J[0 * 7 + j], J[1 * 7 + j], J[2 * 7 + j]) + cross(jr, rc); // COM Jacobian column
        v3 t = mv(Iw, jr) + cross(rc, mp * jp);
        Jft[0 * 7 + j] = t.x; Jft[1 * 7 + j] = t.y; Jft[2 * 7 + j] = t.z;
      } else {
        Jft[0 * 7 + j] = 0.f; Jft[1 * 7 + j] = 0.f; Jft[2 * 7 + j] = 0.f;
      }
    }
  }

  // ---------------- write the arm record
#pragma unroll
  for (int i = 0; i < 49; i++) ab[AB_M + i] = M[i];
#pragma unroll
  for (int j = 0; j < 7; j++) { ab[AB_QS + j] = tau[j] - bias[j] - dm.arm_damp * qd[j]; ab[AB_TAU + j] = tau[j]; }
#pragma unroll
  for (int i = 0; i < 42; i++) ab[AB_JSITE + i] = J[i];
#pragma unroll
  for (int i = 0; i < 21; i++) { ab[AB_JHAND + i] = Jh[i]; ab[AB_JFT + i] = Jft[i]; }
  st3(ab + AB_EEFPOS, k.site);
#pragma unroll
  for (int i = 0; i < 9; i++) ab[AB_EEFR + i] = k.Rs[i];
  st3(ab + AB_PTIP, k.p[NJ - 1] + mv(k.R[NJ - 1], ld3(dm.tool + 15)));
  st3(ab + AB_PBACK, k.p[NJ - 1] + mv(k.R[NJ - 1], ld3(dm.tool + 18)));
  ab[AB_TAU0] = tau0[0]; ab[AB_TAU0 + 1] = tau0[1]; ab[AB_TAU0 + 2] = tau0[2];
  float qx[4];
  mat2quat_xyzw(k.Rs, qx);
  ab[AB_QUAT] = qx[0]; ab[AB_QUAT + 1] = qx[1]; ab[AB_QUAT + 2] = qx[2]; ab[AB_QUAT + 3] = qx[3];
#pragma unroll
  for (int j = 0; j < 7; j++) ab[AB_DX + j] = dx[j];
}

// One thread per env.  Also clears `done` (frozen envs report done = 0; the solve kernel sets it for the envs it steps), and flattens
// the iteration-count bins the previous solve launch filled into the launch order of the next one (highest bin first; soft.cuh NBIN).
template <int NJ>
__global__ void __launch_bounds__(64) arm_kernel(int n, const float* __restrict__ qpos, const float* __restrict__ qvel,
                                                 const float* __restrict__ act, float* __restrict__ task, float* __restrict__ armbuf,
                                                 uint8_t* __restrict__ done, int policy_step, int nbin, const int* __restrict__ bin_cnt_prev,
                                                 const int* __restrict__ bin_items_prev, int* __restrict__ bin_cnt_next,
                                                 int* __restrict__ order, int* __restrict__ queue) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (queue && env == 0) *queue = 0; // work queue of the solve launch that follows
  if (env >= n) return;
  if (order) {
    int off = 0, b = nbin - 1;
    for (; b > 0; b--) {
      const int c = bin_cnt_prev[b];
      if (env < off + c) break;
      off += c;
    }
    order[env] = bin_items_prev[(size_t)b * n + min(env - off, n - 1)];
    for (int k = env; k < nbin; k += n) bin_cnt_next[k] = 0; // (n may be smaller than the number of bins)
  }
  if (done) done[env] = 0;
  float q[7], qd[7];
#pragma unroll
  for (int j = 0; j < 7; j++) { q[j] = qpos[(size_t)env * QPAD + j]; qd[j] = qvel[(size_t)env * QPAD + j]; }
  arm_forward<NJ>(0, policy_step != 0, q, qd, act + (size_t)env * dm.adim, task + (size_t)env * USIM_TASK_DIM, armbuf + (size_t)env * ARMBUF);
}

// Arm part of usim_forward (mj_forward at the live state with the given joint torques), one thread per env: the arm record goes to
// `armbuf`, the handle's forward buffer, never to the live record (its qfrc_smooth feeds the next step's warm-start shift).  Reads
// qpos / qvel / task only.  ctrl: [n][7] joint torques, nullptr: zero; mask: envs to process (nullptr: all).
template <int NJ>
__global__ void __launch_bounds__(32) forward_arm_kernel(int n, const uint8_t* __restrict__ mask, const float* __restrict__ qpos,
                                                         const float* __restrict__ qvel, const float* __restrict__ ctrl,
                                                         float* __restrict__ task, float* __restrict__ armbuf) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n || (mask && !mask[env])) return;
  float q[7], qd[7];
#pragma unroll
  for (int j = 0; j < 7; j++) { q[j] = qpos[(size_t)env * QPAD + j]; qd[j] = qvel[(size_t)env * QPAD + j]; }
  arm_forward<NJ>(1, false, q, qd, ctrl ? ctrl + (size_t)env * 7 : nullptr, task + (size_t)env * USIM_TASK_DIM, armbuf + (size_t)env * ARMBUF);
}

// ---------------------------------------------------------------- reset (ultrasound.py:416-477, :749-887)
// One thread per env: Philox draws keyed by (seed, global env id, episode number), trajectory, DLS inverse kinematics for the
// initial joint pose, state initialisation, then the arm part of the post-reset forward pass (sim.forward() with ctrl = 0,
// ultrasound.py:431); the solve kernel (mode 1) that fills the contact-force statistics and the observation runs afterwards.
// The result depends on nothing but (seed, env id, episode number), so it can be made ahead of time:
//   live mode (items == nullptr): usim_reset -- the envs selected by `mask`, episode number from the live record, rows written to
//     the live state; files a request to prepare episode number + 2 into the slot this episode number belongs to.
//   prepare mode: works through the (env, episode number) requests of `items`; rows go to slot (episode number & 1) of the env
//     (qpos / task: [2][n][...]), the arm record to row `item` of `armbuf`.  A reset state is at rest: no qvel / warm rows.
template <int NJ>
__global__ void __launch_bounds__(32) reset_kernel(int n, const uint8_t* __restrict__ mask, float* __restrict__ qpos, float* __restrict__ qvel,
                                                   float* __restrict__ warm, float* __restrict__ task, float* __restrict__ armbuf,
                                                   const int* __restrict__ items, const int* __restrict__ nitems,
                                                   int* __restrict__ req_list, int* __restrict__ req_cnt) {
  const int total = items ? *nitems : n;
#pragma unroll 1
  for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < total; item += gridDim.x * blockDim.x) {
  int env = item;
  size_t row = item;
  unsigned ep;
  if (items) {
    env = items[2 * item];
    ep = (unsigned)items[2 * item + 1];
    row = (size_t)(ep & 1u) * n + env;
  } else {
    if (mask && !mask[env]) continue;
    ep = (unsigned)task[(size_t)env * USIM_TASK_DIM + USIM_TS_EPISODE];
    if (req_list) {
      const int p = atomicAdd(req_cnt, 1);
      req_list[2 * p] = env; req_list[2 * p + 1] = (int)ep + 2;
    }
  }
  float* ts = task + row * USIM_TASK_DIM;
  float* ab = armbuf + (size_t)item * ARMBUF;
  unsigned gid = (unsigned)(dm.env_off + env), r[4];
  float kst = -dm.solref_smooth[0], bst = -dm.solref_smooth[1];
  if (dm.solref_rand) { // ultrasound.py:291-297
    philox(dm.seed_lo, dm.seed_hi, gid, ep, 0, 0, r);
    kst = 1300.f + (float)(r[0] % 300u);
    bst = 17.f + (float)(r[1] % 24u);
  }
  for (int i = 0; i < USIM_TASK_DIM; i++) ts[i] = 0.f;
  ts[USIM_TS_EPISODE] = (float)(ep + 1);
  ts[USIM_TS_STIFFNESS] = kst; ts[USIM_TS_DAMPING] = bst;
  float* qp = qpos + row * QPAD;
  for (int i = 0; i < QPAD; i++) qp[i] = 0.f;
  if (qvel) {
    float* qv = qvel + row * QPAD;
    float* wm = warm + row * QPAD;
    for (int i = 0; i < QPAD; i++) { qv[i] = 0.f; wm[i] = 0.f; }
  }
  float tx = 0.f, ty = 0.f, tz = 0.8f + 0.005f + 0.0522f;
  if (dm.soft) {
    for (int i = 0; i < 7; i++) qp[7 + i] = dm.torso_qpos0[i];
    tx = dm.torso_qpos0[0]; ty = dm.torso_qpos0[1]; tz = dm.torso_qpos0[2];
  }
  if (dm.det_traj) { // ultrasound.py:762-764
    ts[0] = 0.062f; ts[1] = -0.020f; ts[2] = 0.896f; ts[3] = -0.032f; ts[4] = -0.075f; ts[5] = 0.896f;
  } else {          // :787-788, :805-807
    philox(dm.seed_lo, dm.seed_hi, gid, ep, 1, 0, r);
    float x0 = -dm.traj_xr + tx + 0.03f, x1 = dm.traj_xr + tx, y0 = -dm.traj_yr + ty, y1 = dm.traj_yr + ty;
    for (int wv = 0; wv < 2; wv++) {
      ts[3 * wv + 0] = x0 + (x1 - x0) * (float)(r[2 * wv] % 50u) / 49.f;
      ts[3 * wv + 1] = y0 + (y1 - y0) * (float)(r[2 * wv + 1] % 50u) / 49.f;
      ts[3 * wv + 2] = tz + dm.top_offset;
    }
  }
  philox(dm.seed_lo, dm.seed_hi, gid, ep, 2, 0, r);
  float u0 = ((float)r[0] + 0.5f) * (1.0f / 4294967296.0f);
  u0 = fminf(u0, 0.99999994f);
  ts[USIM_TS_U0] = u0;
  float uc = fminf(fmaxf(u0, 0.f), 1.f);
  v3 tp = mk(ts[0] + uc * (ts[3] - ts[0]), ts[1] + uc * (ts[4] - ts[1]), ts[2] + uc * (ts[5] - ts[2]));
  st3(ts + USIM_TS_TRAJ_PT, tp);
  float q[7];
#pragma unroll
  for (int j = 0; j < 7; j++) q[j] = dm.init_qpos[j];
  ArmKin k;
  if (dm.soft) {
    v3 target = tp;
    if (dm.pos_rand) { // :870-887
      unsigned r2[4];
      philox(dm.seed_lo, dm.seed_hi, gid, ep, 3, 0, r2);
      const float TWO_PI = 6.283185307179586f;
      float u1 = ((float)r[1] + 0.5f) * (1.0f / 4294967296.0f), u2 = ((float)r[2] + 0.5f) * (1.0f / 4294967296.0f);
      float u3 = ((float)r2[0] + 0.5f) * (1.0f / 4294967296.0f), u4 = ((float)r2[1] + 0.5f) * (1.0f / 4294967296.0f);
      u1 = fminf(u1, 0.99999994f); u3 = fminf(u3, 0.99999994f);
      float rad = sqrtf(-2.f * logf(u1));
      target.x += 0.0025f * rad * cosf(TWO_PI * u2);
      target.y += 0.0025f * rad * sinf(TWO_PI * u2);
      target.z += 0.010f * sqrtf(-2.f * logf(u3)) * cosf(TWO_PI * u4);
    }
    target = target + ld3(dm.eef_bias);
    float G[9];
    goal_mat(G);
    float en_prev = 1e30f;
#pragma unroll 1
    for (int it = 0; it < 60; it++) {
      arm_fk<NJ>(q, k);
      v3 ep3 = target - k.site, eo = ori_error(G, k.Rs);
      float err[6] = {ep3.x, ep3.y, ep3.z, eo.x, eo.y, eo.z};
      float en = sqrtf(dot(ep3, ep3) + dot(eo, eo));
      // converged, or stalled on the fp32 floor of the forward kinematics (~1e-6: the residual no longer halves)
      if (en < 2e-6f || (en < 1e-4f && en > 0.5f * en_prev)) break;
      en_prev = en;
      float J[42], A[36];
      arm_jac<NJ>(k, k.site, J);
#pragma unroll
      for (int a = 0; a < 6; a++)
#pragma unroll
        for (int b = 0; b < 6; b++) {
          float s = a == b ? 1e-4f : 0.f;
#pragma unroll
          for (int j = 0; j < 7; j++) s += J[a * 7 + j] * J[b * 7 + j];
          A[a * 6 + b] = s;
        }
      chol<6>(A);
      chol_solve<6>(A, err);
      float dq[7], mx = 0.f;
#pragma unroll
      for (int j = 0; j < 7; j++) {
        float s = 0.f;
#pragma unroll
        for (int a = 0; a < 6; a++) s += J[a * 7 + j] * err[a];
        dq[j] = s;
        mx = fmaxf(mx, fabsf(s));
      }
      float sc = mx > 0.5f ? 0.5f / mx : 1.f;
#pragma unroll
      for (int j = 0; j < 7; j++) q[j] += sc * dq[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 7; j++) { qp[j] = q[j]; ts[USIM_TS_INIT_JOINT + j] = q[j]; }
  arm_fk<NJ>(q, k);
  st3(ts + USIM_TS_GOAL_POS, k.site); // osc.reset_goal
#pragma unroll
  for (int i = 0; i < 9; i++) ts[USIM_TS_GOAL_ORI + i] = k.Rs[i];
  const float qd0[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  arm_forward<NJ>(1, false, q, qd0, nullptr, ts, ab);
  } // work items
}

// Fill both slots of EVERY env: request episode numbers E and E + 1, E = the counter of the env's live task record (the reset
// states its next two auto-resets take over).  Runs after the first reset of a handle (no slot prepared yet) and after
// usim_set_state (the restored counters need not be those the slots were prepared for).
__global__ void fill_requests_kernel(int n, const float* __restrict__ task, int* __restrict__ req_list, int* __restrict__ req_cnt) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  const int E = (int)task[(size_t)env * USIM_TASK_DIM + USIM_TS_EPISODE];
  const int p = atomicAdd(req_cnt, 2);
  req_list[2 * p] = env; req_list[2 * p + 1] = E;
  req_list[2 * p + 2] = env; req_list[2 * p + 3] = E + 1;
}
