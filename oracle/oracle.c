/*
 * oracle.c — float64 CPU restatement of one Ultrasound env step.
 * TEST INFRASTRUCTURE ONLY (see oracle.h).  PARITY UNPINNED at the physics
 * boundary; task layer pinned by tests/golden.
 *
 * Citations: "ultrasound.py" = src/my_environments/ultrasound.py and
 * "quaternion.py" = src/utils/quaternion.py of the reference; [C.x] =
 * SURVEY.md appendix C.x (recalled robosuite / MuJoCo 2.0 behaviour).
 */
#include "oracle.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>

#define MAXCH 16
#define MJMINVAL 1e-15
#define PI 3.14159265358979323846

enum { JN = 0, JH = 1, JS = 2, JF = 3 };
enum { ROW_EQ = 0, ROW_LIMIT = 1, ROW_CONTACT = 2 }; /* ROW_CONTACT marks the normal row; 2 friction rows follow */

typedef struct {
  int geom1, geom2, body1, body2;
  double pos[3], frame[9], dist, friction;
  int row; /* first efc row */
  double force[3];
  int probe_side; /* +1 probe is geom2, -1 probe is geom1, 0 not a probe contact */
  int torso;      /* other geom is a torso particle */
} ocontact;

struct oracle_env {
  const usim_model* m;
  usim_config cfg;
  int gid, nb, nq, nv, npart, adim, repeats;
  double *qpos, *qvel, *warm, ts[USIM_TASK_DIM];
  /* kinematics */
  double *xpos, *xmat, *xcom, *ximat;
  int *chn, *ch; /* chain length / dofs per body */
  double *dax, *danc;
  int *dtype, *dbody;
  double *bw, *bv, *balpha, *bacc;
  /* dynamics */
  double *M, *L, *bias, *passive, *act, *a0, *qacc, *qs, *fcon;
  /* constraint rows */
  int nefc, cap_rows, pool_n, cap_pool;
  int *rstart, *rn, *rtype, *pidx;
  double *pval, *rD, *raref, *rmu, *rfr, *jar, *frc, *jv;
  /* contacts */
  int ncon;
  ocontact con[USIM_MAX_CONTACTS];
  /* solver scratch */
  double *H, *grad, *dir, *Ma, *tmp;
  int solver_iter;
  double solver_grad;
  /* outputs */
  double tau[7], eef_pos[3], eef_mat[9], eef_quat[4], hand_vel[3], cfrc[3], ft_torque[3];
  double Jsite[42], Jhand[21];
  int in_contact;
  double goal_quat_xyzw[4];
};

/* ------------------------------------------------------------------ small math */
static inline double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static inline void cross3(const double* a, const double* b, double* c) {
  double x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  c[0] = x; c[1] = y; c[2] = z;
}
static inline double norm3(const double* a) { return sqrt(dot3(a, a)); }
static void quat2mat(const double* q, double* R) {
  double w = q[0], x = q[1], y = q[2], z = q[3];
  R[0] = 1 - 2 * (y * y + z * z); R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = 1 - 2 * (x * x + z * z); R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = 1 - 2 * (x * x + y * y);
}
static void quatmul(const double* a, const double* b, double* o) {
  double r[4];
  r[0] = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  r[1] = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  r[2] = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  r[3] = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  memcpy(o, r, sizeof r);
}
static void matmul3(const double* A, const double* B, double* C) {
  double r[9];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) r[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
  memcpy(C, r, sizeof r);
}
static void matvec3(const double* A, const double* v, double* o) {
  double r[3] = {A[0] * v[0] + A[1] * v[1] + A[2] * v[2], A[3] * v[0] + A[4] * v[1] + A[5] * v[2],
                 A[6] * v[0] + A[7] * v[1] + A[8] * v[2]};
  o[0] = r[0]; o[1] = r[1]; o[2] = r[2];
}
static void matTvec3(const double* A, const double* v, double* o) {
  double r[3] = {A[0] * v[0] + A[3] * v[1] + A[6] * v[2], A[1] * v[0] + A[4] * v[1] + A[7] * v[2],
                 A[2] * v[0] + A[5] * v[1] + A[8] * v[2]};
  o[0] = r[0]; o[1] = r[1]; o[2] = r[2];
}

/* dense Cholesky A = L L^T in place (lower), returns 0 on success */
static int chol(double* A, int n) {
  for (int j = 0; j < n; j++) {
    double s = A[j * n + j];
    for (int k = 0; k < j; k++) s -= A[j * n + k] * A[j * n + k];
    if (s <= 0) return -1;
    s = sqrt(s);
    A[j * n + j] = s;
    for (int i = j + 1; i < n; i++) {
      double t = A[i * n + j];
      const double *ri = A + i * n, *rj = A + j * n;
      for (int k = 0; k < j; k++) t -= ri[k] * rj[k];
      A[i * n + j] = t / s;
    }
  }
  return 0;
}
static void chol_solve(const double* L, int n, double* x) {
  for (int i = 0; i < n; i++) {
    double t = x[i];
    for (int k = 0; k < i; k++) t -= L[i * n + k] * x[k];
    x[i] = t / L[i * n + i];
  }
  for (int i = n - 1; i >= 0; i--) {
    double t = x[i];
    for (int k = i + 1; k < n; k++) t -= L[k * n + i] * x[k];
    x[i] = t / L[i * n + i];
  }
}

/* symmetric pseudo-inverse via cyclic Jacobi, numpy.linalg.pinv semantics
 * (rcond 1e-15 relative to the largest singular value) [C.2] */
static void sym_pinv(const double* A, int n, double* out) {
  double a[36], V[36];
  memcpy(a, A, sizeof(double) * n * n);
  for (int i = 0; i < n * n; i++) V[i] = 0;
  for (int i = 0; i < n; i++) V[i * n + i] = 1;
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0;
    for (int p = 0; p < n; p++)
      for (int q = p + 1; q < n; q++) off += a[p * n + q] * a[p * n + q];
    if (off < 1e-300) break;
    for (int p = 0; p < n; p++)
      for (int q = p + 1; q < n; q++) {
        double apq = a[p * n + q];
        if (fabs(apq) < 1e-300) continue;
        double th = (a[q * n + q] - a[p * n + p]) / (2 * apq);
        double t = (th >= 0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1));
        double c = 1 / sqrt(t * t + 1), s = t * c;
        for (int k = 0; k < n; k++) {
          double akp = a[k * n + p], akq = a[k * n + q];
          a[k * n + p] = c * akp - s * akq;
          a[k * n + q] = s * akp + c * akq;
        }
        for (int k = 0; k < n; k++) {
          double apk = a[p * n + k], aqk = a[q * n + k];
          a[p * n + k] = c * apk - s * aqk;
          a[q * n + k] = s * apk + c * aqk;
        }
        for (int k = 0; k < n; k++) {
          double vkp = V[k * n + p], vkq = V[k * n + q];
          V[k * n + p] = c * vkp - s * vkq;
          V[k * n + q] = s * vkp + c * vkq;
        }
      }
  }
  double mx = 0;
  for (int i = 0; i < n; i++) mx = fmax(mx, fabs(a[i * n + i]));
  for (int i = 0; i < n * n; i++) out[i] = 0;
  for (int k = 0; k < n; k++) {
    double ev = a[k * n + k];
    if (fabs(ev) <= 1e-15 * mx) continue;
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++) out[i * n + j] += V[i * n + k] * V[j * n + k] / ev;
  }
}

/* ------------------------------------------------------------------ Philox4x32-10 */
void oracle_philox(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t* out) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  uint32_t c[4] = {c0, c1, c2, c3};
  for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  memcpy(out, c, sizeof c);
}
static double u01(uint32_t r) { return ((double)r + 0.5) * (1.0 / 4294967296.0); }

/* ------------------------------------------------------------------ task-layer pure functions */
/* robosuite transform_utils.mat2quat: unit quaternion (x,y,z,w) with w >= 0 [C, A-QUAT-1] */
void oracle_mat2quat_xyzw(const double* m, double* q) {
  double tr = m[0] + m[4] + m[8], w, x, y, z;
  if (tr > 0) {
    double s = sqrt(tr + 1.0) * 2;
    w = 0.25 * s; x = (m[7] - m[5]) / s; y = (m[2] - m[6]) / s; z = (m[3] - m[1]) / s;
  } else if (m[0] > m[4] && m[0] > m[8]) {
    double s = sqrt(1.0 + m[0] - m[4] - m[8]) * 2;
    w = (m[7] - m[5]) / s; x = 0.25 * s; y = (m[1] + m[3]) / s; z = (m[2] + m[6]) / s;
  } else if (m[4] > m[8]) {
    double s = sqrt(1.0 + m[4] - m[0] - m[8]) * 2;
    w = (m[2] - m[6]) / s; x = (m[1] + m[3]) / s; y = 0.25 * s; z = (m[5] + m[7]) / s;
  } else {
    double s = sqrt(1.0 + m[8] - m[0] - m[4]) * 2;
    w = (m[3] - m[1]) / s; x = (m[2] + m[6]) / s; y = (m[5] + m[7]) / s; z = 0.25 * s;
  }
  if (w < 0) { w = -w; x = -x; y = -y; z = -z; }
  q[0] = x; q[1] = y; q[2] = z; q[3] = w;
}

/* quaternion.py:23-35: q1 * conj(q2), arrays treated as (w,x,y,z) */
void oracle_difference_quat(const double* q1, const double* q2, double* out) {
  double c[4] = {q2[0], -q2[1], -q2[2], -q2[3]};
  quatmul(q1, c, out);
}

/* quaternion.py:38-59 (with q_log :4-20) */
double oracle_distance_quat(const double* q1, const double* q2) {
  double m[4];
  oracle_difference_quat(q1, q2, m);
  double v = m[0] < -1 ? -1 : (m[0] > 1 ? 1 : m[0]);
  double un = sqrt(m[1] * m[1] + m[2] * m[2] + m[3] * m[3]);
  double lg[3] = {0, 0, 0};
  if (un != 0) {
    double a = acos(v);
    lg[0] = a * m[1] / un; lg[1] = a * m[2] / un; lg[2] = a * m[3] / un;
  }
  double dist = 2 * norm3(lg);
  if (dist > PI) dist = fabs(2 * PI - dist);
  return dist;
}

static const double GOAL_QUAT_XYZW[4] = {-0.69192486, 0.72186726, -0.00514253, -0.01100909}; /* ultrasound.py:174 */

/* ultrasound.py:230-269 */
double oracle_reward(const double* eef_pos, const double* eef_quat_xyzw, const double* traj_pt, double vel_mean,
                     double fz_mean, double dfz, int in_contact, double* pos_err2, double* ori_err) {
  double cur[4] = {eef_quat_xyzw[3], eef_quat_xyzw[0], eef_quat_xyzw[1], eef_quat_xyzw[2]};
  double des[4] = {GOAL_QUAT_XYZW[3], GOAL_QUAT_XYZW[0], GOAL_QUAT_XYZW[1], GOAL_QUAT_XYZW[2]};
  double e0 = 90 * (eef_pos[0] - traj_pt[0]), e1 = 90 * (eef_pos[1] - traj_pt[1]);
  pos_err2[0] = e0 * e0; pos_err2[1] = e1 * e1;
  double pos_reward = 5 * exp(-sqrt(pos_err2[0] * pos_err2[0] + pos_err2[1] * pos_err2[1]));
  *ori_err = 0.2 * oracle_distance_quat(cur, des);
  double ori_reward = 1 * exp(-*ori_err);
  double ve = 45 * (vel_mean - 0.04); ve = ve * ve;
  double vel_reward = 1 * exp(-fabs(ve));
  double fe = 0.7 * (fz_mean - 5); fe = fe * fe;
  double force_reward = in_contact ? 3 * exp(-fe) : 0;
  double de = 0.01 * (dfz - 0); de = de * de;
  double der_reward = in_contact ? 2 * exp(-de) : 0;
  return pos_reward + ori_reward + vel_reward + force_reward + der_reward;
}

/* ------------------------------------------------------------------ create / destroy */
static double* dalloc(size_t n) { return (double*)calloc(n ? n : 1, sizeof(double)); }
static int* ialloc(size_t n) { return (int*)calloc(n ? n : 1, sizeof(int)); }

oracle_env* oracle_create(const usim_model* m, const usim_config* cfg, int gid) {
  oracle_env* e = (oracle_env*)calloc(1, sizeof(oracle_env));
  e->m = m; e->cfg = *cfg; e->gid = gid;
  e->nb = m->nbody; e->nq = m->nq; e->nv = m->nv; e->npart = m->soft ? m->npart : 0;
  e->repeats = 1;
  e->adim = cfg->impedance_mode == USIM_MODE_VARIABLE_Z ? 7 : 6;
  int nb = e->nb, nv = e->nv, nq = e->nq;
  e->qpos = dalloc(nq); e->qvel = dalloc(nv); e->warm = dalloc(nv);
  e->xpos = dalloc(3 * nb); e->xmat = dalloc(9 * nb); e->xcom = dalloc(3 * nb); e->ximat = dalloc(9 * nb);
  e->chn = ialloc(nb); e->ch = ialloc(MAXCH * nb);
  e->dax = dalloc(3 * nv); e->danc = dalloc(3 * nv); e->dtype = ialloc(nv); e->dbody = ialloc(nv);
  e->bw = dalloc(3 * nb); e->bv = dalloc(3 * nb); e->balpha = dalloc(3 * nb); e->bacc = dalloc(3 * nb);
  e->M = dalloc((size_t)nv * nv); e->L = dalloc((size_t)nv * nv); e->H = dalloc((size_t)nv * nv);
  e->bias = dalloc(nv); e->passive = dalloc(nv); e->act = dalloc(nv); e->a0 = dalloc(nv); e->qacc = dalloc(nv);
  e->qs = dalloc(nv); e->fcon = dalloc(nv); e->grad = dalloc(nv); e->dir = dalloc(nv); e->Ma = dalloc(nv);
  e->tmp = dalloc(nv);
  e->cap_rows = 3 * USIM_MAX_CONTACTS + 2 * e->npart + m->npair + 32;
  e->cap_pool = e->cap_rows * 16 + e->npart + 64;
  e->rstart = ialloc(e->cap_rows); e->rn = ialloc(e->cap_rows); e->rtype = ialloc(e->cap_rows);
  e->pidx = ialloc(e->cap_pool); e->pval = dalloc(e->cap_pool);
  e->rD = dalloc(e->cap_rows); e->raref = dalloc(e->cap_rows); e->rmu = dalloc(e->cap_rows);
  e->rfr = dalloc(e->cap_rows); e->jar = dalloc(e->cap_rows); e->frc = dalloc(e->cap_rows); e->jv = dalloc(e->cap_rows);
  /* dof chains */
  for (int b = 1; b < nb; b++) {
    int par = m->body_parent[b], n = 0;
    if (par > 0) { n = e->chn[par]; memcpy(e->ch + MAXCH * b, e->ch + MAXCH * par, sizeof(int) * n); }
    int jt = m->body_jnt_type[b], d = m->body_dofadr[b];
    int nd = jt == JF ? 6 : (jt == JN ? 0 : 1);
    for (int k = 0; k < nd; k++) {
      e->ch[MAXCH * b + n++] = d + k;
      e->dbody[d + k] = b;
      e->dtype[d + k] = jt == JF ? (k < 3 ? 10 : 11) : jt; /* 10 free-trans, 11 free-rot */
    }
    e->chn[b] = n;
  }
  memcpy(e->qpos, m->qpos0, sizeof(double) * nq);
  memcpy(e->goal_quat_xyzw, GOAL_QUAT_XYZW, sizeof GOAL_QUAT_XYZW);
  e->ts[USIM_TS_STIFFNESS] = -m->solref_smooth[0];
  e->ts[USIM_TS_DAMPING] = -m->solref_smooth[1];
  e->ts[USIM_TS_DONE] = 1; /* must reset before stepping */
  return e;
}

void oracle_destroy(oracle_env* e) {
  if (!e) return;
  double* d[] = {e->qpos, e->qvel, e->warm, e->xpos, e->xmat, e->xcom, e->ximat, e->dax, e->danc, e->bw, e->bv,
                 e->balpha, e->bacc, e->M, e->L, e->H, e->bias, e->passive, e->act, e->a0, e->qacc, e->qs, e->fcon,
                 e->grad, e->dir, e->Ma, e->tmp, e->pval, e->rD, e->raref, e->rmu, e->rfr, e->jar, e->frc, e->jv};
  for (size_t i = 0; i < sizeof d / sizeof d[0]; i++) free(d[i]);
  int* ii[] = {e->chn, e->ch, e->dtype, e->dbody, e->rstart, e->rn, e->rtype, e->pidx};
  for (size_t i = 0; i < sizeof ii / sizeof ii[0]; i++) free(ii[i]);
  free(e);
}
void oracle_set_forward_repeats(oracle_env* e, int n) { e->repeats = n < 1 ? 1 : n; }

/* ------------------------------------------------------------------ kinematics (mj_kinematics, mj_comPos) */
static void kinematics(oracle_env* e) {
  const usim_model* m = e->m;
  double I3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  memcpy(e->xmat, I3, sizeof I3);
  for (int b = 1; b < e->nb; b++) {
    int par = m->body_parent[b], jt = m->body_jnt_type[b], qa = m->body_qposadr[b], d = m->body_dofadr[b];
    double* R = e->xmat + 9 * b;
    double* p = e->xpos + 3 * b;
    if (jt == JF) {
      double* q = e->qpos + qa + 3;
      double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
      for (int k = 0; k < 4; k++) q[k] /= n; /* mj_normalizeQuat */
      memcpy(p, e->qpos + qa, 3 * sizeof(double));
      quat2mat(q, R);
      for (int k = 0; k < 3; k++) {
        e->dax[3 * (d + k)] = k == 0; e->dax[3 * (d + k) + 1] = k == 1; e->dax[3 * (d + k) + 2] = k == 2;
        e->dax[3 * (d + 3 + k)] = R[k]; e->dax[3 * (d + 3 + k) + 1] = R[3 + k]; e->dax[3 * (d + 3 + k) + 2] = R[6 + k];
        memcpy(e->danc + 3 * (d + 3 + k), p, 3 * sizeof(double));
      }
    } else {
      double pos[3] = {m->body_pos[3 * b], m->body_pos[3 * b + 1], m->body_pos[3 * b + 2]};
      double Rl[9];
      quat2mat(m->body_quat + 4 * b, Rl);
      const double* ax = m->body_jnt_axis + 3 * b;
      if (jt == JS) {
        for (int k = 0; k < 3; k++) pos[k] += ax[k] * e->qpos[qa];
      } else if (jt == JH) {
        double a = e->qpos[qa], qj[4] = {cos(a / 2), sin(a / 2) * ax[0], sin(a / 2) * ax[1], sin(a / 2) * ax[2]}, Rj[9];
        quat2mat(qj, Rj);
        matmul3(Rl, Rj, Rl);
      }
      double wp[3];
      matvec3(e->xmat + 9 * par, pos, wp);
      for (int k = 0; k < 3; k++) p[k] = e->xpos[3 * par + k] + wp[k];
      matmul3(e->xmat + 9 * par, Rl, R);
      if (jt == JH || jt == JS) {
        matvec3(R, ax, e->dax + 3 * d);
        memcpy(e->danc + 3 * d, p, 3 * sizeof(double));
      }
    }
    double c[3];
    matvec3(R, m->body_ipos + 3 * b, c);
    for (int k = 0; k < 3; k++) e->xcom[3 * b + k] = p[k] + c[k];
    double T[9], Rt[9] = {R[0], R[3], R[6], R[1], R[4], R[7], R[2], R[5], R[8]};
    matmul3(R, m->body_inertia + 9 * b, T);
    matmul3(T, Rt, e->ximat + 9 * b);
  }
}

/* Jacobian columns of world point `pt` attached to body b, over the body's dof chain */
static int jac_point(const oracle_env* e, int b, const double* pt, double* Jp, double* Jr, const int** dofs) {
  int n = e->chn[b];
  const int* ch = e->ch + MAXCH * b;
  for (int i = 0; i < n; i++) {
    int d = ch[i], t = e->dtype[d];
    const double* ax = e->dax + 3 * d;
    double* jp = Jp + 3 * i;
    double* jr = Jr + 3 * i;
    if (t == JS || t == 10) {
      memcpy(jp, ax, 3 * sizeof(double));
      jr[0] = jr[1] = jr[2] = 0;
    } else {
      double r[3] = {pt[0] - e->danc[3 * d], pt[1] - e->danc[3 * d + 1], pt[2] - e->danc[3 * d + 2]};
      cross3(ax, r, jp);
      memcpy(jr, ax, 3 * sizeof(double));
    }
  }
  *dofs = ch;
  return n;
}

/* velocities and velocity-product accelerations, world frame (mj_comVel + the qacc=0 pass of mj_rne) */
static void velocities(oracle_env* e) {
  const usim_model* m = e->m;
  for (int b = 1; b < e->nb; b++) {
    int par = m->body_parent[b], jt = m->body_jnt_type[b], d = m->body_dofadr[b];
    double *w = e->bw + 3 * b, *v = e->bv + 3 * b, *al = e->balpha + 3 * b, *ac = e->bacc + 3 * b;
    const double *wp = e->bw + 3 * par, *vp = e->bv + 3 * par, *alp = e->balpha + 3 * par, *acp = e->bacc + 3 * par;
    if (jt == JF) {
      memcpy(v, e->qvel + d, 3 * sizeof(double));
      matvec3(e->xmat + 9 * b, e->qvel + d + 3, w);
      al[0] = al[1] = al[2] = 0; ac[0] = ac[1] = ac[2] = 0;
      continue;
    }
    double r[3], t1[3], t2[3];
    for (int k = 0; k < 3; k++) r[k] = e->xpos[3 * b + k] - e->xpos[3 * par + k];
    cross3(wp, r, t1);
    for (int k = 0; k < 3; k++) { w[k] = wp[k]; v[k] = vp[k] + t1[k]; al[k] = alp[k]; }
    cross3(wp, t1, t2);
    cross3(alp, r, t1);
    for (int k = 0; k < 3; k++) ac[k] = acp[k] + t1[k] + t2[k];
    if (jt == JH) {
      double qa[3] = {e->dax[3 * d] * e->qvel[d], e->dax[3 * d + 1] * e->qvel[d], e->dax[3 * d + 2] * e->qvel[d]};
      cross3(wp, qa, t1);
      for (int k = 0; k < 3; k++) { w[k] += qa[k]; al[k] += t1[k]; }
    } else if (jt == JS) {
      double qa[3] = {e->dax[3 * d] * e->qvel[d], e->dax[3 * d + 1] * e->qvel[d], e->dax[3 * d + 2] * e->qvel[d]};
      cross3(wp, qa, t1);
      for (int k = 0; k < 3; k++) { v[k] += qa[k]; ac[k] += 2 * t1[k]; }
    }
  }
}

/* COM acceleration (velocity-product part) of body b */
static void com_acc_vp(const oracle_env* e, int b, double* a) {
  double c[3], t1[3], t2[3];
  for (int k = 0; k < 3; k++) c[k] = e->xcom[3 * b + k] - e->xpos[3 * b + k];
  cross3(e->balpha + 3 * b, c, t1);
  cross3(e->bw + 3 * b, c, t2);
  cross3(e->bw + 3 * b, t2, t2);
  for (int k = 0; k < 3; k++) a[k] = e->bacc[3 * b + k] + t1[k] + t2[k];
}

/* M (Jacobian-sum form of mj_crb) and qfrc_bias (mj_rne with qacc = 0) */
static void inertia_bias(oracle_env* e) {
  const usim_model* m = e->m;
  int nv = e->nv;
  memset(e->M, 0, sizeof(double) * nv * nv);
  memset(e->bias, 0, sizeof(double) * nv);
  double Jp[3 * MAXCH], Jr[3 * MAXCH];
  for (int b = 1; b < e->nb; b++) {
    double mass = m->body_mass[b];
    if (mass <= 0 || e->chn[b] == 0) continue;
    const int* dofs;
    int n = jac_point(e, b, e->xcom + 3 * b, Jp, Jr, &dofs);
    const double* Iw = e->ximat + 9 * b;
    double IJr[3 * MAXCH];
    for (int i = 0; i < n; i++) matvec3(Iw, Jr + 3 * i, IJr + 3 * i);
    for (int i = 0; i < n; i++)
      for (int j = 0; j < n; j++)
        e->M[dofs[i] * nv + dofs[j]] += mass * dot3(Jp + 3 * i, Jp + 3 * j) + dot3(Jr + 3 * i, IJr + 3 * j);
    double a[3], F[3], N[3], Iw_w[3], t[3];
    com_acc_vp(e, b, a);
    for (int k = 0; k < 3; k++) F[k] = mass * (a[k] - m->gravity[k]);
    matvec3(Iw, e->bw + 3 * b, Iw_w);
    cross3(e->bw + 3 * b, Iw_w, t);
    matvec3(Iw, e->balpha + 3 * b, N);
    for (int k = 0; k < 3; k++) N[k] += t[k];
    for (int i = 0; i < n; i++) e->bias[dofs[i]] += dot3(Jp + 3 * i, F) + dot3(Jr + 3 * i, N);
  }
}

/* ------------------------------------------------------------------ OSC_POSE controller [C.2, C.3] */
static void eef_state(oracle_env* e) {
  const usim_model* m = e->m;
  int pb = m->probe_body, hb = m->hand_body;
  double Jp[3 * MAXCH], Jr[3 * MAXCH];
  const int* dofs;
  int n = jac_point(e, pb, e->xpos + 3 * pb, Jp, Jr, &dofs); /* grip_site == probe body origin */
  for (int i = 0; i < n; i++)
    for (int k = 0; k < 3; k++) { e->Jsite[7 * k + dofs[i]] = Jp[3 * i + k]; e->Jsite[7 * (3 + k) + dofs[i]] = Jr[3 * i + k]; }
  n = jac_point(e, hb, e->xpos + 3 * hb, Jp, Jr, &dofs);
  for (int i = 0; i < n; i++)
    for (int k = 0; k < 3; k++) e->Jhand[7 * k + dofs[i]] = Jp[3 * i + k];
  memcpy(e->eef_pos, e->xpos + 3 * pb, 3 * sizeof(double));
  memcpy(e->eef_mat, e->xmat + 9 * pb, 9 * sizeof(double));
  oracle_mat2quat_xyzw(e->eef_mat, e->eef_quat);
}

static double scale1(double a, double imin, double imax, double omin, double omax) {
  a = a < imin ? imin : (a > imax ? imax : a);
  return (a - 0.5 * (imax + imin)) * (fabs(omax - omin) / fabs(imax - imin)) + 0.5 * (omax + omin);
}

static void xyzw2mat(const double* q, double* R) {
  double w[4] = {q[3], q[0], q[1], q[2]};
  double n = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2] + w[3] * w[3]);
  for (int k = 0; k < 4; k++) w[k] /= n;
  quat2mat(w, R);
}

/* 0.5 * sum_i cur[:,i] x des[:,i]  (robosuite control_utils.orientation_error) */
static void ori_error(const double* des, const double* cur, double* err) {
  err[0] = err[1] = err[2] = 0;
  for (int i = 0; i < 3; i++) {
    double c[3] = {cur[i], cur[3 + i], cur[6 + i]}, d[3] = {des[i], des[3 + i], des[6 + i]}, x[3];
    cross3(c, d, x);
    for (int k = 0; k < 3; k++) err[k] += 0.5 * x[k];
  }
}

/* osc.set_goal on the policy step: goal pose into the task state */
static void set_goal(oracle_env* e, const double* action) {
  const usim_config* c = &e->cfg;
  double* gp = e->ts + USIM_TS_GOAL_POS;
  double* gR = e->ts + USIM_TS_GOAL_ORI;
  if (c->impedance_mode == USIM_MODE_FIXED) {
    double delta[6];
    for (int i = 0; i < 6; i++) delta[i] = scale1(action[i], c->input_min, c->input_max, c->output_min[i], c->output_max[i]);
    for (int k = 0; k < 3; k++) gp[k] = e->eef_pos[k] + delta[k];
    /* goal_ori only moves when some ori delta is non-zero (math.isclose(elem, 0.)); otherwise it persists */
    if (delta[3] != 0 || delta[4] != 0 || delta[5] != 0) {
      double ang = sqrt(delta[3] * delta[3] + delta[4] * delta[4] + delta[5] * delta[5]);
      double q[4] = {cos(ang / 2), sin(ang / 2) * delta[3] / ang, sin(ang / 2) * delta[4] / ang, sin(ang / 2) * delta[5] / ang}, Rd[9];
      quat2mat(q, Rd);
      matmul3(Rd, e->eef_mat, gR);
    }
  } else if (c->impedance_mode != USIM_MODE_WRENCH) { /* tracking / variable_z: goal = trajectory point + goal_quat [C.3] */
    for (int k = 0; k < 3; k++) gp[k] = e->ts[USIM_TS_TRAJ_PT + k];
    if (c->impedance_mode == USIM_MODE_VARIABLE_Z) gp[2] += scale1(action[6], -1, 1, -0.05, 0.05);
    xyzw2mat(GOAL_QUAT_XYZW, gR);
  }
}

/* osc.run_controller; needs kinematics(), velocities(), inertia_bias(), eef_state() at the current state */
static void controller(oracle_env* e, const double* action, double* tau) {
  const usim_config* c = &e->cfg;
  double kp[6], kd[6];
  const double* goal_pos = e->ts + USIM_TS_GOAL_POS;
  const double* goal_R = e->ts + USIM_TS_GOAL_ORI;
  const double* J = e->Jsite;
  int wrench_mode = c->impedance_mode == USIM_MODE_WRENCH;
  for (int i = 0; i < 6; i++) {
    if (c->impedance_mode == USIM_MODE_FIXED) { kp[i] = c->kp[i]; kd[i] = 2 * sqrt(kp[i]) * c->damping_ratio[i]; }
    else { kp[i] = scale1(action[i], c->kp_input_min, c->kp_input_max, c->kp_limits[0], c->kp_limits[1]); kd[i] = 2 * sqrt(kp[i]); }
  }
  double vel[6] = {0};
  for (int r = 0; r < 6; r++)
    for (int j = 0; j < 7; j++) vel[r] += J[7 * r + j] * e->qvel[j];
  double F[6];
  if (wrench_mode) {
    for (int i = 0; i < 6; i++) F[i] = action[i] < -10 ? -10 : (action[i] > 10 ? 10 : action[i]);
  } else {
    double eo[3];
    ori_error(goal_R, e->eef_mat, eo);
    for (int k = 0; k < 3; k++) {
      F[k] = kp[k] * (goal_pos[k] - e->eef_pos[k]) - kd[k] * vel[k];
      F[3 + k] = kp[3 + k] * eo[k] - kd[3 + k] * vel[3 + k];
    }
  }
  /* opspace matrices */
  double Ma[49], Minv[49];
  for (int i = 0; i < 7; i++)
    for (int j = 0; j < 7; j++) Ma[7 * i + j] = e->M[i * e->nv + j];
  { /* inv(M) through Cholesky (np.linalg.inv of an SPD matrix) */
    double Lc[49];
    memcpy(Lc, Ma, sizeof Lc);
    chol(Lc, 7);
    for (int j = 0; j < 7; j++) {
      double col[7] = {0};
      col[j] = 1;
      chol_solve(Lc, 7, col);
      for (int i = 0; i < 7; i++) Minv[7 * i + j] = col[i];
    }
  }
  double MiJt[42]; /* 7x6 */
  for (int i = 0; i < 7; i++)
    for (int r = 0; r < 6; r++) {
      double s = 0;
      for (int k = 0; k < 7; k++) s += Minv[7 * i + k] * J[7 * r + k];
      MiJt[6 * i + r] = s;
    }
  double Lfi[36], Lf[36], Lpi[9], Lp[9], Loi[9], Lo[9];
  for (int r = 0; r < 6; r++)
    for (int s2 = 0; s2 < 6; s2++) {
      double s = 0;
      for (int k = 0; k < 7; k++) s += J[7 * r + k] * MiJt[6 * k + s2];
      Lfi[6 * r + s2] = s;
    }
  for (int r = 0; r < 3; r++)
    for (int s2 = 0; s2 < 3; s2++) { Lpi[3 * r + s2] = Lfi[6 * r + s2]; Loi[3 * r + s2] = Lfi[6 * (3 + r) + 3 + s2]; }
  sym_pinv(Lfi, 6, Lf); sym_pinv(Lpi, 3, Lp); sym_pinv(Loi, 3, Lo);
  double W[6];
  if (wrench_mode) {
    memcpy(W, F, sizeof W);
  } else if (c->uncouple_pos_ori) {
    matvec3(Lp, F, W); matvec3(Lo, F + 3, W + 3);
  } else {
    for (int r = 0; r < 6; r++) { W[r] = 0; for (int k = 0; k < 6; k++) W[r] += Lf[6 * r + k] * F[k]; }
  }
  for (int j = 0; j < 7; j++) {
    double s = e->bias[j];
    for (int r = 0; r < 6; r++) s += J[7 * r + j] * W[r];
    tau[j] = s;
  }
  /* null-space torques: N^T M (kp (q_init - q) - kv qd), kp 10, kv 2 sqrt(10) */
  double pose[7], Mp[7], Jbar[42]; /* Jbar 7x6 = Minv J^T Lf */
  for (int j = 0; j < 7; j++) pose[j] = 10.0 * (e->ts[USIM_TS_INIT_JOINT + j] - e->qpos[j]) - 2 * sqrt(10.0) * e->qvel[j];
  for (int i = 0; i < 7; i++) { Mp[i] = 0; for (int j = 0; j < 7; j++) Mp[i] += Ma[7 * i + j] * pose[j]; }
  for (int i = 0; i < 7; i++)
    for (int r = 0; r < 6; r++) {
      double s = 0;
      for (int k = 0; k < 6; k++) s += MiJt[6 * i + k] * Lf[6 * k + r];
      Jbar[6 * i + r] = s;
    }
  /* N = I - Jbar J ; tau += N^T Mp */
  for (int j = 0; j < 7; j++) {
    double s = Mp[j];
    for (int i = 0; i < 7; i++) {
      double nij = 0; /* (Jbar J)[i][j] */
      for (int r = 0; r < 6; r++) nij += Jbar[6 * i + r] * J[7 * r + j];
      s -= nij * Mp[i];
    }
    tau[j] += s;
  }
  for (int j = 0; j < 7; j++) {
    double lim = e->m->ctrl_range[j];
    tau[j] = tau[j] < -lim ? -lim : (tau[j] > lim ? lim : tau[j]);
  }
}

/* ------------------------------------------------------------------ collision (mj_collision) [C.5] */
static void make_frame(const double* n, double* F) {
  double t[3] = {0, 0, 0};
  if (n[1] < 0.5 && n[1] > -0.5) t[1] = 1; else t[2] = 1;
  double d = dot3(n, t), y[3] = {t[0] - n[0] * d, t[1] - n[1] * d, t[2] - n[2] * d}, l = norm3(y), z[3];
  for (int k = 0; k < 3; k++) y[k] /= l;
  cross3(n, y, z);
  memcpy(F, n, 3 * sizeof(double)); memcpy(F + 3, y, 3 * sizeof(double)); memcpy(F + 6, z, 3 * sizeof(double));
}

static void add_contact(oracle_env* e, int g1, int g2, int b1, int b2, const double* pos, const double* n, double dist,
                        double fr, int probe_side, int torso) {
  if (e->ncon >= USIM_MAX_CONTACTS) return;
  ocontact* c = &e->con[e->ncon++];
  c->geom1 = g1; c->geom2 = g2; c->body1 = b1; c->body2 = b2; c->dist = dist; c->friction = fr;
  memcpy(c->pos, pos, sizeof c->pos);
  make_frame(n, c->frame);
  c->probe_side = probe_side; c->torso = torso;
  c->force[0] = c->force[1] = c->force[2] = 0;
}

/* closest points of two segments (Ericson, Real-Time Collision Detection 5.1.9) */
static void seg_seg(const double* p1, const double* q1, const double* p2, const double* q2, double* c1, double* c2) {
  double d1[3], d2[3], r[3];
  for (int k = 0; k < 3; k++) { d1[k] = q1[k] - p1[k]; d2[k] = q2[k] - p2[k]; r[k] = p1[k] - p2[k]; }
  double a = dot3(d1, d1), ee = dot3(d2, d2), f = dot3(d2, r), s, t;
  double c = dot3(d1, r), b = dot3(d1, d2), den = a * ee - b * b;
  if (den > 1e-14 * a * ee) { s = (b * f - c * ee) / den; s = s < 0 ? 0 : (s > 1 ? 1 : s); } else s = 0;
  t = (b * s + f) / ee;
  if (t < 0) { t = 0; s = -c / a; s = s < 0 ? 0 : (s > 1 ? 1 : s); }
  else if (t > 1) { t = 1; s = (b - c) / a; s = s < 0 ? 0 : (s > 1 ? 1 : s); }
  for (int k = 0; k < 3; k++) { c1[k] = p1[k] + d1[k] * s; c2[k] = p2[k] + d2[k] * t; }
}

static void collide(oracle_env* e) {
  const usim_model* m = e->m;
  e->ncon = 0;
  int pb = m->probe_body;
  double ptip[3], pback[3], t[3];
  matvec3(e->xmat + 9 * pb, m->probe_seg, t);
  for (int k = 0; k < 3; k++) ptip[k] = e->xpos[3 * pb + k] + t[k];
  matvec3(e->xmat + 9 * pb, m->probe_seg + 3, t);
  for (int k = 0; k < 3; k++) pback[k] = e->xpos[3 * pb + k] + t[k];
  double up[3] = {0, 0, 1}, down[3] = {0, 0, -1};
  /* body pair (table, probe): table body id is lowest.  geom1 = table (box), geom2 = probe (mesh in the reference) */
  const double* ends[2] = {ptip, pback};
  for (int i = 0; i < 2; i++) {
    const double* c = ends[i];
    double dist = c[2] - m->probe_radius - m->table_top_z;
    if (dist < 0 && fabs(c[0]) <= m->table_half_xy && fabs(c[1]) <= m->table_half_xy) {
      double pos[3] = {c[0], c[1], m->table_top_z + 0.5 * dist};
      add_contact(e, 1, 2, m->table_body, pb, pos, up, dist, fmax(m->table_friction, m->probe_friction), +1, 0);
    }
  }
  if (!m->soft) return;
  /* (table, particle k): geom1 = particle capsule, geom2 = table box -> normal points down */
  for (int k = 0; k < e->npart; k++) {
    int b = m->part_body0 + k;
    const double* segs[2] = {m->part_seg_outer + 3 * k, m->part_seg_inner + 3 * k};
    for (int i = 0; i < 2; i++) {
      double c[3];
      matvec3(e->xmat + 9 * b, segs[i], c);
      for (int j = 0; j < 3; j++) c[j] += e->xpos[3 * b + j];
      double dist = c[2] - m->cap_radius - m->table_top_z;
      if (dist < 0 && fabs(c[0]) <= m->table_half_xy && fabs(c[1]) <= m->table_half_xy) {
        double pos[3] = {c[0], c[1], m->table_top_z + 0.5 * dist};
        add_contact(e, 4 + k, 1, b, m->table_body, pos, down, dist, fmax(m->table_friction, m->particle_friction), 0, 0);
      }
    }
  }
  /* (probe, particle k): geom1 = particle capsule, geom2 = probe */
  for (int k = 0; k < e->npart; k++) {
    int b = m->part_body0 + k;
    double a0[3], a1[3], c1[3], c2[3];
    matvec3(e->xmat + 9 * b, m->part_seg_outer + 3 * k, a0);
    matvec3(e->xmat + 9 * b, m->part_seg_inner + 3 * k, a1);
    for (int j = 0; j < 3; j++) { a0[j] += e->xpos[3 * b + j]; a1[j] += e->xpos[3 * b + j]; }
    seg_seg(a0, a1, ptip, pback, c1, c2);
    double d[3] = {c2[0] - c1[0], c2[1] - c1[1], c2[2] - c1[2]}, len = norm3(d);
    double dist = len - m->cap_radius - m->probe_radius;
    if (dist < 0) {
      double n[3] = {0, 0, 1};
      if (len > 1e-12) for (int j = 0; j < 3; j++) n[j] = d[j] / len;
      double pos[3];
      for (int j = 0; j < 3; j++) pos[j] = c1[j] + n[j] * (m->cap_radius + 0.5 * dist);
      add_contact(e, 4 + k, 2, b, pb, pos, n, dist, fmax(m->particle_friction, m->probe_friction), +1, 1);
    }
  }
}

/* ------------------------------------------------------------------ constraint rows (mj_makeConstraint) [C.5] */
static void kbi(const oracle_env* e, const double* solref, const double* solimp, double pos, double* K, double* B, double* imp) {
  double dmin = solimp[0], dmax = solimp[1], width = solimp[2], mid = solimp[3], power = solimp[4];
  double x = fabs(pos) / width, y;
  if (x >= 1) y = 1;
  else if (x <= mid) y = pow(x, power) / pow(mid, power - 1);
  else y = 1 - pow(1 - x, power) / pow(1 - mid, power - 1);
  double d = dmin + y * (dmax - dmin);
  d = d < 1e-4 ? 1e-4 : (d > 0.9999 ? 0.9999 : d);
  *imp = d;
  if (solref[0] > 0) {
    double tc = fmax(solref[0], 2 * e->m->timestep), dr = solref[1];
    *K = 1.0 / (dmax * dmax * tc * tc * dr * dr);
    *B = 2.0 / (dmax * tc);
  } else {
    *K = -solref[0] / (dmax * dmax);
    *B = -solref[1] / dmax;
  }
}

static int new_row(oracle_env* e, int type, int n) {
  int r = e->nefc++;
  e->rstart[r] = e->pool_n; e->rn[r] = n; e->rtype[r] = type;
  e->pool_n += n;
  e->rmu[r] = 0; e->rfr[r] = 0;
  return r;
}

static void finish_row(oracle_env* e, int r, const double* solref, double pos, double diag, int use_pos) {
  double K, B, imp, vel = 0;
  for (int i = 0; i < e->rn[r]; i++) vel += e->pval[e->rstart[r] + i] * e->qvel[e->pidx[e->rstart[r] + i]];
  kbi(e, solref, e->m->solimp, pos, &K, &B, &imp);
  e->raref[r] = -B * vel - (use_pos ? K * imp * pos : 0);
  double R = fmax(MJMINVAL, (1 - imp) / imp * diag);
  e->rD[r] = 1 / R;
}

static void make_constraints(oracle_env* e) {
  const usim_model* m = e->m;
  e->nefc = 0; e->pool_n = 0;
  if (m->soft) {
    double srs[2] = {-e->ts[USIM_TS_STIFFNESS], -e->ts[USIM_TS_DAMPING]};
    for (int i = 0; i < e->npart; i++) { /* "fix": q_i - 0 = 0 */
      int d = 13 + i, r = new_row(e, ROW_EQ, 1);
      e->pidx[e->rstart[r]] = d; e->pval[e->rstart[r]] = 1;
      finish_row(e, r, m->solref, e->qpos[14 + i], m->dof_invweight0[d], 1);
    }
    for (int p = 0; p < m->npair; p++) { /* "smooth": q_a - q_b = 0, carries solrefsmooth */
      int a = m->eq_pairs[2 * p], b = m->eq_pairs[2 * p + 1], r = new_row(e, ROW_EQ, 2);
      e->pidx[e->rstart[r]] = 13 + a; e->pval[e->rstart[r]] = 1;
      e->pidx[e->rstart[r] + 1] = 13 + b; e->pval[e->rstart[r] + 1] = -1;
      finish_row(e, r, srs, e->qpos[14 + a] - e->qpos[14 + b], m->dof_invweight0[13 + a] + m->dof_invweight0[13 + b], 1);
    }
    { /* tendon: sum q = 0 */
      int r = new_row(e, ROW_EQ, e->npart);
      double s = 0;
      for (int i = 0; i < e->npart; i++) { e->pidx[e->rstart[r] + i] = 13 + i; e->pval[e->rstart[r] + i] = 1; s += e->qpos[14 + i]; }
      finish_row(e, r, m->solref, s, m->tendon_invweight0, 1);
    }
  }
  for (int j = 0; j < 7; j++) { /* joint limits, margin 0 */
    double lo = m->jnt_range[2 * j], hi = m->jnt_range[2 * j + 1], q = e->qpos[j];
    for (int side = 0; side < 2; side++) {
      double dist = side == 0 ? q - lo : hi - q;
      if (dist < 0) {
        int r = new_row(e, ROW_LIMIT, 1);
        e->pidx[e->rstart[r]] = j; e->pval[e->rstart[r]] = side == 0 ? 1 : -1;
        finish_row(e, r, m->solref, dist, m->dof_invweight0[j], 1);
      }
    }
  }
  double Jp[3 * MAXCH], Jr[3 * MAXCH];
  for (int ci = 0; ci < e->ncon; ci++) {
    ocontact* c = &e->con[ci];
    const int *d1, *d2;
    int n1 = e->chn[c->body1], n2 = e->chn[c->body2];
    int r0 = -1;
    for (int j = 0; j < 3; j++) {
      int r = new_row(e, j == 0 ? ROW_CONTACT : ROW_EQ + 100, n1 + n2);
      if (j == 0) r0 = r;
    }
    c->row = r0;
    int n = jac_point(e, c->body1, c->pos, Jp, Jr, &d1);
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) {
        e->pidx[e->rstart[r0 + j] + i] = d1[i];
        e->pval[e->rstart[r0 + j] + i] = -dot3(c->frame + 3 * j, Jp + 3 * i);
      }
    n = jac_point(e, c->body2, c->pos, Jp, Jr, &d2);
    for (int i = 0; i < n; i++)
      for (int j = 0; j < 3; j++) {
        e->pidx[e->rstart[r0 + j] + n1 + i] = d2[i];
        e->pval[e->rstart[r0 + j] + n1 + i] = dot3(c->frame + 3 * j, Jp + 3 * i);
      }
    double diag = m->body_invweight0[2 * c->body1] + m->body_invweight0[2 * c->body2];
    finish_row(e, r0, m->solref, c->dist, diag, 1);
    double Rn = 1 / e->rD[r0], Rt = Rn / m->impratio;
    e->rmu[r0] = c->friction * sqrt(Rt / Rn);
    for (int j = 1; j < 3; j++) {
      finish_row(e, r0 + j, m->solref, c->dist, diag, 0); /* aref = -B vel, same impedance as the normal */
      e->rD[r0 + j] = 1 / Rt;
      e->rfr[r0 + j] = c->friction;
    }
    e->rfr[r0] = c->friction;
  }
}

/* forces, cost, and (optionally) per-contact 3x3 Hessian wrt jar; returns cost of the constraint part */
static double constraint_update(oracle_env* e, const double* jar, double* frc, double* hc /* 9 per contact or NULL */) {
  double cost = 0;
  int ci = 0;
  for (int r = 0; r < e->nefc; r++) {
    int t = e->rtype[r];
    if (t == ROW_EQ) {
      frc[r] = -e->rD[r] * jar[r];
      cost += 0.5 * e->rD[r] * jar[r] * jar[r];
    } else if (t == ROW_LIMIT) {
      if (jar[r] < 0) { frc[r] = -e->rD[r] * jar[r]; cost += 0.5 * e->rD[r] * jar[r] * jar[r]; }
      else frc[r] = 0;
    } else if (t == ROW_CONTACT) {
      double mu = e->rmu[r], fr = e->rfr[r];
      double U0 = jar[r] * mu, U1 = jar[r + 1] * fr, U2 = jar[r + 2] * fr;
      double N = U0, T = sqrt(U1 * U1 + U2 * U2);
      double* h = hc ? hc + 9 * ci : NULL;
      if (h) memset(h, 0, 9 * sizeof(double));
      if (N >= mu * T || (T <= 0 && N >= 0)) { /* top zone */
        frc[r] = frc[r + 1] = frc[r + 2] = 0;
      } else if (mu * N + T <= 0 || (T <= 0 && N < 0)) { /* bottom zone */
        for (int j = 0; j < 3; j++) {
          frc[r + j] = -e->rD[r + j] * jar[r + j];
          cost += 0.5 * e->rD[r + j] * jar[r + j] * jar[r + j];
          if (h) h[4 * j] = e->rD[r + j];
        }
      } else { /* middle zone */
        double Dm = e->rD[r] / (mu * mu * (1 + mu * mu)), NmT = N - mu * T;
        cost += 0.5 * Dm * NmT * NmT;
        frc[r] = -Dm * NmT * mu;
        frc[r + 1] = -frc[r] / T * U1 * fr;
        frc[r + 2] = -frc[r] / T * U2 * fr;
        if (h) {
          double g[3] = {1, -mu * U1 / T, -mu * U2 / T}, s[3] = {mu, fr, fr}, u[2] = {U1 / T, U2 / T};
          double HU[9];
          for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++) HU[3 * a + b] = Dm * g[a] * g[b];
          double k = -Dm * mu * NmT / T;
          for (int a = 0; a < 2; a++)
            for (int b = 0; b < 2; b++) HU[3 * (a + 1) + b + 1] += k * ((a == b) - u[a] * u[b]);
          for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++) h[3 * a + b] = s[a] * HU[3 * a + b] * s[b];
        }
      }
      ci++;
      r += 2;
    }
  }
  return cost;
}

static void row_mul(const oracle_env* e, const double* x, double* out) { /* out = J x */
  for (int r = 0; r < e->nefc; r++) {
    double s = 0;
    const int* idx = e->pidx + e->rstart[r];
    const double* val = e->pval + e->rstart[r];
    for (int i = 0; i < e->rn[r]; i++) s += val[i] * x[idx[i]];
    out[r] = s;
  }
}

static void sym_mul(const double* M, int n, const double* x, double* y) {
  for (int i = 0; i < n; i++) {
    double s = 0;
    const double* r = M + (size_t)i * n;
    for (int j = 0; j < n; j++) s += r[j] * x[j];
    y[i] = s;
  }
}

/* Newton solver of the primal problem (mj_solNewton semantics: exact Hessian, exact line search) */
static void solve(oracle_env* e) {
  int nv = e->nv, nefc = e->nefc;
  double* a = e->qacc;
  double* hc = (double*)malloc(sizeof(double) * 9 * (e->ncon + 1));
  double* dcost = (double*)malloc(sizeof(double) * (nefc + 1));
  /* warm start: pick the cheaper of qacc_warmstart and qacc_smooth */
  double best = 1e300;
  for (int trial = 0; trial < 2; trial++) {
    const double* x = trial == 0 ? e->warm : e->a0;
    row_mul(e, x, e->jar);
    for (int r = 0; r < nefc; r++) e->jar[r] -= e->raref[r];
    double c = constraint_update(e, e->jar, e->frc, NULL);
    for (int i = 0; i < nv; i++) e->tmp[i] = x[i] - e->a0[i];
    sym_mul(e->M, nv, e->tmp, e->Ma);
    for (int i = 0; i < nv; i++) c += 0.5 * e->tmp[i] * e->Ma[i];
    if (c < best) { best = c; memcpy(a, x, sizeof(double) * nv); }
  }
  double qsn = 0;
  for (int i = 0; i < nv; i++) qsn += e->qs[i] * e->qs[i];
  qsn = sqrt(qsn);
  e->solver_iter = 0;
  for (int it = 0; it < 100; it++) {
    sym_mul(e->M, nv, a, e->Ma);
    row_mul(e, a, e->jar);
    for (int r = 0; r < nefc; r++) e->jar[r] -= e->raref[r];
    constraint_update(e, e->jar, e->frc, hc);
    for (int i = 0; i < nv; i++) e->grad[i] = e->Ma[i] - e->qs[i];
    for (int r = 0; r < nefc; r++) {
      double f = e->frc[r];
      if (f == 0) continue;
      const int* idx = e->pidx + e->rstart[r];
      const double* val = e->pval + e->rstart[r];
      for (int i = 0; i < e->rn[r]; i++) e->grad[idx[i]] -= val[i] * f;
    }
    double gn = 0;
    for (int i = 0; i < nv; i++) gn += e->grad[i] * e->grad[i];
    gn = sqrt(gn);
    e->solver_grad = gn;
    if (gn <= 1e-11 * (1 + qsn)) break;
    e->solver_iter = it + 1;
    /* Hessian */
    memcpy(e->H, e->M, sizeof(double) * nv * nv);
    int ci = 0;
    for (int r = 0; r < nefc; r++) {
      int t = e->rtype[r];
      const int* idx = e->pidx + e->rstart[r];
      const double* val = e->pval + e->rstart[r];
      int n = e->rn[r];
      if (t == ROW_EQ || (t == ROW_LIMIT && e->jar[r] < 0)) {
        double D = e->rD[r];
        for (int i = 0; i < n; i++)
          for (int j = 0; j < n; j++) e->H[idx[i] * nv + idx[j]] += D * val[i] * val[j];
      } else if (t == ROW_CONTACT) {
        const double* h = hc + 9 * ci;
        for (int a2 = 0; a2 < 3; a2++)
          for (int b2 = 0; b2 < 3; b2++) {
            double hab = h[3 * a2 + b2];
            if (hab == 0) continue;
            const double* va = e->pval + e->rstart[r + a2];
            const double* vb = e->pval + e->rstart[r + b2];
            for (int i = 0; i < n; i++)
              for (int j = 0; j < n; j++) e->H[idx[i] * nv + idx[j]] += hab * va[i] * vb[j];
          }
        ci++;
        r += 2;
      }
    }
    if (chol(e->H, nv) != 0) break;
    for (int i = 0; i < nv; i++) e->dir[i] = -e->grad[i];
    chol_solve(e->H, nv, e->dir);
    /* exact line search on phi'(alpha) */
    row_mul(e, e->dir, e->jv);
    sym_mul(e->M, nv, e->dir, e->tmp);
    double g0 = 0, g2 = 0; /* Gauss part: phi' = g0 + alpha g2 */
    for (int i = 0; i < nv; i++) { g0 += e->dir[i] * (e->Ma[i] - e->qs[i]); g2 += e->dir[i] * e->tmp[i]; }
    double lo = 0, hi = -1, alpha = 1, d0 = 0;
    double* jt = dcost; /* scratch: jar at alpha */
    double* ft = (double*)malloc(sizeof(double) * (nefc + 1));
    for (int ls = 0; ls < 80; ls++) {
      for (int r = 0; r < nefc; r++) jt[r] = e->jar[r] + alpha * e->jv[r];
      constraint_update(e, jt, ft, hc);
      double d1 = g0 + alpha * g2, d2 = g2;
      int cj = 0;
      for (int r = 0; r < nefc; r++) {
        d1 -= ft[r] * e->jv[r];
        int t = e->rtype[r];
        if (t == ROW_EQ || (t == ROW_LIMIT && jt[r] < 0)) d2 += e->rD[r] * e->jv[r] * e->jv[r];
        else if (t == ROW_CONTACT) {
          const double* h = hc + 9 * cj;
          for (int a2 = 0; a2 < 3; a2++)
            for (int b2 = 0; b2 < 3; b2++) d2 += h[3 * a2 + b2] * e->jv[r + a2] * e->jv[r + b2];
          for (int j = 1; j < 3; j++) d1 -= ft[r + j] * e->jv[r + j];
          cj++;
          r += 2;
        }
      }
      if (ls == 0) d0 = fabs(g0) + 1e-300;
      if (fabs(d1) <= 1e-14 * d0) break;
      if (d1 < 0) lo = alpha; else hi = alpha;
      double an = alpha - d1 / d2;
      if (hi < 0) { if (an <= lo) an = 2 * alpha; }
      else if (an <= lo || an >= hi) an = 0.5 * (lo + hi);
      if (fabs(an - alpha) <= 1e-16 * fabs(alpha)) { alpha = an; break; }
      alpha = an;
    }
    free(ft);
    for (int i = 0; i < nv; i++) a[i] += alpha * e->dir[i];
  }
  /* final forces */
  row_mul(e, a, e->jar);
  for (int r = 0; r < nefc; r++) e->jar[r] -= e->raref[r];
  constraint_update(e, e->jar, e->frc, NULL);
  memset(e->fcon, 0, sizeof(double) * nv);
  for (int r = 0; r < nefc; r++) {
    const int* idx = e->pidx + e->rstart[r];
    const double* val = e->pval + e->rstart[r];
    for (int i = 0; i < e->rn[r]; i++) e->fcon[idx[i]] += val[i] * e->frc[r];
  }
  free(hc); free(dcost);
}

/* ------------------------------------------------------------------ forward / integrate */
static void forward_posvel(oracle_env* e) {
  kinematics(e);
  velocities(e);
  inertia_bias(e);
  eef_state(e);
}

/* mj_rnePostConstraint + sensors for the probe body: cfrc_ext force, F/T torque at ft_frame */
static void post_constraint(oracle_env* e) {
  const usim_model* m = e->m;
  int pb = m->probe_body;
  const double* site = e->xpos + 3 * pb;
  double F[3] = {0, 0, 0}, Tq[3] = {0, 0, 0};
  e->in_contact = 0;
  for (int ci = 0; ci < e->ncon; ci++) {
    ocontact* c = &e->con[ci];
    for (int j = 0; j < 3; j++) c->force[j] = e->frc[c->row + j];
    if (!c->probe_side) continue;
    double f[3];
    for (int k = 0; k < 3; k++)
      f[k] = c->probe_side * (c->force[0] * c->frame[k] + c->force[1] * c->frame[3 + k] + c->force[2] * c->frame[6 + k]);
    double r[3] = {c->pos[0] - site[0], c->pos[1] - site[1], c->pos[2] - site[2]}, t[3];
    cross3(r, f, t);
    for (int k = 0; k < 3; k++) { F[k] += f[k]; Tq[k] += t[k]; }
    if (c->torso) e->in_contact = 1;
  }
  memcpy(e->cfrc, F, sizeof F);
  /* body acceleration of the probe from qacc */
  double Jp[3 * MAXCH], Jr[3 * MAXCH], acom[3], alpha[3];
  const int* dofs;
  int n = jac_point(e, pb, e->xcom + 3 * pb, Jp, Jr, &dofs);
  com_acc_vp(e, pb, acom);
  memcpy(alpha, e->balpha + 3 * pb, sizeof alpha);
  for (int i = 0; i < n; i++)
    for (int k = 0; k < 3; k++) { acom[k] += Jp[3 * i + k] * e->qacc[dofs[i]]; alpha[k] += Jr[3 * i + k] * e->qacc[dofs[i]]; }
  const double* Iw = e->ximat + 9 * pb;
  double Ia[3], Iw_w[3], gy[3], lin[3], r[3], t[3], tau[3];
  matvec3(Iw, alpha, Ia);
  matvec3(Iw, e->bw + 3 * pb, Iw_w);
  cross3(e->bw + 3 * pb, Iw_w, gy);
  for (int k = 0; k < 3; k++) { lin[k] = m->body_mass[pb] * (acom[k] - m->gravity[k]); r[k] = e->xcom[3 * pb + k] - site[k]; }
  cross3(r, lin, t);
  for (int k = 0; k < 3; k++) tau[k] = Ia[k] + gy[k] + t[k] - Tq[k];
  matTvec3(e->xmat + 9 * pb, tau, e->ft_torque);
}

static void forward_acc(oracle_env* e, const double* ctrl) {
  const usim_model* m = e->m;
  int nv = e->nv;
  for (int i = 0; i < nv; i++) { e->passive[i] = -m->dof_damping[i] * e->qvel[i]; e->act[i] = 0; }
  for (int j = 0; j < 7; j++) e->act[j] = ctrl[j];
  memcpy(e->L, e->M, sizeof(double) * nv * nv);
  chol(e->L, nv);
  for (int i = 0; i < nv; i++) e->a0[i] = e->passive[i] - e->bias[i] + e->act[i];
  memcpy(e->qs, e->a0, sizeof(double) * nv); /* qfrc_smooth */
  chol_solve(e->L, nv, e->a0);
  collide(e);
  make_constraints(e);
  solve(e);
  post_constraint(e);
}

void oracle_forward(oracle_env* e, const double* ctrl) {
  forward_posvel(e);
  forward_acc(e, ctrl);
}

/* The problem of the last forward pass (rows, a0, M, J, D, aref) evaluated at a given qacc; the env is left as it was.
 * rhs and Hx are formed as the device solver forms them: M plus the equality rows (fix, smooth, tendon) is its quadratic part H,
 *   rhs = qfrc_smooth + sum_eq J^T D aref,   Hx = H qacc - rhs (the kernel's Hx row holds the gradient of the quadratic part),
 *   grad = Hx - sum_other J^T f = M (qacc - a0) - J^T f,
 * and its stopping rule is |grad| <= tol (1 + |rhs| + |Hx|): norms[0] = |grad|, norms[1] = |rhs|, norms[2] = |Hx|. */
int oracle_evaluate(oracle_env* e, const double* qacc, double* grad, double* cost, double* efc_force, double* contact_force,
                    double* cfrc, double* ft_torque, double* norms) {
  int nv = e->nv, nefc = e->nefc;
  double* save_qacc = dalloc(nv);
  double* save_jar = dalloc(nefc);
  double* save_frc = dalloc(nefc);
  double* rhs = dalloc(nv);
  double* hx = dalloc(nv);
  double* g = dalloc(nv);
  double save_force[USIM_MAX_CONTACTS][3], save_cfrc[3], save_ft[3];
  int save_in_contact = e->in_contact;
  memcpy(save_qacc, e->qacc, sizeof(double) * nv);
  memcpy(save_jar, e->jar, sizeof(double) * nefc);
  memcpy(save_frc, e->frc, sizeof(double) * nefc);
  for (int c = 0; c < e->ncon; c++) memcpy(save_force[c], e->con[c].force, sizeof save_force[c]);
  memcpy(save_cfrc, e->cfrc, sizeof save_cfrc);
  memcpy(save_ft, e->ft_torque, sizeof save_ft);

  memcpy(e->qacc, qacc, sizeof(double) * nv);
  row_mul(e, qacc, e->jar);
  for (int r = 0; r < nefc; r++) e->jar[r] -= e->raref[r];
  double c = constraint_update(e, e->jar, e->frc, NULL);
  sym_mul(e->M, nv, qacc, hx);
  memcpy(rhs, e->qs, sizeof(double) * nv);
  for (int i = 0; i < nv; i++) e->tmp[i] = qacc[i] - e->a0[i];
  sym_mul(e->M, nv, e->tmp, g);
  for (int i = 0; i < nv; i++) c += 0.5 * e->tmp[i] * g[i];
  for (int r = 0; r < nefc; r++) {
    const int* idx = e->pidx + e->rstart[r];
    const double* val = e->pval + e->rstart[r];
    for (int i = 0; i < e->rn[r]; i++) {
      g[idx[i]] -= val[i] * e->frc[r];
      if (e->rtype[r] == ROW_EQ) {
        hx[idx[i]] += val[i] * e->rD[r] * (e->jar[r] + e->raref[r]);
        rhs[idx[i]] += val[i] * e->rD[r] * e->raref[r];
      }
    }
  }
  double gn = 0, rn = 0, hn = 0;
  for (int i = 0; i < nv; i++) { gn += g[i] * g[i]; rn += rhs[i] * rhs[i]; hn += (hx[i] - rhs[i]) * (hx[i] - rhs[i]); }
  post_constraint(e);
  if (grad) memcpy(grad, g, sizeof(double) * nv);
  if (cost) *cost = c;
  if (efc_force) memcpy(efc_force, e->frc, sizeof(double) * nefc);
  if (contact_force)
    for (int k = 0; k < e->ncon; k++) memcpy(contact_force + 3 * k, e->con[k].force, 3 * sizeof(double));
  if (cfrc) memcpy(cfrc, e->cfrc, sizeof e->cfrc);
  if (ft_torque) memcpy(ft_torque, e->ft_torque, sizeof e->ft_torque);
  if (norms) { norms[0] = sqrt(gn); norms[1] = sqrt(rn); norms[2] = sqrt(hn); }

  memcpy(e->qacc, save_qacc, sizeof(double) * nv);
  memcpy(e->jar, save_jar, sizeof(double) * nefc);
  memcpy(e->frc, save_frc, sizeof(double) * nefc);
  for (int k = 0; k < e->ncon; k++) memcpy(e->con[k].force, save_force[k], sizeof save_force[k]);
  memcpy(e->cfrc, save_cfrc, sizeof save_cfrc);
  memcpy(e->ft_torque, save_ft, sizeof save_ft);
  e->in_contact = save_in_contact;
  free(save_qacc); free(save_jar); free(save_frc); free(rhs); free(hx); free(g);
  return nefc;
}

/* row type of every constraint row of the last forward pass: 0 equality, 1 joint limit, 2 contact normal, 100 contact friction */
void oracle_efc_type(const oracle_env* e, int* type) { memcpy(type, e->rtype, sizeof(int) * e->nefc); }

/* mj_Euler: implicit joint damping, semi-implicit update, quaternion integration */
static void integrate(oracle_env* e) {
  const usim_model* m = e->m;
  int nv = e->nv;
  double h = m->timestep;
  memcpy(e->warm, e->qacc, sizeof(double) * nv);
  sym_mul(e->M, nv, e->qacc, e->tmp);
  memcpy(e->H, e->M, sizeof(double) * nv * nv);
  for (int i = 0; i < nv; i++) e->H[i * nv + i] += h * m->dof_damping[i];
  chol(e->H, nv);
  chol_solve(e->H, nv, e->tmp);
  for (int i = 0; i < nv; i++) e->qvel[i] += h * e->tmp[i];
  for (int b = 1; b < e->nb; b++) {
    int jt = m->body_jnt_type[b], qa = m->body_qposadr[b], d = m->body_dofadr[b];
    if (jt == JH || jt == JS) e->qpos[qa] += h * e->qvel[d];
    else if (jt == JF) {
      for (int k = 0; k < 3; k++) e->qpos[qa + k] += h * e->qvel[d + k];
      double* w = e->qvel + d + 3;
      double ang = h * norm3(w);
      if (ang > 0) {
        double s = sin(ang / 2) / norm3(w), qr[4] = {cos(ang / 2), s * w[0], s * w[1], s * w[2]};
        double* q = e->qpos + qa + 3;
        quatmul(q, qr, q);
        double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
        for (int k = 0; k < 4; k++) q[k] /= n;
      }
    }
  }
}

/* ------------------------------------------------------------------ task layer */
static void traj_eval(const oracle_env* e, double u, double* pt) { /* klampt Trajectory.eval, times [0,1], end behaviour "halt" */
  u = u < 0 ? 0 : (u > 1 ? 1 : u);
  for (int k = 0; k < 3; k++) pt[k] = e->ts[USIM_TS_TRAJ_START + k] + u * (e->ts[USIM_TS_TRAJ_END + k] - e->ts[USIM_TS_TRAJ_START + k]);
}

static void write_obs(const oracle_env* e, double* obs) { /* ultrasound.py:363-401 */
  if (!obs) return;
  for (int k = 0; k < 3; k++) { obs[k] = e->cfrc[k]; obs[3 + k] = e->ft_torque[k]; obs[6 + k] = e->hand_vel[k]; }
  obs[9] = e->ts[USIM_TS_FZ_MEAN] - 5;
  obs[10] = e->ts[USIM_TS_DFZ] - 0;
  obs[11] = e->ts[USIM_TS_VEL_MEAN] - 0.04;
  for (int k = 0; k < 3; k++) obs[12 + k] = e->eef_pos[k] - e->ts[USIM_TS_TRAJ_PT + k];
  oracle_difference_quat(e->eef_quat, GOAL_QUAT_XYZW, obs + 15); /* xyzw arrays fed to a wxyz routine (:390) */
}

static void hand_velocity(oracle_env* e) { /* robosuite _hand_vel: (stale) body Jacobian times current qvel */
  for (int k = 0; k < 3; k++) {
    double s = 0;
    for (int j = 0; j < 7; j++) s += e->Jhand[7 * k + j] * e->qvel[j];
    e->hand_vel[k] = s;
  }
}

void oracle_ik(oracle_env* e, const double* target, double* q7) {
  double Rg[9];
  xyzw2mat(GOAL_QUAT_XYZW, Rg);
  double save[7];
  memcpy(save, e->qpos, sizeof save);
  memcpy(e->qpos, e->m->init_qpos, sizeof save);
  for (int it = 0; it < 100; it++) {
    kinematics(e);
    eef_state(e);
    double err[6], eo[3];
    ori_error(Rg, e->eef_mat, eo);
    for (int k = 0; k < 3; k++) { err[k] = target[k] - e->eef_pos[k]; err[3 + k] = eo[k]; }
    double en = 0;
    for (int k = 0; k < 6; k++) en += err[k] * err[k];
    if (sqrt(en) < 1e-10) break;
    double A[36];
    for (int r = 0; r < 6; r++)
      for (int s = 0; s < 6; s++) {
        double v = r == s ? 1e-4 : 0;
        for (int j = 0; j < 7; j++) v += e->Jsite[7 * r + j] * e->Jsite[7 * s + j];
        A[6 * r + s] = v;
      }
    chol(A, 6);
    chol_solve(A, 6, err);
    double dq[7], mx = 0;
    for (int j = 0; j < 7; j++) {
      dq[j] = 0;
      for (int r = 0; r < 6; r++) dq[j] += e->Jsite[7 * r + j] * err[r];
      mx = fmax(mx, fabs(dq[j]));
    }
    double sc = mx > 0.5 ? 0.5 / mx : 1;
    for (int j = 0; j < 7; j++) e->qpos[j] += sc * dq[j];
  }
  memcpy(q7, e->qpos, sizeof save);
  memcpy(e->qpos, save, sizeof save);
}

void oracle_grid_point2(double tx, double ty, double tz, double xr, double yr, double top, int ix, int iy, double* pt);

void oracle_reset(oracle_env* e, double* obs) {
  const usim_model* m = e->m;
  const usim_config* c = &e->cfg;
  double* ts = e->ts;
  uint32_t ep = (uint32_t)ts[USIM_TS_EPISODE], r[4];
  /* hard reset: stiffness / damping re-drawn (ultrasound.py:291-297) */
  double k = -m->solref_smooth[0], b = -m->solref_smooth[1];
  if (c->solref_randomization) {
    oracle_philox(c->seed, (uint32_t)e->gid, ep, 0, 0, r);
    k = 1300 + (double)(r[0] % 300u);
    b = 17 + (double)(r[1] % 24u);
  }
  memset(ts, 0, sizeof e->ts);
  ts[USIM_TS_EPISODE] = ep + 1;
  ts[USIM_TS_STIFFNESS] = k; ts[USIM_TS_DAMPING] = b;
  memcpy(e->qpos, m->qpos0, sizeof(double) * e->nq);
  memset(e->qvel, 0, sizeof(double) * e->nv);
  memset(e->warm, 0, sizeof(double) * e->nv);
  /* trajectory (ultrasound.py:749-809) */
  double tx = 0, ty = 0, tz = 0.8 + 0.005 + 0.0522;
  if (m->soft) { tx = m->qpos0[7]; ty = m->qpos0[8]; tz = m->qpos0[9]; }
  if (c->deterministic_trajectory) {
    double s[3] = {0.062, -0.020, 0.896}, en[3] = {-0.032, -0.075, 0.896};
    memcpy(ts + USIM_TS_TRAJ_START, s, sizeof s); memcpy(ts + USIM_TS_TRAJ_END, en, sizeof en);
  } else {
    oracle_philox(c->seed, (uint32_t)e->gid, ep, 1, 0, r);
    oracle_grid_point2(tx, ty, tz, m->traj_x_range, m->traj_y_range, m->top_torso_offset, (int)(r[0] % 50u), (int)(r[1] % 50u), ts + USIM_TS_TRAJ_START);
    oracle_grid_point2(tx, ty, tz, m->traj_x_range, m->traj_y_range, m->top_torso_offset, (int)(r[2] % 50u), (int)(r[3] % 50u), ts + USIM_TS_TRAJ_END);
  }
  oracle_philox(c->seed, (uint32_t)e->gid, ep, 2, 0, r);
  ts[USIM_TS_U0] = u01(r[0]); /* ultrasound.py:443 (unseeded in the reference) */
  traj_eval(e, ts[USIM_TS_U0], ts + USIM_TS_TRAJ_PT);
  /* initial joint pose (ultrasound.py:812-887) */
  double q[7];
  memcpy(q, m->init_qpos, sizeof q);
  if (m->soft) {
    double target[3] = {ts[USIM_TS_TRAJ_PT], ts[USIM_TS_TRAJ_PT + 1], ts[USIM_TS_TRAJ_PT + 2]};
    if (c->probe_pos_randomization) {
      uint32_t r2[4];
      oracle_philox(c->seed, (uint32_t)e->gid, ep, 3, 0, r2);
      double rad = sqrt(-2 * log(u01(r[1]))), ang = 2 * PI * u01(r[2]);
      target[0] += 0.010 / 4 * rad * cos(ang);
      target[1] += 0.010 / 4 * rad * sin(ang);
      target[2] += 0.010 * sqrt(-2 * log(u01(r2[0]))) * cos(2 * PI * u01(r2[1]));
    }
    for (int j = 0; j < 3; j++) target[j] += c->reset_eef_bias[j];
    oracle_ik(e, target, q);
  }
  memcpy(e->qpos, q, sizeof q);
  memcpy(ts + USIM_TS_INIT_JOINT, q, sizeof q);
  /* sim.forward() with ctrl = 0 (new MjSim after a hard reset) */
  double zero[7] = {0};
  oracle_forward(e, zero);
  hand_velocity(e);
  ts[USIM_TS_FZ_PREV] = 0; ts[USIM_TS_DFZ] = 0;
  ts[USIM_TS_VEL_MEAN] = norm3(e->hand_vel);
  ts[USIM_TS_FZ_MEAN] = e->cfrc[2];
  ts[USIM_TS_TOUCHED] = 0; ts[USIM_TS_TIMESTEP] = 0; ts[USIM_TS_DONE] = 0;
  ts[USIM_TS_IN_CONTACT] = e->in_contact;
  memcpy(ts + USIM_TS_GOAL_ORI, e->eef_mat, sizeof e->eef_mat); /* osc.reset_goal via update_initial_joints (:465) */
  memcpy(ts + USIM_TS_GOAL_POS, e->eef_pos, sizeof e->eef_pos);
  memset(e->tau, 0, sizeof e->tau);
  write_obs(e, obs);
}

static void post_action_impl(double* ts, int horizon, int ignore_done, double control_freq, int early_termination, const double* jnt_range,
                             const double* eef_pos, const double* eef_quat_xyzw, const double* hand_vel, double fz, int in_contact,
                             const double* qpos7, double* reward, int* done);

int oracle_step(oracle_env* e, const double* action, double* obs, double* reward, int* done) {
  const usim_model* m = e->m;
  const usim_config* c = &e->cfg;
  double* ts = e->ts;
  if (ts[USIM_TS_DONE] != 0) return -1; /* "executing action in terminated episode" */
  ts[USIM_TS_TIMESTEP] += 1;
  int substeps = (int)((1.0 / c->control_freq) / m->timestep + 1e-9);
  if (substeps < 1) substeps = 1;
  for (int s = 0; s < substeps; s++) {
    /* the reference runs mj_forward three times per substep at the same state; the first two only differ by using
       the previous ctrl and leave no trace in the state (SURVEY 3.2).  `repeats` re-does them for timing only. */
    for (int rep = 1; rep < e->repeats; rep++) { forward_posvel(e); forward_acc(e, e->tau); }
    forward_posvel(e);
    if (s == 0) set_goal(e, action);
    controller(e, action, e->tau);
    forward_acc(e, e->tau);
    integrate(e);
  }
  hand_velocity(e);
  /* robosuite's MujocoEnv.step samples the observables inside the substep loop (_update_observables, after sim.step) and returns
     the cached values: the observation of step t is assembled BEFORE _post_action updates the task state, i.e. obs[9..14] carry
     traj_pt / running means / dFz of step t-1 -- exactly what reward() reads (ultrasound.py:525 before :528-546).  Pinned by the
     shipped artifacts: every (old_obs, old_reward) row reproduces its reward from its observation (tests/test_task_golden.py). */
  write_obs(e, obs);
  post_action_impl(ts, c->horizon, c->ignore_done, c->control_freq, c->early_termination, m->jnt_range, e->eef_pos, e->eef_quat,
                   e->hand_vel, e->cfrc[2], e->in_contact, e->qpos, reward, done);
  return 0;
}

/* Ultrasound._post_action (ultrasound.py:512-550) with reward (:230-269) and _check_terminated (:635-670); pure:
 * reads the post-physics measurements, updates the task record `ts` in place (timestep already incremented). */
void oracle_post_action(double* ts, int horizon, double control_freq, int early_termination, const double* jnt_range,
                        const double* eef_pos, const double* eef_quat_xyzw, const double* hand_vel, double fz, int in_contact,
                        const double* qpos7, double* reward, int* done) {
  post_action_impl(ts, horizon, 0, control_freq, early_termination, jnt_range, eef_pos, eef_quat_xyzw, hand_vel, fz, in_contact, qpos7,
                   reward, done);
}
static void post_action_impl(double* ts, int horizon, int ignore_done, double control_freq, int early_termination, const double* jnt_range,
                             const double* eef_pos, const double* eef_quat_xyzw, const double* hand_vel, double fz, int in_contact,
                             const double* qpos7, double* reward, int* done) {
  /* reward first, with the task state of the previous step (:525); the contact query latches has_touched_torso (:733) */
  if (in_contact) ts[USIM_TS_TOUCHED] = 1;
  double pe[2], oe;
  *reward = oracle_reward(eef_pos, eef_quat_xyzw, ts + USIM_TS_TRAJ_PT, ts[USIM_TS_VEL_MEAN], ts[USIM_TS_FZ_MEAN], ts[USIM_TS_DFZ],
                          in_contact, pe, &oe);
  ts[USIM_TS_POS_ERR] = pe[0]; ts[USIM_TS_POS_ERR + 1] = pe[1]; ts[USIM_TS_ORI_ERR] = oe;
  ts[USIM_TS_IN_CONTACT] = in_contact;
  double t = ts[USIM_TS_TIMESTEP];
  int dn = t >= horizon && !ignore_done; /* robosuite MujocoEnv._post_action */
  double u = t / (double)horizon + ts[USIM_TS_U0]; /* :528-532, two waypoints; klampt eval clamps ("halt") */
  u = u < 0 ? 0 : (u > 1 ? 1 : u);
  for (int k = 0; k < 3; k++) ts[USIM_TS_TRAJ_PT + k] = ts[USIM_TS_TRAJ_START + k] + u * (ts[USIM_TS_TRAJ_END + k] - ts[USIM_TS_TRAJ_START + k]);
  ts[USIM_TS_VEL_MEAN] += (norm3(hand_vel) - ts[USIM_TS_VEL_MEAN]) / t;     /* :538 */
  ts[USIM_TS_DFZ] = (fz - ts[USIM_TS_FZ_PREV]) / (1.0 / control_freq);      /* :542 */
  ts[USIM_TS_FZ_PREV] = fz;
  ts[USIM_TS_FZ_MEAN] = 0.1 * fz + 0.9 * ts[USIM_TS_FZ_MEAN];               /* :546 */
  if (early_termination) { /* :635-670 */
    int term = 0;
    if (qpos7)
      for (int j = 0; j < 7; j++) /* robosuite check_q_limits, tolerance 0.1 */
        if (!(jnt_range[2 * j] + 0.1 < qpos7[j] && qpos7[j] < jnt_range[2 * j + 1] - 0.1)) term = 1;
    if (sqrt(pe[0] * pe[0] + pe[1] * pe[1]) > 1.0) term = 1;
    if (in_contact && oe > 0.10) term = 1;
    if (ts[USIM_TS_TOUCHED] != 0 && !in_contact) term = 1;
    dn = dn || term;
  }
  ts[USIM_TS_DONE] = dn;
  *done = dn;
}

/* waypoint grid of get_trajectory (ultrasound.py:787-788,805-807): value of grid index i in [0,50) */
void oracle_grid_point2(double tx, double ty, double tz, double xr, double yr, double top, int ix, int iy, double* pt) {
  double x0 = -xr + tx + 0.03, x1 = xr + tx, y0 = -yr + ty, y1 = yr + ty;
  pt[0] = x0 + (x1 - x0) * (double)ix / 49.0;
  pt[1] = y0 + (y1 - y0) * (double)iy / 49.0;
  pt[2] = tz + top;
}
void oracle_grid_point(double tx, double ty, double tz, int ix, int iy, double* pt) { /* box torso constants */
  oracle_grid_point2(tx, ty, tz, 0.15, 0.09, 0.039, ix, iy, pt);
}

/* ------------------------------------------------------------------ state access / introspection */
void oracle_get_state(const oracle_env* e, double* qpos, double* qvel, double* warm, double* task) {
  if (qpos) memcpy(qpos, e->qpos, sizeof(double) * e->nq);
  if (qvel) memcpy(qvel, e->qvel, sizeof(double) * e->nv);
  if (warm) memcpy(warm, e->warm, sizeof(double) * e->nv);
  if (task) memcpy(task, e->ts, sizeof e->ts);
}
void oracle_set_state(oracle_env* e, const double* qpos, const double* qvel, const double* warm, const double* task) {
  if (qpos) memcpy(e->qpos, qpos, sizeof(double) * e->nq);
  if (qvel) memcpy(e->qvel, qvel, sizeof(double) * e->nv);
  if (warm) memcpy(e->warm, warm, sizeof(double) * e->nv);
  if (task) memcpy(e->ts, task, sizeof e->ts);
}
int oracle_ncon(const oracle_env* e) { return e->ncon; }
void oracle_contacts(const oracle_env* e, int* g1, int* g2, double* dist, double* pos, double* frame, double* force) {
  for (int i = 0; i < e->ncon; i++) {
    if (g1) g1[i] = e->con[i].geom1;
    if (g2) g2[i] = e->con[i].geom2;
    if (dist) dist[i] = e->con[i].dist;
    if (pos) memcpy(pos + 3 * i, e->con[i].pos, 3 * sizeof(double));
    if (frame) memcpy(frame + 9 * i, e->con[i].frame, 9 * sizeof(double));
    if (force) memcpy(force + 3 * i, e->con[i].force, 3 * sizeof(double));
  }
}
int oracle_nefc(const oracle_env* e) { return e->nefc; }
int oracle_solver_iter(const oracle_env* e) { return e->solver_iter; }
const double* oracle_qacc(const oracle_env* e) { return e->qacc; }
const double* oracle_qacc_smooth(const oracle_env* e) { return e->a0; }
const double* oracle_M(const oracle_env* e) { return e->M; }
const double* oracle_bias(const oracle_env* e) { return e->bias; }
const double* oracle_tau(const oracle_env* e) { return e->tau; }
void oracle_diag(const oracle_env* e, double* d) {
  for (int k = 0; k < 3; k++) { d[k] = e->cfrc[k]; d[3 + k] = e->ft_torque[k]; d[6 + k] = e->eef_pos[k]; }
  for (int k = 0; k < 4; k++) d[9 + k] = e->eef_quat[k];
  for (int k = 0; k < 7; k++) d[13 + k] = e->tau[k];
  d[20] = e->solver_iter; d[21] = e->solver_grad; d[22] = e->ncon; d[23] = e->nefc;
  for (int k = 24; k < USIM_DIAG_DIM; k++) d[k] = 0;
}
void oracle_eef(const oracle_env* e, double* J, double* pos, double* mat) {
  if (J) memcpy(J, e->Jsite, sizeof e->Jsite);
  if (pos) memcpy(pos, e->eef_pos, sizeof e->eef_pos);
  if (mat) memcpy(mat, e->eef_mat, sizeof e->eef_mat);
}
void oracle_controller(oracle_env* e, const double* action, double* tau) {
  forward_posvel(e);
  set_goal(e, action);
  controller(e, action, tau);
}

typedef struct {
  oracle_env** envs;
  int n, steps, adim, auto_reset, tid, nthreads;
  const double* actions;
  long total;
  double rs;
} rollout_job;

static void* rollout_worker(void* arg) {
  rollout_job* j = (rollout_job*)arg;
  for (int i = j->tid; i < j->n; i += j->nthreads) {
    double obs[USIM_OBS_DIM], rew;
    int done;
    for (int s = 0; s < j->steps; s++) {
      if (j->envs[i]->ts[USIM_TS_DONE] != 0) {
        if (!j->auto_reset) break;
        oracle_reset(j->envs[i], obs);
      }
      oracle_step(j->envs[i], j->actions + ((size_t)s * j->n + i) * j->adim, obs, &rew, &done);
      j->rs += rew;
      j->total++;
    }
  }
  return NULL;
}

long oracle_rollout(oracle_env** envs, int n, const double* actions, int steps, int adim, int auto_reset, int threads,
                    double* reward_sum) {
  if (threads < 1) threads = 1;
  if (threads > n) threads = n;
  if (threads > 256) threads = 256;
  pthread_t th[256];
  rollout_job jobs[256];
  for (int t = 0; t < threads; t++) {
    rollout_job j = {envs, n, steps, adim, auto_reset, t, threads, actions, 0, 0.0};
    jobs[t] = j;
    pthread_create(&th[t], NULL, rollout_worker, &jobs[t]);
  }
  long total = 0;
  double rs = 0;
  for (int t = 0; t < threads; t++) { pthread_join(th[t], NULL); total += jobs[t].total; rs += jobs[t].rs; }
  if (reward_sum) *reward_sum = rs;
  return total;
}

/* one env step of n envs over `threads` host threads, outputs per env (parity tests: the GPU batch is compared step by step).
 * rc[i] = oracle_step's return (-1: env i was already done, its outputs are left untouched) */
typedef struct {
  oracle_env** envs;
  int n, adim, tid, nthreads;
  const double* actions;
  double *obs, *rew;
  int *done, *rc;
} stepb_job;
static void* stepb_worker(void* arg) {
  stepb_job* j = (stepb_job*)arg;
  for (int i = j->tid; i < j->n; i += j->nthreads)
    j->rc[i] = oracle_step(j->envs[i], j->actions + (size_t)i * j->adim, j->obs + (size_t)i * USIM_OBS_DIM, j->rew + i, j->done + i);
  return NULL;
}
void oracle_step_batch(oracle_env** envs, int n, const double* actions, int adim, int threads, double* obs, double* rew, int* done,
                       int* rc) {
  if (threads < 1) threads = 1;
  if (threads > n) threads = n;
  if (threads > 256) threads = 256;
  pthread_t th[256];
  stepb_job jobs[256];
  for (int t = 0; t < threads; t++) {
    stepb_job j = {envs, n, adim, t, threads, actions, obs, rew, done, rc};
    jobs[t] = j;
    pthread_create(&th[t], NULL, stepb_worker, &jobs[t]);
  }
  for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
}
