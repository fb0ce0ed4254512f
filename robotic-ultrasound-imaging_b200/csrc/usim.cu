// usim.cu — C ABI (include/usim.h) over the sm_100a kernels.  Owns the per-env state in HBM.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "arm.cuh"
#include "arm_warp.cuh"
#include "common.cuh"
#include "soft.cuh"

#ifndef PREP_GRID
#define PREP_GRID 296 // CTAs of the forward-only solve launch that prepares reset states (walks the request list)
#endif
#ifndef ARM_BLOCK
#define ARM_BLOCK 32 // threads per CTA of the thread-per-env arm kernel (latency bound: 128 one-warp CTAs on 128 SMs; measured 21.7 us vs 25.0 us for 64)
#endif

static thread_local std::string g_err;
static int fail(const std::string& m) {
  g_err = m;
  return -1;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(e_));        \
  } while (0)

struct usim_handle {
  int device = 0, n = 0, nq = 0, nv = 0, adim = 6, soft = 0, substeps = 1, narm = 7;
  DevModel hm;
  // per-env state, env-major rows (one warp owns one row -> one coalesced 128-B aligned stream)
  float *qpos = nullptr, *qvel = nullptr, *warm = nullptr, *task = nullptr, *armbuf = nullptr, *diag = nullptr;
  int *ncon = nullptr, *geom1 = nullptr, *geom2 = nullptr;
  float* cdist = nullptr;
  // contact record (usim_set_contact_record): [n][DEV_MAXC][CREC_DIM], allocated on the first enable; complete once every env has
  // been through a recorded launch (a step, or a reset without mask)
  float* crec = nullptr;
  bool crec_on = false, crec_complete = false;
  int* counters = nullptr; // [0] env steps that produced a non-finite solution (episode force-ended), [1] env steps whose contact list overflowed
  // model tables
  float4 *ax4 = nullptr, *ps4 = nullptr; // (axis, dof_invweight0), (rest position, body_invweight0)
  int4* nb4 = nullptr;                   // packed neighbour / pair stencil
  int2* eq_pairs = nullptr;
  // staging for the host-buffer path: page-locked buffers, the device aliases of the output ones, and the actions on the device
  float *h_act = nullptr, *h_obs = nullptr, *h_rew = nullptr, *h_tobs = nullptr;
  uint8_t* h_done = nullptr;
  float *map_obs = nullptr, *map_rew = nullptr, *map_tobs = nullptr;
  uint8_t* map_done = nullptr;
  float* d_act = nullptr;
  // launch order of the solve kernel (longest solve first): bins filled by launch T, flattened by the arm kernel of launch T + 1
  int *bin_cnt = nullptr, *bin_items = nullptr, *order = nullptr; // [2][NBIN], [2][NBIN][n], [n]
  int* queue = nullptr;  // work queue of a persistent step launch (next launch slot)
  unsigned long long* trace = nullptr;  // developer trace of the step launches (USIM_TRACE=<file>): [n][3] = start ns, end ns, SM id
  std::string trace_path;
  int step_grid = 0;     // CTAs of a step launch: every resident slot of the device once (0: one CTA per env)
  int64_t solve_tick = 0;
  // reset pipeline: two prepared reset states per env (slot k holds an episode number of parity k), made on a side stream
  float *slot_qpos = nullptr, *slot_task = nullptr, *slot_obs = nullptr, *prep_armbuf = nullptr;
  // usim_forward, allocated on its first call: arm record ([n][ARMBUF]; the live one is left alone) and padded qacc rows ([n][QPAD])
  float *fwd_armbuf = nullptr, *fwd_qacc = nullptr;
  int *req_list = nullptr, *req_cnt = nullptr; // [2][2 * 3n], [2]: request lists, double buffered by producer tick
  int64_t prod_tick = 0;
  bool slots_init = false;
  cudaStream_t prep_stream = nullptr;
  cudaEvent_t ev_prod = nullptr, ev_prep[2] = {nullptr, nullptr};
  bool ev_prep_valid[2] = {false, false};
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev_state = nullptr; // recorded on the caller's stream after every state-mutating call: usim_step_host waits on it
  bool ev_state_valid = false, timing = false, arm_thread = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
  int64_t launches = 0, timed_launches = 0;
  double timed_ms = 0.0;
};

static usim_handle* g_active = nullptr; // handle whose DevModel currently sits in the constant block

const char* usim_last_error(void) { return g_err.c_str(); }
int usim_abi_version(void) { return USIM_ABI_VERSION; }
size_t usim_sizeof_model(void) { return sizeof(usim_model); }
size_t usim_sizeof_config(void) { return sizeof(usim_config); }

template <typename T>
static cudaError_t upload(T** dst, const std::vector<T>& v) {
  cudaError_t e = cudaMalloc((void**)dst, std::max<size_t>(v.size(), 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  if (!v.empty()) e = cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
  return e;
}

int usim_create(const usim_model* m, const usim_config* c, int device, usim_handle** out) {
  if (!m || !c || !out) return fail("usim_create: null argument");
  if (c->abi_version != USIM_ABI_VERSION) return fail("usim_create: ABI version mismatch");
  if (c->num_envs <= 0) return fail("usim_create: num_envs must be positive");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("usim_create: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail("usim_create: bad device index");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail("usim_create: kernels are built for sm_100a only; found sm_" + std::to_string(prop.major * 10 + prop.minor));
  if (m->soft && (m->npart > NPART_MAX || m->npair > NPAIR_MAX)) return fail("usim_create: composite larger than the compiled limits");
  if (m->narm != 7 && m->narm != 6) return fail("usim_create: the arm kernels are compiled for 7 (Panda) or 6 (UR5e) joints");
  // physics substeps per control step: int(control_timestep / model_timestep) [robosuite MujocoEnv.step]; 1 at rl_config.yaml's
  // 500 Hz, 25 at the env's own default of 20 Hz (ultrasound.py:119)
  if (!(c->control_freq > 0.0)) return fail("usim_create: control_freq must be positive");
  int substeps = (int)((1.0 / c->control_freq) / m->timestep + 1e-9);
  if (substeps < 1) return fail("usim_create: control_freq above 1/timestep (less than one physics step per control step)");

  usim_handle* h = new usim_handle();
  h->device = device; h->n = c->num_envs; h->nq = m->nq; h->nv = m->nv; h->soft = m->soft; h->substeps = substeps; h->narm = m->narm;
  h->adim = c->impedance_mode == USIM_MODE_VARIABLE_Z ? 7 : 6;
  DevModel& d = h->hm;
  memset(&d, 0, sizeof d);
  for (int j = 0; j < 7; j++) {
    const double* L = m->arm_link + 22 * j;
    for (int k = 0; k < 3; k++) { d.link_pos[j][k] = (float)L[k]; d.link_com[j][k] = (float)L[12 + k]; }
    for (int k = 0; k < 9; k++) d.link_R[j][k] = (float)L[3 + k];
    d.link_mass[j] = (float)L[15];
    for (int k = 0; k < 6; k++) d.link_I[j][k] = (float)L[16 + k];
    d.jnt_lo[j] = (float)m->jnt_range[2 * j]; d.jnt_hi[j] = (float)m->jnt_range[2 * j + 1];
    d.ctrl[j] = (float)m->ctrl_range[j]; d.init_qpos[j] = (float)m->init_qpos[j];
    d.iw_arm[j] = (float)m->dof_invweight0[j];
  }
  for (int k = 0; k < 34; k++) d.tool[k] = (float)m->arm_tool[k];
  d.arm_damp = (float)m->dof_damping[0];
  d.h = (float)m->timestep; d.impratio = (float)m->impratio;
  for (int k = 0; k < 3; k++) d.g[k] = (float)m->gravity[k];
  for (int k = 0; k < 2; k++) { d.solref[k] = (float)m->solref[k]; d.solref_smooth[k] = (float)m->solref_smooth[k]; }
  for (int k = 0; k < 5; k++) d.solimp[k] = (float)m->solimp[k];
  d.table_z = (float)m->table_top_z; d.table_half = (float)m->table_half_xy;
  d.fr_table_probe = (float)fmax(m->table_friction, m->probe_friction);
  d.fr_table_part = (float)fmax(m->table_friction, m->particle_friction);
  d.fr_probe_part = (float)fmax(m->probe_friction, m->particle_friction);
  d.probe_r = (float)m->probe_radius; d.cap_r = (float)m->cap_radius;
  d.iw_probe = (float)m->body_invweight0[2 * m->probe_body]; d.iw_table = 0.f;
  d.top_offset = (float)m->top_torso_offset; d.traj_xr = (float)m->traj_x_range; d.traj_yr = (float)m->traj_y_range;
  d.soft = m->soft; d.npart = m->soft ? m->npart : 0; d.npair = m->soft ? m->npair : 0;
  std::vector<float> ppos, paxis, iwd, iwb;
  std::vector<int> nbr, pairs;
  std::vector<short> nbrp;
  if (m->soft) {
    int np = m->npart;
    d.tendon_iw = (float)m->tendon_invweight0;
    d.free_damp = (float)m->dof_damping[7];
    d.part_mass = (float)m->body_mass[m->part_body0];
    d.center_mass = (float)m->body_mass[m->torso_body];
    for (int k = 0; k < 7; k++) d.torso_qpos0[k] = (float)m->qpos0[7 + k];
    // capsule half length from the two segment ends of particle 0
    double dd = 0;
    for (int k = 0; k < 3; k++) { double t = m->part_seg_outer[k] - m->part_seg_inner[k]; dd += t * t; }
    d.cap_hl = (float)(0.5 * sqrt(dd));
    // constant rotational inertia: sum of the body-frame inertias of every torso body about its own COM
    double rot[6] = {0, 0, 0, 0, 0, 0};
    for (int b = m->torso_body; b < m->torso_body + 1 + np; b++) {
      const double* I = m->body_inertia + 9 * b;
      rot[0] += I[0]; rot[1] += I[4]; rot[2] += I[8]; rot[3] += I[1]; rot[4] += I[2]; rot[5] += I[5];
    }
    for (int k = 0; k < 6; k++) d.rot_I[k] = (float)rot[k];
    for (int i = 0; i < np; i++) {
      for (int k = 0; k < 3; k++) { ppos.push_back((float)m->part_pos[3 * i + k]); paxis.push_back((float)m->part_axis[3 * i + k]); }
      iwd.push_back((float)m->dof_invweight0[13 + i]);
      iwb.push_back((float)m->body_invweight0[2 * (m->part_body0 + i)]);
      for (int k = 0; k < 6; k++) nbr.push_back(m->part_nbr[6 * i + k]);
    }
    nbrp.assign((size_t)np * 6, -1);
    for (int p = 0; p < m->npair; p++) {
      int a = m->eq_pairs[2 * p], b = m->eq_pairs[2 * p + 1];
      pairs.push_back(a); pairs.push_back(b);
      for (int side = 0; side < 2; side++) {
        int i = side ? b : a, j = side ? a : b;
        for (int k = 0; k < 6; k++)
          if (nbr[6 * i + k] == j) nbrp[6 * i + k] = (short)p;
      }
    }
  }
  d.mode = c->impedance_mode; d.horizon = c->horizon; d.early_term = c->early_termination; d.ignore_done = c->ignore_done;
  d.solref_rand = c->solref_randomization; d.pos_rand = c->probe_pos_randomization; d.det_traj = c->deterministic_trajectory;
  d.uncouple = c->uncouple_pos_ori; d.iters = c->solver_iterations > 0 ? c->solver_iterations : 40;
  d.max_rebuilds = c->precond_rebuilds > 0 ? c->precond_rebuilds : 8; // preconditioner rebuilds per solve when contact zones change
  d.adim = h->adim; d.env_off = c->env_id_offset; d.nq = m->nq; d.nv = m->nv;
  d.seed_lo = (unsigned)(c->seed & 0xffffffffu); d.seed_hi = (unsigned)(c->seed >> 32);
  d.ctrl_freq = (float)c->control_freq;
  for (int k = 0; k < 6; k++) { d.kp[k] = (float)c->kp[k]; d.dr[k] = (float)c->damping_ratio[k]; d.out_max[k] = (float)c->output_max[k]; d.out_min[k] = (float)c->output_min[k]; }
  d.in_max = (float)c->input_max; d.in_min = (float)c->input_min;
  d.kp_lim[0] = (float)c->kp_limits[0]; d.kp_lim[1] = (float)c->kp_limits[1];
  d.kp_in_max = (float)c->kp_input_max; d.kp_in_min = (float)c->kp_input_min;
  d.tol = c->solver_tolerance > 0 ? (float)c->solver_tolerance : 1e-6f;
  for (int k = 0; k < 3; k++) d.eef_bias[k] = (float)c->reset_eef_bias[k];

#define CKH(call)                                                                                                  \
  do {                                                                                                             \
    cudaError_t e_ = (call);                                                                                       \
    if (e_ != cudaSuccess) { g_err = std::string(#call) + ": " + cudaGetErrorString(e_); usim_destroy(h); return -1; } \
  } while (0)
  size_t N = (size_t)h->n;
  CKH(cudaMalloc((void**)&h->qpos, N * QPAD * sizeof(float)));
  CKH(cudaMalloc((void**)&h->qvel, N * QPAD * sizeof(float)));
  CKH(cudaMalloc((void**)&h->warm, N * QPAD * sizeof(float)));
  CKH(cudaMalloc((void**)&h->task, N * USIM_TASK_DIM * sizeof(float)));
  CKH(cudaMalloc((void**)&h->armbuf, N * ARMBUF * sizeof(float)));
  CKH(cudaMalloc((void**)&h->diag, N * USIM_DIAG_DIM * sizeof(float)));
  CKH(cudaMalloc((void**)&h->ncon, N * sizeof(int)));
  CKH(cudaMalloc((void**)&h->geom1, N * DEV_MAXC * sizeof(int)));
  CKH(cudaMalloc((void**)&h->geom2, N * DEV_MAXC * sizeof(int)));
  CKH(cudaMalloc((void**)&h->cdist, N * DEV_MAXC * sizeof(float)));
  CKH(cudaMemset(h->qpos, 0, N * QPAD * sizeof(float)));
  CKH(cudaMemset(h->qvel, 0, N * QPAD * sizeof(float)));
  CKH(cudaMemset(h->warm, 0, N * QPAD * sizeof(float)));
  CKH(cudaMemset(h->armbuf, 0, N * ARMBUF * sizeof(float)));
  CKH(cudaMemset(h->diag, 0, N * USIM_DIAG_DIM * sizeof(float)));
  CKH(cudaMemset(h->ncon, 0, N * sizeof(int)));
  CKH(cudaMalloc((void**)&h->counters, 2 * sizeof(int)));
  CKH(cudaMemset(h->counters, 0, 2 * sizeof(int)));
  { // task records: everything zero except DONE = 1 (must reset before stepping)
    std::vector<float> t(N * USIM_TASK_DIM, 0.f);
    for (size_t e = 0; e < N; e++) t[e * USIM_TASK_DIM + USIM_TS_DONE] = 1.f;
    CKH(cudaMemcpy(h->task, t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  {
    const int np = d.npart;
    std::vector<float4> a4(np), p4(np);
    std::vector<int4> n4(np);
    std::vector<int2> p2(d.npair);
    for (int i = 0; i < np; i++) {
      a4[i] = make_float4(paxis[3 * i], paxis[3 * i + 1], paxis[3 * i + 2], iwd[i]);
      p4[i] = make_float4(ppos[3 * i], ppos[3 * i + 1], ppos[3 * i + 2], iwb[i]);
      int e[4], cnt = 0;
      for (int k = 0; k < 6; k++)
        if (nbr[6 * i + k] >= 0) {
          if (cnt == 4 || nbrp[6 * i + k] < 0) { g_err = "usim_create: the composite's pair stencil has more than 4 neighbours per element (compiled limit)"; usim_destroy(h); return -1; }
          const int pr = nbrp[6 * i + k];
          e[cnt++] = (pr << 16) | (pairs[2 * pr + 1] == i ? 0x8000 : 0) | nbr[6 * i + k]; // bit 15: this slider is the pair's SECOND element
        }
      for (; cnt < 4; cnt++) e[cnt] = (d.npair << 16) | i;
      n4[i] = make_int4(e[0], e[1], e[2], e[3]);
    }
    for (int p = 0; p < d.npair; p++) p2[p] = make_int2(pairs[2 * p], pairs[2 * p + 1]);
    CKH(upload(&h->ax4, a4)); CKH(upload(&h->ps4, p4)); CKH(upload(&h->nb4, n4)); CKH(upload(&h->eq_pairs, p2));
  }
  CKH(cudaMallocHost((void**)&h->h_act, N * USIM_MAX_ACTION * sizeof(float)));
  CKH(cudaMallocHost((void**)&h->h_obs, N * USIM_OBS_DIM * sizeof(float)));
  CKH(cudaMallocHost((void**)&h->h_tobs, N * USIM_OBS_DIM * sizeof(float)));
  CKH(cudaMallocHost((void**)&h->h_rew, N * sizeof(float)));
  CKH(cudaMallocHost((void**)&h->h_done, N));
  // the solve kernel writes the output staging buffers through these (UVA maps every page-locked allocation)
  CKH(cudaHostGetDevicePointer((void**)&h->map_obs, h->h_obs, 0));
  CKH(cudaHostGetDevicePointer((void**)&h->map_tobs, h->h_tobs, 0));
  CKH(cudaHostGetDevicePointer((void**)&h->map_rew, h->h_rew, 0));
  CKH(cudaHostGetDevicePointer((void**)&h->map_done, h->h_done, 0));
  CKH(cudaMalloc((void**)&h->d_act, N * USIM_MAX_ACTION * sizeof(float)));
  CKH(cudaEventCreateWithFlags(&h->ev_state, cudaEventDisableTiming));
  CKH(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  {
    // launch-order bins: before the first launch every env sits in bin 0 of buffer 1 (identity order)
    CKH(cudaMalloc((void**)&h->bin_cnt, 2 * NBIN * sizeof(int)));
    CKH(cudaMalloc((void**)&h->bin_items, 2 * (size_t)NBIN * N * sizeof(int)));
    CKH(cudaMalloc((void**)&h->order, N * sizeof(int)));
    CKH(cudaMalloc((void**)&h->queue, sizeof(int)));
    CKH(cudaMemset(h->queue, 0, sizeof(int)));
    std::vector<int> cnt(2 * NBIN, 0), ident(N);
    cnt[NBIN] = (int)N;
    for (size_t e = 0; e < N; e++) ident[e] = (int)e;
    CKH(cudaMemcpy(h->bin_cnt, cnt.data(), cnt.size() * sizeof(int), cudaMemcpyHostToDevice));
    CKH(cudaMemcpy(h->bin_items + (size_t)NBIN * N, ident.data(), N * sizeof(int), cudaMemcpyHostToDevice));
    CKH(cudaMemcpy(h->order, ident.data(), N * sizeof(int), cudaMemcpyHostToDevice));
    // reset slots + request lists (at most n requests per producer launch, 2n at the first reset)
    CKH(cudaMalloc((void**)&h->slot_qpos, 2 * N * QPAD * sizeof(float)));
    CKH(cudaMalloc((void**)&h->slot_task, 2 * N * USIM_TASK_DIM * sizeof(float)));
    CKH(cudaMalloc((void**)&h->slot_obs, 2 * N * SLOT_OBS * sizeof(float)));
    CKH(cudaMalloc((void**)&h->prep_armbuf, 3 * N * ARMBUF * sizeof(float)));
    CKH(cudaMalloc((void**)&h->req_list, 2 * 2 * 3 * N * sizeof(int)));
    CKH(cudaMalloc((void**)&h->req_cnt, 2 * sizeof(int)));
    CKH(cudaMemset(h->slot_qpos, 0, 2 * N * QPAD * sizeof(float)));
    CKH(cudaMemset(h->slot_task, 0, 2 * N * USIM_TASK_DIM * sizeof(float)));
    CKH(cudaMemset(h->slot_obs, 0, 2 * N * SLOT_OBS * sizeof(float)));
    CKH(cudaMemset(h->req_cnt, 0, 2 * sizeof(int)));
    int lo = 0, hi = 0;
    CKH(cudaDeviceGetStreamPriorityRange(&lo, &hi)); // (hi = numerically lowest = greatest priority)
    CKH(cudaStreamCreateWithPriority(&h->prep_stream, cudaStreamNonBlocking, hi));
    CKH(cudaEventCreateWithFlags(&h->ev_prod, cudaEventDisableTiming));
    CKH(cudaEventCreateWithFlags(&h->ev_prep[0], cudaEventDisableTiming));
    CKH(cudaEventCreateWithFlags(&h->ev_prep[1], cudaEventDisableTiming));
  }
  if (const char* at = getenv("USIM_ARM_THREAD")) h->arm_thread = atoi(at) != 0;
  if (const char* tp = getenv("USIM_TRACE")) { // developer knob: the last step launch's per-env timeline is written to this file at destroy
    h->trace_path = tp;
    CKH(cudaMalloc((void**)&h->trace, (size_t)h->n * 3 * sizeof(unsigned long long)));
    CKH(cudaMemset(h->trace, 0, (size_t)h->n * 3 * sizeof(unsigned long long)));
  }
  if (const char* pg = getenv("USIM_PERSISTENT")) { // developer knob: persistent step launch, one CTA per resident slot
    int per_sm = 0;
    if (atoi(pg) != 0 && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, solve_kernel, NT, sizeof(WS)) == cudaSuccess && per_sm > 0)
      h->step_grid = std::min(h->n, per_sm * prop.multiProcessorCount);
  }
  CKH(cudaFuncSetAttribute(solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WS)));
  CKH(cudaDeviceSynchronize());
  *out = h;
  return 0;
}

int usim_destroy(usim_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (g_active == h) g_active = nullptr;
  if (h->trace) {
    std::vector<unsigned long long> t((size_t)h->n * 3);
    if (cudaMemcpy(t.data(), h->trace, t.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost) == cudaSuccess) {
      if (FILE* f = fopen(h->trace_path.c_str(), "wb")) { fwrite(t.data(), sizeof(unsigned long long), t.size(), f); fclose(f); }
    }
    cudaFree(h->trace);
  }
  for (auto& p : h->pending) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
  void* dev[] = {h->counters, h->qpos, h->qvel, h->warm, h->task, h->armbuf, h->diag, h->ncon, h->geom1, h->geom2, h->cdist, h->crec, h->ax4,
                 h->ps4, h->nb4, h->eq_pairs, h->d_act, h->bin_cnt, h->bin_items, h->order, h->queue, h->slot_qpos, h->slot_task, h->slot_obs, h->prep_armbuf,
                 h->fwd_armbuf, h->fwd_qacc, h->req_list, h->req_cnt};
  for (void* p : dev) if (p) cudaFree(p);
  void* host[] = {h->h_act, h->h_obs, h->h_tobs, h->h_rew, h->h_done};
  for (void* p : host) if (p) cudaFreeHost(p);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->ev_state) cudaEventDestroy(h->ev_state);
  if (h->prep_stream) cudaStreamDestroy(h->prep_stream);
  for (cudaEvent_t e : {h->ev_prod, h->ev_prep[0], h->ev_prep[1]}) if (e) cudaEventDestroy(e);
  delete h;
  return 0;
}

static PartTables tables(const usim_handle* h) { return PartTables{h->ax4, h->ps4, h->nb4}; }

// launches: the DevModel symbol is per-process; re-upload if another handle changed it
static int activate(usim_handle* h) {
  CK(cudaSetDevice(h->device));
  if (g_active != h) {
    // the contract is one handle per (process, GPU); switching handles is supported but drains the device first,
    // because kernels of the previous handle may still be reading the constant block
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyToSymbol(dm, &h->hm, sizeof(DevModel)));
    g_active = h;
  }
  return 0;
}

// state-mutating calls on the caller's stream end with this: the host-buffer entry point (private stream) orders itself after it
static int mark_state(usim_handle* h, cudaStream_t s) {
  CK(cudaEventRecord(h->ev_state, s));
  h->ev_state_valid = true;
  return 0;
}

// the arm / reset kernels are compiled per joint count (arm.cuh NJ)
// (arm_thread: developer knob USIM_ARM_THREAD=1, the thread-per-env kernel of round 1 -- kept for A/B measurements and as a second opinion)
#define ARM_LAUNCH(h, stream, ...)                                                                                        \
  do {                                                                                                                    \
    const int n_ = (h)->n;                                                                                                \
    if ((h)->arm_thread) {                                                                                                \
      if ((h)->narm == 7) arm_kernel<7><<<(n_ + ARM_BLOCK - 1) / ARM_BLOCK, ARM_BLOCK, 0, stream>>>(__VA_ARGS__);         \
      else arm_kernel<6><<<(n_ + ARM_BLOCK - 1) / ARM_BLOCK, ARM_BLOCK, 0, stream>>>(__VA_ARGS__);                        \
    } else {                                                                                                              \
      const int epb_ = ARMW_BLOCK / GW;                                                                                   \
      if ((h)->narm == 7) arm_kernel_w<7><<<(n_ + epb_ - 1) / epb_, ARMW_BLOCK, 0, stream>>>(__VA_ARGS__);                \
      else arm_kernel_w<6><<<(n_ + epb_ - 1) / epb_, ARMW_BLOCK, 0, stream>>>(__VA_ARGS__);                               \
    }                                                                                                                     \
  } while (0)
#define RESET_LAUNCH(h, grid, block, stream, ...)                                                 \
  do {                                                                                            \
    if ((h)->narm == 7) reset_kernel<7><<<grid, block, 0, stream>>>(__VA_ARGS__);                 \
    else reset_kernel<6><<<grid, block, 0, stream>>>(__VA_ARGS__);                                \
  } while (0)

static SolveArgs base_args(usim_handle* h, int mode) {
  SolveArgs a;
  memset(&a, 0, sizeof a);
  a.n = h->n; a.mode = mode;
  a.qpos = h->qpos; a.qvel = h->qvel; a.warm = h->warm; a.task = h->task; a.armbuf = h->armbuf;
  a.pt = tables(h); a.eq_pairs = h->eq_pairs;
  a.diag = h->diag; a.ncon_out = h->ncon; a.geom1_out = h->geom1; a.geom2_out = h->geom2; a.dist_out = h->cdist;
  a.counters = h->counters;
  a.crec_out = h->crec_on && mode != 2 ? h->crec : nullptr; // an intermediate substep's contacts are superseded by the last one's
  a.slot_qpos = h->slot_qpos; a.slot_task = h->slot_task; a.slot_obs = h->slot_obs;
  return a;
}

// Producer launches (the last solve launch of an auto-reset step, an explicit reset) append prepare requests to list (tick & 1).
// Before one starts, the prepare run that last worked through that list (two producers ago) must have finished -- it always has,
// in practice: it had a whole step to do so.  This also orders every slot write before the step that may read it.
static int producer_begin(usim_handle* h, cudaStream_t s) {
  const int b = (int)(h->prod_tick & 1);
  if (h->ev_prep_valid[b]) CK(cudaStreamWaitEvent(s, h->ev_prep[b], 0));
  return 0;
}
// After the producer: work through its request list on the side stream (reset kernel in prepare mode, forward-only solve on the
// slots), concurrently with whatever the caller's stream does next.
static int producer_end(usim_handle* h, cudaStream_t s) {
  const int b = (int)(h->prod_tick & 1), n = h->n;
  int* list = h->req_list + (size_t)b * 2 * 3 * n;
  int* cnt = h->req_cnt + b;
  CK(cudaEventRecord(h->ev_prod, s));
  CK(cudaStreamWaitEvent(h->prep_stream, h->ev_prod, 0));
  RESET_LAUNCH(h, 64, 32, h->prep_stream, n, nullptr, h->slot_qpos, nullptr, nullptr, h->slot_task, h->prep_armbuf, list, cnt, nullptr, nullptr);
  SolveArgs a = base_args(h, 1);
  a.prep = 1; a.armbuf = h->prep_armbuf; a.prep_items = list; a.prep_n = cnt;
  a.diag = nullptr; a.ncon_out = nullptr; a.geom1_out = nullptr; a.geom2_out = nullptr; a.dist_out = nullptr; a.crec_out = nullptr;
  solve_kernel<<<PREP_GRID, NT, sizeof(WS), h->prep_stream>>>(a);
  CK(cudaMemsetAsync(cnt, 0, sizeof(int), h->prep_stream));
  CK(cudaEventRecord(h->ev_prep[b], h->prep_stream));
  h->ev_prep_valid[b] = true;
  h->launches += 2;
  h->prod_tick += 1;
  CK(cudaGetLastError());
  return 0;
}

// A producer of its own that fills both slots of every env from its live episode counter (fill_requests_kernel).  Stream s then
// waits for the prepare run: the very next step may end an episode and take over either slot, whereas producer_begin orders a step
// only after the slots filled two producers before it.
static int prepare_slots(usim_handle* h, cudaStream_t s) {
  const int b = (int)(h->prod_tick & 1), n = h->n;
  if (producer_begin(h, s)) return -1;
  fill_requests_kernel<<<(n + 127) / 128, 128, 0, s>>>(n, h->task, h->req_list + (size_t)b * 2 * 3 * n, h->req_cnt + b);
  h->launches += 1;
  if (producer_end(h, s)) return -1;
  CK(cudaStreamWaitEvent(s, h->ev_prep[b], 0));
  return 0;
}

// One control step: int(control_timestep / timestep) physics substeps of (arm kernel, solve kernel); the OSC goal is set on the
// first substep, the task epilogue -- and, with auto_reset, the hand-over to a prepared reset state -- runs in the last solve launch
// [robosuite MujocoEnv.step].
static int launch_step(usim_handle* h, const float* act, float* obs, float* rew, uint8_t* done, float* tobs, int auto_reset, cudaStream_t s) {
  const int n = h->n, nsub = h->substeps;
  for (int sub = 0; sub < nsub; sub++) {
    const bool last = sub == nsub - 1;
    const int b = (int)(h->solve_tick & 1); // this launch files into bins b; its order comes from bins 1 - b
    ARM_LAUNCH(h, s, n, h->qpos, h->qvel, act, h->task, h->armbuf, sub == 0 ? done : nullptr,
               sub == 0, NBIN, h->bin_cnt + (1 - b) * NBIN, h->bin_items + (size_t)(1 - b) * NBIN * n, h->bin_cnt + b * NBIN, h->order,
               h->step_grid ? h->queue : nullptr);
    SolveArgs a = base_args(h, last ? 0 : 2);
    a.obs = obs; a.rew = rew; a.done = done; a.tobs = tobs;
    a.order = h->order; a.bin_cnt = h->bin_cnt + b * NBIN; a.bin_items = h->bin_items + (size_t)b * NBIN * n;
    a.queue = h->step_grid ? h->queue : nullptr;
    a.trace = h->trace;
    if (last && auto_reset) {
      if (producer_begin(h, s)) return -1;
      a.auto_reset = 1;
      a.req_list = h->req_list + (size_t)(h->prod_tick & 1) * 2 * 3 * n; a.req_cnt = h->req_cnt + (h->prod_tick & 1);
    }
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool timed = h->timing && h->pending.size() < 4096; // bounded: the caller drains with usim_kernel_time
    if (timed) {
      CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
      CK(cudaEventRecord(e0, s));
    }
    solve_kernel<<<h->step_grid ? h->step_grid : n, NT, sizeof(WS), s>>>(a);
    if (timed) {
      CK(cudaEventRecord(e1, s));
      h->pending.emplace_back(e0, e1);
    }
    h->launches += 2;
    h->solve_tick += 1;
    if (last && auto_reset && producer_end(h, s)) return -1;
  }
  if (h->crec_on) h->crec_complete = true;
  CK(cudaGetLastError());
  return 0;
}

int usim_reset(usim_handle* h, const uint8_t* mask_dev, float* obs_dev, void* stream) {
  if (!h) return fail("usim_reset: null handle");
  if (activate(h)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const int n = h->n;
  const bool first = !h->slots_init;
  int *list = nullptr, *cnt = nullptr;
  if (!first) { // the live reset of an env with counter E files a request for episode E + 2 (the slot of E is stale from here on)
    if (producer_begin(h, s)) return -1;
    list = h->req_list + (size_t)(h->prod_tick & 1) * 2 * 3 * n;
    cnt = h->req_cnt + (h->prod_tick & 1);
  }
  // the reset itself, in place and in stream order: reset kernel (live mode) + forward-only solve on the live state
  RESET_LAUNCH(h, (n + 31) / 32, 32, s, n, mask_dev, h->qpos, h->qvel, h->warm, h->task, h->armbuf, nullptr, nullptr, list, cnt);
  SolveArgs a = base_args(h, 1);
  a.mask = mask_dev; a.obs = obs_dev;
  solve_kernel<<<n, NT, sizeof(WS), s>>>(a);
  h->launches += 2;
  CK(cudaGetLastError());
  if (h->crec_on && !mask_dev) h->crec_complete = true;
  if (first) { // nothing prepared yet: both slots of every env, from the counters this reset left
    h->slots_init = true;
    if (prepare_slots(h, s)) return -1;
  } else if (producer_end(h, s)) {
    return -1;
  }
  return mark_state(h, s);
}

// padded qacc rows of usim_forward -> the caller's dense [n][nv] array, rows of the selected envs only
__global__ void qacc_rows_kernel(int n, int nv, const uint8_t* __restrict__ mask, const float* __restrict__ src, float* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * nv) return;
  const int e = i / nv, k = i - e * nv;
  if (!mask || mask[e]) dst[i] = src[(size_t)e * QPAD + k];
}

// mj_forward at the live state: the arm pass into the forward buffer, then the solve kernel in forward mode (mode 1 as after a
// reset, but warm-started from the live qacc_warmstart, the task record read and never written, no launch-order bins, no counters)
int usim_forward(usim_handle* h, const uint8_t* mask_dev, const float* ctrl_dev, float* obs_dev, float* qacc_dev, void* stream) {
  if (!h) return fail("usim_forward: null handle");
  if (!h->slots_init) return fail("usim_forward: no state to evaluate before the first usim_reset");
  if (activate(h)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const int n = h->n;
  if (!h->fwd_armbuf) CK(cudaMalloc((void**)&h->fwd_armbuf, (size_t)n * ARMBUF * sizeof(float)));
  if (qacc_dev && !h->fwd_qacc) CK(cudaMalloc((void**)&h->fwd_qacc, (size_t)n * QPAD * sizeof(float)));
  const int grid = (n + ARM_BLOCK - 1) / ARM_BLOCK;
  if (h->narm == 7) forward_arm_kernel<7><<<grid, ARM_BLOCK, 0, s>>>(n, mask_dev, h->qpos, h->qvel, ctrl_dev, h->task, h->fwd_armbuf);
  else forward_arm_kernel<6><<<grid, ARM_BLOCK, 0, s>>>(n, mask_dev, h->qpos, h->qvel, ctrl_dev, h->task, h->fwd_armbuf);
  SolveArgs a = base_args(h, 1);
  a.fwd = 1; a.armbuf = h->fwd_armbuf; a.mask = mask_dev; a.obs = obs_dev; a.qacc_out = qacc_dev ? h->fwd_qacc : nullptr;
  a.counters = nullptr;
  solve_kernel<<<n, NT, sizeof(WS), s>>>(a);
  h->launches += 2;
  if (qacc_dev) { // (the solve kernel stores whole 16-byte aligned rows by TMA: a dense [n][nv] row is not aligned)
    const int tot = n * h->nv;
    qacc_rows_kernel<<<(tot + 255) / 256, 256, 0, s>>>(n, h->nv, mask_dev, h->fwd_qacc, qacc_dev);
    h->launches += 1;
  }
  CK(cudaGetLastError());
  if (h->crec_on && !mask_dev) h->crec_complete = true;
  return mark_state(h, s);
}

int usim_step(usim_handle* h, const float* act_dev, float* obs_dev, float* rew_dev, uint8_t* done_dev, float* term_obs_dev,
              int auto_reset, void* stream) {
  if (!h) return fail("usim_step: null handle");
  if (!act_dev || !done_dev) return fail("usim_step: act_dev and done_dev are required");
  if (activate(h)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  if (auto_reset && !h->slots_init) return fail("usim_step: auto_reset needs a usim_reset first (no reset state has been prepared)");
  if (launch_step(h, act_dev, obs_dev, rew_dev, done_dev, term_obs_dev, auto_reset, s)) return -1;
  return mark_state(h, s);
}

// page-locked host memory (cudaHostAlloc / cudaHostRegister / torch pin_memory) can be the DMA end point itself
static bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

// device-side alias of a page-locked host buffer (UVA: cudaHostAlloc / cudaHostRegister / torch pin_memory are mapped), or nullptr
static void* mapped_alias(const void* p) {
  void* d = nullptr;
  if (!p || !is_pinned(p)) return nullptr;
  if (cudaHostGetDevicePointer(&d, const_cast<void*>(p), 0) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return d;
}

int usim_step_host(usim_handle* h, const float* act, float* obs, float* rew, uint8_t* done, float* tobs, int auto_reset) {
  if (!h) return fail("usim_step_host: null handle");
  if (!act) return fail("usim_step_host: act is required");
  if (activate(h)) return -1;
  cudaStream_t s = h->own_stream;
  size_t N = (size_t)h->n;
  const size_t row = USIM_OBS_DIM * sizeof(float);
  // A page-locked action array is copied from directly; a pageable one goes through the library's pinned staging buffer.
  const float* a_src = act;
  if (!is_pinned(act)) { memcpy(h->h_act, act, N * h->adim * sizeof(float)); a_src = h->h_act; }
  // Observation rows, reward, done flag -- and the terminal rows of the envs that finish in this step, typically ~N / episode length
  // of them -- are written by the solve kernel STRAIGHT into page-locked host memory (one coalesced 76-byte row per env, posted PCIe
  // writes that overlap the rest of the launch): no device->host copy after the kernel, no second round trip for the terminal rows,
  // and only the rows of finished envs are touched in `term_obs_host`.  A caller buffer with a device alias is written in place; any
  // other goes through the library's staging buffer.
  float* o_dev = (float*)mapped_alias(obs);
  float* t_dev = (float*)mapped_alias(tobs);
  float* r_dev = (float*)mapped_alias(rew);
  uint8_t* d_dev = (uint8_t*)mapped_alias(done);
  float* o_host = o_dev ? obs : h->h_obs;
  float* t_host = t_dev ? tobs : h->h_tobs;
  float* r_host = r_dev ? rew : h->h_rew;
  uint8_t* d_host = d_dev ? done : h->h_done;
  if (!o_dev) o_dev = h->map_obs;
  if (!t_dev) t_dev = h->map_tobs;
  if (!r_dev) r_dev = h->map_rew;
  if (!d_dev) d_dev = h->map_done;
  // the private stream is ordered after the last state-mutating call made on a caller's stream (usim_reset / usim_step /
  // usim_set_state), and this call synchronises it before returning: the two kinds of call may be mixed freely
  if (h->ev_state_valid) CK(cudaStreamWaitEvent(s, h->ev_state, 0));
  CK(cudaMemcpyAsync(h->d_act, a_src, N * h->adim * sizeof(float), cudaMemcpyHostToDevice, s));
  if (usim_step(h, h->d_act, o_dev, r_dev, d_dev, tobs ? t_dev : nullptr, auto_reset, s)) return -1;
  CK(cudaStreamSynchronize(s));
  if (obs && o_host != obs) memcpy(obs, o_host, N * row);
  if (rew && r_host != rew) memcpy(rew, r_host, N * sizeof(float));
  if (done && d_host != done) memcpy(done, d_host, N);
  if (tobs && t_host != tobs) { // the kernel wrote the finished envs' rows into the staging buffer
    for (size_t e = 0; e < N; e++)
      if (d_host[e]) memcpy(tobs + e * USIM_OBS_DIM, t_host + e * USIM_OBS_DIM, row);
  }
  return 0;
}

// strided row copies between the padded internal rows and the caller's dense [n][dim] arrays
__global__ void rows_copy(int n, int dim, int src_pitch, int dst_pitch, const float* __restrict__ src, float* __restrict__ dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * dim) return;
  int e = i / dim, k = i - e * dim;
  dst[(size_t)e * dst_pitch + k] = src[(size_t)e * src_pitch + k];
}
static void rc(usim_handle* h, int dim, int sp, int dp, const float* src, float* dst, cudaStream_t s) {
  int tot = h->n * dim;
  rows_copy<<<(tot + 255) / 256, 256, 0, s>>>(h->n, dim, sp, dp, src, dst);
  h->launches += 1;
}

int usim_get_state(usim_handle* h, float* qpos, float* qvel, float* warm, float* task, void* stream) {
  if (!h) return fail("usim_get_state: null handle");
  if (activate(h)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  if (qpos) rc(h, h->nq, QPAD, h->nq, h->qpos, qpos, s);
  if (qvel) rc(h, h->nv, QPAD, h->nv, h->qvel, qvel, s);
  if (warm) rc(h, h->nv, QPAD, h->nv, h->warm, warm, s);
  if (task) rc(h, USIM_TASK_DIM, USIM_TASK_DIM, USIM_TASK_DIM, h->task, task, s);
  CK(cudaGetLastError());
  return 0;
}
int usim_set_state(usim_handle* h, const float* qpos, const float* qvel, const float* warm, const float* task, void* stream) {
  if (!h) return fail("usim_set_state: null handle");
  if (activate(h)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  if (qpos) rc(h, h->nq, h->nq, QPAD, qpos, h->qpos, s);
  if (qvel) rc(h, h->nv, h->nv, QPAD, qvel, h->qvel, s);
  if (warm) rc(h, h->nv, h->nv, QPAD, warm, h->warm, s);
  if (task) rc(h, USIM_TASK_DIM, USIM_TASK_DIM, USIM_TASK_DIM, task, h->task, s);
  CK(cudaGetLastError());
  // the slots hold the reset states of the counters before the restore: prepare them again from the restored ones (bit-identical
  // slots where a counter did not change, since a prepared state depends on nothing but (seed, env id, episode number))
  if (task && h->slots_init && prepare_slots(h, s)) return -1;
  return mark_state(h, s);
}

int usim_get_arm_record(usim_handle* h, float* rec, void* stream) {
  if (!h || !rec) return fail("usim_get_arm_record: null argument");
  static_assert(USIM_ARM_RECORD_DIM == ARMBUF, "the ABI's arm-record pitch is the kernels' row pitch");
  CK(cudaMemcpyAsync(rec, h->armbuf, (size_t)h->n * ARMBUF * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int usim_get_contacts(usim_handle* h, int32_t* ncon, int32_t* g1, int32_t* g2, float* dist, void* stream) {
  if (!h) return fail("usim_get_contacts: null handle");
  cudaStream_t s = (cudaStream_t)stream;
  size_t N = (size_t)h->n;
  if (ncon) CK(cudaMemcpyAsync(ncon, h->ncon, N * sizeof(int), cudaMemcpyDeviceToDevice, s));
  if (g1) CK(cudaMemcpyAsync(g1, h->geom1, N * DEV_MAXC * sizeof(int), cudaMemcpyDeviceToDevice, s));
  if (g2) CK(cudaMemcpyAsync(g2, h->geom2, N * DEV_MAXC * sizeof(int), cudaMemcpyDeviceToDevice, s));
  if (dist) CK(cudaMemcpyAsync(dist, h->cdist, N * DEV_MAXC * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}
int usim_set_contact_record(usim_handle* h, int enable) {
  if (!h) return fail("usim_set_contact_record: null handle");
  if (enable && !h->crec) {
    CK(cudaSetDevice(h->device));
    CK(cudaMalloc((void**)&h->crec, (size_t)h->n * DEV_MAXC * CREC_DIM * sizeof(float)));
  }
  if (!enable || !h->crec_on) h->crec_complete = false; // the record no longer follows the contact list until every env is launched again
  h->crec_on = enable != 0;
  return 0;
}

// record row -> MuJoCo layouts: contact frame (rows: normal, then the tangents of the make_frame rule: the world y axis, or z when the
// normal is within 60 degrees of y, orthogonalised against the normal; third = normal x second) and the force in that frame
__global__ void contact_forces_kernel(int n, const int* __restrict__ ncon, const float* __restrict__ rec, float* __restrict__ pos,
                                      float* __restrict__ frame, float* __restrict__ force) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * DEV_MAXC) return;
  const int c = i % DEV_MAXC;
  float p[3] = {0, 0, 0}, fm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, f[3] = {0, 0, 0};
  if (c < ncon[i / DEV_MAXC]) {
    const float* r = rec + (size_t)i * CREC_DIM;
    const v3 nn = mk(r[3], r[4], r[5]), F = mk(r[6], r[7], r[8]);
    const v3 t = fabsf(nn.y) < 0.5f ? mk(0, 1, 0) : mk(0, 0, 1);
    v3 y = t - dot(nn, t) * nn;
    y = (1.f / norm(y)) * y;
    const v3 z = cross(nn, y);
    p[0] = r[0]; p[1] = r[1]; p[2] = r[2];
    fm[0] = nn.x; fm[1] = nn.y; fm[2] = nn.z; fm[3] = y.x; fm[4] = y.y; fm[5] = y.z; fm[6] = z.x; fm[7] = z.y; fm[8] = z.z;
    f[0] = dot(nn, F); f[1] = dot(y, F); f[2] = dot(z, F);
  }
  if (pos) for (int k = 0; k < 3; k++) pos[(size_t)i * 3 + k] = p[k];
  if (frame) for (int k = 0; k < 9; k++) frame[(size_t)i * 9 + k] = fm[k];
  if (force) for (int k = 0; k < 3; k++) force[(size_t)i * 3 + k] = f[k];
}

int usim_get_contact_forces(usim_handle* h, float* pos, float* frame, float* force, void* stream) {
  if (!h) return fail("usim_get_contact_forces: null handle");
  if (!h->crec) return fail("usim_get_contact_forces: contact recording was never enabled (usim_set_contact_record)");
  if (!h->crec_complete)
    return fail("usim_get_contact_forces: no step or reset of every env has run since contact recording was enabled");
  if (!pos && !frame && !force) return 0;
  CK(cudaSetDevice(h->device));
  const int tot = h->n * DEV_MAXC;
  contact_forces_kernel<<<(tot + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->n, h->ncon, h->crec, pos, frame, force);
  h->launches += 1;
  CK(cudaGetLastError());
  return 0;
}
int usim_get_diag(usim_handle* h, float* diag, void* stream) {
  if (!h || !diag) return fail("usim_get_diag: null argument");
  CK(cudaMemcpyAsync(diag, h->diag, (size_t)h->n * USIM_DIAG_DIM * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int usim_num_envs(const usim_handle* h) { return h ? h->n : -1; }
int usim_nq(const usim_handle* h) { return h ? h->nq : -1; }
int usim_nv(const usim_handle* h) { return h ? h->nv : -1; }
int usim_action_dim(const usim_handle* h) { return h ? h->adim : -1; }
int64_t usim_launch_count(const usim_handle* h) { return h ? h->launches : -1; }
int usim_divergence_count(usim_handle* h, int64_t* count) {
  if (!h || !count) return fail("usim_divergence_count: null argument");
  int c = 0;
  CK(cudaMemcpy(&c, h->counters, sizeof(int), cudaMemcpyDeviceToHost)); // synchronises the device
  *count = c;
  return 0;
}
int usim_contact_overflow_count(usim_handle* h, int64_t* count) {
  if (!h || !count) return fail("usim_contact_overflow_count: null argument");
  int c = 0;
  CK(cudaMemcpy(&c, h->counters + 1, sizeof(int), cudaMemcpyDeviceToHost)); // synchronises the device
  *count = c;
  return 0;
}
int usim_substeps(const usim_handle* h) { return h ? h->substeps : -1; }
int usim_set_timing(usim_handle* h, int enable) {
  if (!h) return fail("usim_set_timing: null handle");
  h->timing = enable != 0;
  return 0;
}

int usim_kernel_time(usim_handle* h, int reset, double* total_ms, int64_t* launches) {
  if (!h) return fail("usim_kernel_time: null handle");
  for (auto& p : h->pending) {
    CK(cudaEventSynchronize(p.second));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, p.first, p.second));
    h->timed_ms += ms;
    h->timed_launches += 1;
    cudaEventDestroy(p.first); cudaEventDestroy(p.second);
  }
  h->pending.clear();
  if (total_ms) *total_ms = h->timed_ms;
  if (launches) *launches = h->timed_launches;
  if (reset) { h->timed_ms = 0.0; h->timed_launches = 0; }
  return 0;
}
