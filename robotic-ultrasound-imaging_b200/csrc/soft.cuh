// soft.cuh — K3..K9 fused: one CTA of two warps per env, the whole env state staged in shared memory.
//
//   K3 torso kinematics + inertia + bias   (free body + 270 radial sliders, arrow-structured M)
//   K4 collision: table<->particle, probe<->particle, table<->probe, deterministic MuJoCo ordering
//   K5 constraint parameters: solref/solimp -> aref, D; equality rows folded into a 270-node stencil
//   K6 primal nonlinear CG (Polak-Ribiere, exact Newton line search, elliptic cones) with an
//      arrow preconditioner (6x6 Schur complement over the slider diagonal) + 7x7 arm block
//   K7 semi-implicit Euler, quaternion integration      K8 cfrc_ext / F-T torque of the probe
//   K9 reward, running statistics, termination, observation (ultrasound.py:230-269,363-401,512-550,635-670)
//
// Unknown vector layout (nv = 283): [0..6] arm, [7..9] free translation (world), [10..12] free
// rotation (body frame), [13+i] slider i.  No constraint Jacobian is ever materialised: contact
// rows are evaluated as rigid-body point velocities / wrenches, equality rows as a graph stencil.
//
// Structure of one CG iteration (every dot product rides on a pass that exists anyway; 5 warp reductions):
//   applyH(s) [+ s.Hx, s.Hs]  ->  contact rows J s  ->  line search (Newton on phi')  ->  x, Hx, grad, jar updates [+ |Hx|^2]
//   ->  contact forces into grad [+ probe wrench, zone changes]  ->  (preconditioner rebuild if the active set moved, from the fourth iteration on)
//   ->  pg = P^-1 grad [+ grad.pg_old, grad.pg, |grad|^2, the slider sums of pg that the next applyH needs]  ->  s = -pg + beta s
#pragma once
#include "common.cuh"

// One env per CTA: no CTA waits for a slower env (measured 1/2/4/8 envs per CTA: 2.17/2.12/1.96/1.82 M steps/s).
// WPE warps cooperate on that env over the same shared-memory image: twice the resident warps per SM for the same shared memory,
// half the latency of one env (a 4096-env launch is only ~3.5 waves of CTAs: the tail matters), one instruction stream fetched for two warps.
// Every cross-lane / cross-warp accumulation has a fixed association order: results are bit-reproducible for a given WPE.
#ifndef WPE
#define WPE 2
#endif
#ifndef USIM_TRACE
#define USIM_TRACE 0 // 1 (developer build, scripts/trace_tail.py): every work item records (start ns, end ns, SM id) when the USIM_TRACE=<file> environment variable is set
#endif
#define NT (32 * WPE)
#ifndef MINB
#define MINB (WPE <= 2 ? 8 : 16 / WPE) // resident CTAs per SM the register allocation is sized for
#endif
// More resident envs per SM do not pay (measured, 32 768 envs, round 2): with the preconditioner-only arrays in bfloat16, one-byte
// contact slots and aliased reduction zones the env image shrinks to 24.3 KB = 9 CTAs per SM, but the 9th needs <= 112 registers:
// 120 regs / 8 CTAs 8.83 M env-steps/s, 112 / 9: 8.47 M, 96 / 9: 8.34 M, 96 / 8: 8.00 M -- the register-capped schedule costs 5-9 %, the
// extra CTA returns 4 %.  Three or four warps per env at 8 envs per SM (24 / 32 warps, 80 / 72 registers): 7.22 / 6.22 M against 7.82 M.
// Fewer resident envs (USIM_SMEM_PAD): 7 / 6 / 5 CTAs per SM = 8.18 / 7.70 / 7.22 M.
#define NPAIR_MAX 544
#define SLOT_OBS 20 // row pitch of a prepared observation (19 used)
// Slider block of the preconditioner, D - W (D: diagonal, W: the pair couplings of the shell grid), inverted by a polynomial in
// N = D^-1 W.  PREC3 = 0: second order, D^-1 (I + N).  PREC3 = 1: third order with Chebyshev weights, D^-1 (I + c (N + N^2)),
// c = 4 / (4 - 3 rho^2): the cubic (1 - x) p(x) = 1 - T3(x / rho) / T3(1 / rho) deviates least from 1 on the spectrum [-rho, rho]
// of N.  rho ~ 0.7 for this model (sum of a slider's pair D over its diagonal) -> c = 1.6; measured at 4096 envs:
// second order 0.513 ms, c = 1.0 (plain Neumann) 0.513, 1.4: 0.485, 1.7: 0.483, 2.0: 0.488, 2.4: 0.506, 3.0: 0.578;
// fourth order (three stencil passes, a0 (z0 + z1) + a2 (z2 + z3)): 0.488 ms vs 0.464 for the cubic -- not kept.
// Round 2, after the rebuild policy (most solves keep the preconditioner of their warm start): the SECOND-order block does as well as the
// cubic in iterations and saves a stencil pass -- PREC3 = 0: 0.428 ms / 5.73 iterations, PREC3 = 1 (c = 1.1): 0.442 / 5.79; Jacobi
// (PREC_JACOBI): 0.473 / 7.05; weight 0.8 / 1.2 / 1.4 on the first-order term (PREC2_C): 0.441 / 0.449 / 0.503.
#ifndef PREC3
#define PREC3 0
#endif
// Re-measured on the final kernel of round 2 (calibrated probe, line-search tolerance 0.03; kernel ms / CG iterations): 0.9: 0.487 / 5.31,
// 1.0: 0.479 / 5.32, 1.1: 0.480 / 5.33, 1.2: 0.479 / 5.34, 1.3: 0.483 / 5.37, 1.4: 0.483 / 5.41, 1.5: 0.485 / 5.45, 1.6: 0.486 / 5.50,
// 1.8: 0.497 / 5.65 -- the optimum is a plateau from the plain Neumann series (1.0) to 1.2: the contact terms on the diagonal have
// lowered the effective rho.
#ifndef CHEB_C
#define CHEB_C 1.1f
#endif
// Arm part of the warm start: the previous qacc shifted by M^-1 (qfrc_smooth_now - qfrc_smooth_previous), computed by the arm kernel
// with the Cholesky factor it holds anyway.  A fresh action every step moves qfrc_smooth of the arm by the change of the controller
// torque; without the shift the previous qacc is a poor start for the 7 arm unknowns (6.4 CG iterations with random actions, 4.0 with
// a constant one).
#ifndef ARM_SHIFT
#define ARM_SHIFT 1
#endif
#ifndef WARP_SOLVE
#define WARP_SOLVE 0 // 1: dense blocks of the preconditioner solved by one warp with shuffles (chol7_solve_warp2) instead of replicated in every thread.  Measured at 4096 envs: 0.441 ms vs 0.4245 ms replicated -- ~150 instead of ~290 instructions, but the 28 dependent shuffles are the longer chain and the kernel is latency bound: not kept.  Re-measured with the first stencil pass on the second warp (SPLIT_Z1): 0.5064 vs 0.4993 ms
#endif
#ifndef SPLIT_SOLVE
#define SPLIT_SOLVE (WPE == 2 && PREC3 && !WARP_SOLVE) // 1: the first warp solves the dense blocks while the second runs the first stencil pass of the slider block for all sliders (instead of both warps doing both)
#endif
#ifndef SPLIT_DENSE
#define SPLIT_DENSE 0 // 1 (needs WPE == 2, PREC3 == 0): the first warp solves the 7x7 arm block, the second the 6x6 torso block, one more barrier, instead of both warps solving both.  Measured: 0.4280 vs 0.4281 ms -- parity green, no gain, not shipped
#endif
#ifndef SPLIT_Z1
#define SPLIT_Z1 (SPLIT_SOLVE || (WARP_SOLVE && WPE == 2 && PREC3)) // the first stencil pass belongs to the second warp alone
#endif
#ifndef NORESTART
#define NORESTART 1 // 1: keep the Polak-Ribiere direction across a preconditioner rebuild (flexible CG: beta uses the previous pg, made with the previous preconditioner) instead of restarting; measured 0.464 ms vs 0.485 ms
#endif
#ifndef LS_TOL
#define LS_TOL 0.03f // line search: stop when |phi'| has dropped by this factor.  An inexact search is enough for nonlinear CG (the
                     // converged solution does not depend on it, only the path).  Measured at 4096 envs on the final kernel of round 2
                     // (kernel ms / CG iterations / line-search evaluations per env-step): 1e-3: 0.498 / 5.45 / 13.2, 1e-2: 0.490 / 5.47 / 12.1,
                     // 0.02: 0.488 / 5.48 / 11.9, 0.03: 0.487 / 5.50 / 11.85, 0.05: 0.487 / 5.52 / 11.75, 0.1: 0.488 / 5.57 / 11.7, 0.3: 0.501 / 5.64 / 11.7
                     // (round 1: 1e-5 cost one more evaluation per iteration for nothing in fp32)
#endif
#ifndef LS_MAX
#define LS_MAX 8 // evaluations of phi'(alpha) per line search (Newton with bracketing; 1 = one quadratic step, unverified)
#endif
// unroll factor of the NT-strided loops inside the CG iteration (each warp runs only 4-5 trips of a slider loop, 1-2 of a contact loop):
// trades ILP against the size of the loop body in the instruction cache (`no_instruction` is the top stall with 16 warps per SM)
#define USIM_STR2(x) #x
#define USIM_STR(x) USIM_STR2(x)
// measured, 4096 envs: compiler default 6.52 M steps/s (7456 SASS instructions), unroll 1: 6.61 M (7096), unroll 2: 5.79 M (8296);
// final kernel of round 2: unroll 1 7.87 M, the per-slider loops alone x2 (HOT_UNROLL_S=2) 7.31 M, every hot loop x2 5.11 M -- the
// loop body sits at the edge of the instruction cache: +400 instructions cost 8 %, +1200 cost 35 %
#ifndef HOT_UNROLL
#define HOT_UNROLL 1
#endif
#define PRAGMA_HOT _Pragma(USIM_STR(unroll HOT_UNROLL))
#ifndef HOT_UNROLL_S
#define HOT_UNROLL_S HOT_UNROLL // the per-slider / per-unknown loops alone (4-5 trips per warp); the per-contact loops run 1-2 trips
#endif
#define PRAGMA_HOT_S _Pragma(USIM_STR(unroll HOT_UNROLL_S))

struct __align__(16) WS {
  // ---- landing zones of the 1-D TMA bulk copies (whole HBM rows, 16-byte aligned; written back the same way) ----
  float qrow[QPAD];                                    // qpos row: [0..6] arm, [7..9] torso position, [10..13] torso quaternion, [14+i] slider i
  // Hx holds (M+E)x - rhs; during set-up `grad` accumulates rhs (= qfrc_smooth + J_eq^T D aref).
  // x <- qacc_warmstart row; hs <- qvel row (slider velocity lives in hs[13..] until the CG loop starts)
  float x[QPAD], Hx[QPAD], grad[QPAD], pg[QPAD], s[QPAD], hs[QPAD];
  float ab[ARMBUF];
  float ts[USIM_TASK_DIM];
  unsigned long long bar;                              // mbarrier of the load
#if USIM_TRACE
  unsigned long long t0;                               // developer trace: start time of this work item
#endif
  // ----
  float dg[NPART_MAX], dgm[NPART_MAX];                 // dg: slider diagonal of the preconditioner, stored INVERTED; dgm: M+E diagonal w/o tendon
  float Dp[NPAIR_MAX];                                 // D of each "smooth" pair
  float cpos[3][DEV_MAXC], cn[3][DEV_MAXC], cjar[3][DEV_MAXC], cjv[3][DEV_MAXC]; // cjv holds aref until the first J*x
  float cD[DEV_MAXC];
  float cfs[DEV_MAXC];                                 // per-contact scratch: penetration depth until K5, then the contact's share of a slider row
  float sk[3][DEV_MAXC], sc[3][DEV_MAXC];              // per owner slot of a slider with contacts: K a (world), lever x K a
  short cslot[NPART_MAX];                              // first contact slot of a slider (its "owner slot"), -1 = no contact
  short cslot2[NPART_MAX];                             // slot of the slider's probe contact, -1 = none
  short cpart[DEV_MAXC];
  unsigned char ctype[DEV_MAXC], czone[DEV_MAXC];
  float R[9], p[3], vf[6], qdarm[7];
  float Mff[36], Mfw[21], Sf[49], Pa[49];              // Mfw: free-body inertia, world-frame omega, packed upper triangle; Sf/Pa: 7x7 Cholesky factors
  float dv[12];
  // landing zones of the warp reductions, one per call site, one row per warp (readers add the rows in a fixed order: rd())
  float r3[WPE][24], rg[WPE][16], rp[WPE][16], rq[WPE][8], rl[2][WPE][4], rb1[WPE][24], rb2[WPE][24], rb3[WPE][24];
  float lsign[7], lD[7], laref[7];
  float yS[8];                                         // torso part of P^-1 grad (world frame), warp 0 -> all threads
  float Dt, areft;
  int ncon, okf;
  int consume;                                         // this env's episode ended and a prepared reset slot takes over (K9 -> all threads)
  int item;                                            // work item fetched from the launch's queue (thread 0 -> all threads)
  int cnt[2][WPE];                                     // cross-warp prefix of the contact compaction (double buffered)
  float orow[SLOT_OBS];                                // observation row of this step (K9, thread 0) -> written out as ONE coalesced row
};
#ifndef SKIP_SMEM_ASSERT
static_assert(sizeof(WS) + 1024 <= 233472 / MINB, "WS must leave room for MINB CTAs per SM");
#endif
static_assert(2 * QPAD >= NPAIR_MAX + 1, "pg|s double as the pair scratch of K3");

__device__ __forceinline__ void env_sync() {
  if (WPE == 1) __syncwarp(); else __syncthreads();
}
// total of entry k of a reduction landing zone (rows = warps, added in warp order)
template <int N>
__device__ __forceinline__ float rd(const float (*z)[N], int k) {
  float t = z[0][k];
#pragma unroll
  for (int q = 1; q < WPE; q++) t += z[q][k];
  return t;
}

// ---- 1-D TMA bulk copies (cp.async.bulk, SASS UBLKCP): whole state rows HBM <-> shared memory, issued by one thread ----
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned phase) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "USIM_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra USIM_DONE;\n"
      "bra USIM_WAIT;\n"
      "USIM_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(phase) : "memory");
}
__device__ __forceinline__ void tma_load_row(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_store_row(void* dst_gmem, const void* src_smem, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (before a bulk store reads them)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_store_commit_wait() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// Transposing warp reduction of K values: K-1 shuffles instead of 5K.  Returns, in lane l, the warp total of entry
// l & (KP-1), KP = K rounded up to a power of two.  Fixed association order -> bit-reproducible.
template <int K>
__device__ __forceinline__ float tsum(const float (&v)[K], int lane) {
  constexpr int KP = K <= 1 ? 1 : K <= 2 ? 2 : K <= 4 ? 4 : K <= 8 ? 8 : K <= 16 ? 16 : 32;
  static_assert(K <= 32, "tsum: at most 32 values");
  float t[KP];
#pragma unroll
  for (int k = 0; k < KP; k++) t[k] = k < K ? v[k] : 0.f;
#pragma unroll
  for (int n = KP; n > 1; n >>= 1) {
    const int o = n >> 1;
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int j = 0; j < o; j++) {
      float a = t[j], b = t[j + o];
      float send = up ? a : b, keep = up ? b : a;
      t[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
#pragma unroll
  for (int o = KP; o < 32; o <<= 1) t[0] += __shfl_xor_sync(0xffffffffu, t[0], o);
  return t[0];
}
// reduce K values and land them in shared memory (dst[0..K-1]); the caller syncs before reading
template <int K>
__device__ __forceinline__ void tsum_to(const float (&v)[K], int lane, float* dst) {
  float r = tsum(v, lane);
  if (lane < K) dst[lane] = r;
}

// (row, col) of entry l of a packed upper triangle of a 6x6, row-major
__constant__ unsigned char c_tri6[21] = {0x00, 0x01, 0x02, 0x03, 0x04, 0x05, 0x11, 0x12, 0x13, 0x14, 0x15,
                                         0x22, 0x23, 0x24, 0x25, 0x33, 0x34, 0x35, 0x44, 0x45, 0x55};
__device__ __forceinline__ constexpr int tri6(int a, int b) { return a <= b ? a * 6 - a * (a - 1) / 2 + (b - a) : b * 6 - b * (b - 1) / 2 + (a - b); }

// Elliptic cone (condim 3) in WORLD coordinates.  The cone is isotropic in the tangent plane (one friction coefficient, one
// tangential D), so no tangent basis is needed: a contact row triple is kept as the world vector j = J x - aref, split as
// j = jn n + jt.  Returns the world force on geom2 and the zone (0 = top / inactive, 1 = middle, 2 = bottom / quadratic).
__device__ __forceinline__ v3 cone_force(v3 j, v3 n, float Dn, float Dt, float mu, float fr, int& zone) {
  const float jn = dot(j, n);
  const v3 jt = j - jn * n;
  const float N = jn * mu, T = fr * norm(jt);
  if (N >= mu * T || (T <= 0.f && N >= 0.f)) { zone = 0; return mk(0, 0, 0); }
  if (mu * N + T <= 0.f || (T <= 0.f && N < 0.f)) { zone = 2; return (-Dn * jn) * n - Dt * jt; }
  zone = 1;
  const float Dm = Dn / (mu * mu * (1.f + mu * mu)), f0 = -Dm * (N - mu * T) * mu;
  return f0 * n - (f0 * fr * fr / T) * jt;
}
// first / second directional derivative of the cone cost at j along v
__device__ __forceinline__ void cone_ls(v3 j, v3 v, v3 n, float Dn, float Dt, float mu, float fr, float& d1, float& d2) {
  const float jn = dot(j, n), vn = dot(v, n);
  const v3 jt = j - jn * n, vt = v - vn * n; // explicit tangential parts: |j|^2 - jn^2 would cancel when the load is mostly normal
  const float tt = dot(jt, jt), tv = dot(jt, vt), vv = dot(vt, vt);
  const float N = jn * mu, T = fr * sqrtf(tt);
  if (N >= mu * T || (T <= 0.f && N >= 0.f)) { d1 = 0.f; d2 = 0.f; }
  else if (mu * N + T <= 0.f || (T <= 0.f && N < 0.f)) {
    d1 = Dn * jn * vn + Dt * tv;
    d2 = Dn * vn * vn + Dt * vv;
  } else {
    const float Dm = Dn / (mu * mu * (1.f + mu * mu)), g = N - mu * T, f2 = fr * fr;
    const float Tp = f2 * tv / T;
    const float Tpp = (f2 * vv - Tp * Tp) / T;
    const float gp = mu * vn - mu * Tp;
    d1 = Dm * g * gp;
    d2 = Dm * (gp * gp - g * mu * Tpp);
  }
}

__device__ __forceinline__ void contact_params(int type, float& fr, float& mu) {
  fr = type == 0 ? dm.fr_table_part : (type == 1 ? dm.fr_probe_part : dm.fr_table_probe);
  mu = fr * rsqrtf(dm.impratio);
}

// closest points between segments (p1,q1) and (p2,q2) — same branch structure as the oracle
__device__ __forceinline__ void seg_seg(v3 p1, v3 q1, v3 p2, v3 q2, v3& c1, v3& c2) {
  v3 d1 = q1 - p1, d2 = q2 - p2, r = p1 - p2;
  float a = dot(d1, d1), e = dot(d2, d2), f = dot(d2, r), c = dot(d1, r), b = dot(d1, d2), den = a * e - b * b, s, t;
  if (den > 1e-14f * a * e) s = fminf(fmaxf((b * f - c * e) / den, 0.f), 1.f); else s = 0.f;
  t = (b * s + f) / e;
  if (t < 0.f) { t = 0.f; s = fminf(fmaxf(-c / a, 0.f), 1.f); }
  else if (t > 1.f) { t = 1.f; s = fminf(fmaxf((b - c) / a, 0.f), 1.f); }
  c1 = p1 + s * d1;
  c2 = p2 + t * d2;
}

// In-place Cholesky of TWO 7x7 matrices (row-major, pitch 7, both triangles valid on entry) held in shared memory, by one warp:
// one matrix row per lane (lanes 0-6 -> A0, lanes 8-14 -> A1; A1 may be null), right-looking, rows in registers, columns exchanged by shuffles.
// The factors are left in the lower triangles with their diagonals INVERTED (the solves multiply).  Returns false in the lanes of a
// matrix that met a non-positive pivot (the pivot is clamped).  Every loop has a constant trip count: nothing is indexed dynamically.
__device__ __forceinline__ bool chol7_warp2(float* A0, float* A1, int lane) {
  const int base = lane & 8, r = lane & 7;
  float* A = base ? A1 : A0;
  const bool act = lane < 16 && r < 7 && A != nullptr; // A1 == nullptr: factorise A0 only
  float row[7];
#pragma unroll
  for (int k = 0; k < 7; k++) row[k] = act ? A[r * 7 + k] : (k == r ? 1.f : 0.f);
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 7; j++) {
    float d = __shfl_sync(0xffffffffu, row[j], base + j);
    if (!(d > 0.f)) { ok = false; d = 1e-20f; }
    const float inv = rsqrtf(d);
    const float l = row[j] * inv; // L[r][j] for r > j, sqrt(d) for r == j, unused above the diagonal
#pragma unroll
    for (int k = 0; k < 7; k++) {
      if (k > j) row[k] -= l * __shfl_sync(0xffffffffu, l, base + k);
    }
    row[j] = r == j ? inv : l;
  }
#pragma unroll
  for (int k = 0; k < 7; k++)
    if (act && k <= r) A[r * 7 + k] = row[k];
  return ok;
}
// x <- (L L^T)^-1 b for TWO factors written by chol7_warp2, at once, by one warp: lane r (0..6) holds entry r of the right-hand side of
// A0, lane 8 + r that of A1; the solution entry comes back in the same lane.  Column-oriented substitution: one broadcast shuffle and
// one FMA per column (28 shuffles in all) instead of the ~290 replicated, fully unrolled instructions of chol7_solve<7> + <6> in every
// thread -- the loop body of the solver has to fit the 32 KB instruction cache.
__device__ __forceinline__ float chol7_solve_warp2(const float* A0, const float* A1, float b, int lane) {
  const int base = lane & 8, r = lane & 7;
  const float* A = base ? A1 : A0;
  const bool act = lane < 16 && r < 7;
  float Lr[7], Lc[7]; // row r of L left of the diagonal, column r below it (zero elsewhere: no predicates in the loops)
#pragma unroll
  for (int k = 0; k < 7; k++) {
    Lr[k] = (act && k < r) ? A[r * 7 + k] : 0.f;
    Lc[k] = (act && k > r) ? A[k * 7 + r] : 0.f;
  }
  const float dinv = act ? A[r * 7 + r] : 1.f;
  if (!act) b = 0.f;
#pragma unroll
  for (int j = 0; j < 7; j++) { // L y = b
    if (r == j) b *= dinv;
    b -= Lr[j] * __shfl_sync(0xffffffffu, b, base + j);
  }
#pragma unroll
  for (int j = 6; j >= 0; j--) { // L^T x = y
    if (r == j) b *= dinv;
    b -= Lc[j] * __shfl_sync(0xffffffffu, b, base + j);
  }
  return b;
}

// Launch slots are ordered longest-solve-first: every launch files its envs into NBIN bins by the number of CG iterations they
// took; the arm kernel of the next physics step flattens the bins (highest first) into `order`, and CTA j of the next solve launch
// takes env order[j].  The block scheduler hands CTAs out in index order, so the slow envs start first and the tail of the launch
// (3.5 waves at 4096 envs) is made of the quick ones.  Which CTA runs an env never changes its result.
#define NBIN 16

// Reset pipeline.  The state an env is reset to is a pure function of (seed, global env id, episode number): it is PREPARED ahead of
// time, off the critical path, into one of two per-env slots (slot k holds an episode number with parity k), by the reset kernel +
// this kernel in forward-only mode on a side stream.  When an episode ends inside a step (auto-reset, SB3 VecEnv semantics) the CTA
// that stepped the env copies the prepared rows over the live state -- no extra launch -- and files a request to prepare the
// episode after next into the slot it has just emptied.
struct SolveArgs {
  int n;          // envs of this handle
  int mode;       // 0 = env step (last physics substep of a control step: integrates, then the task epilogue), 1 = reset forward (no
                  // integration; initialises the running statistics), 2 = intermediate physics substep (integrates, no task epilogue)
  int prep;       // 1: prepare mode (mode must be 1): work items and state rows come from the request list / the slots
  int auto_reset; // mode 0: an env whose episode ends takes over its prepared slot
  const uint8_t* mask; // mode 1, live: envs to process (nullptr: all)
  float *qpos, *qvel, *warm, *task;
  const float* armbuf; // live: [n][ARMBUF]; prepare mode: [items][ARMBUF]
  PartTables pt;
  const int2* eq_pairs;
  float *obs, *rew;
  uint8_t* done;
  float* tobs;
  float* diag;
  int *ncon_out, *geom1_out, *geom2_out;
  float* dist_out;
  int* counters;  // [0] diverged env steps, [1] env steps whose contact list overflowed
  const int* order;          // env of launch slot j (nullptr: identity)
  int *bin_cnt, *bin_items;  // [NBIN], [NBIN][n]: where this launch files its envs (nullptr: not filed)
  float *slot_qpos, *slot_task, *slot_obs; // [2][n][QPAD | USIM_TASK_DIM | SLOT_OBS]
  int *req_list, *req_cnt;         // (env, episode number) pairs to prepare, appended by this launch
  const int *prep_items, *prep_n;  // prepare mode: the requests this launch works through
  unsigned long long* trace;       // developer trace (USIM_TRACE): per env (start ns, end ns, SM id) of the launch, nullptr: off
  int* queue;                      // persistent launch (grid = resident CTAs): next launch slot, fetched with atomicAdd (nullptr: item = blockIdx.x + k gridDim.x)
  float* crec_out;                 // contact record [n][DEV_MAXC][CREC_DIM] (rows c < ncon), nullptr: recording off (usim_set_contact_record)
};
// one contact of the record: point (world), normal (geom1 -> geom2), world force on geom2 -- usim_get_contact_forces turns it into
// MuJoCo's contact frame and frame-coordinate force
#define CREC_DIM 9

// Contact record of one env (rows c < ncon): point, normal, cone_force of the final j -- every exit of the CG loop follows an
// update_grad on the final cjar (the line search moves cjar right before it), so these are the forces the probe wrench was summed
// from.  Runs after K9 and reads only shared memory; not inlined, so that the solve kernel's register allocation and schedule (the CG
// loop instruction for instruction) stay those of the kernel without the record.  A diverged env records zero forces, as K9 zeroes
// its cfrc: a non-finite solution (the x norm of the divergence guard, in rq) or probe wrench -- a non-finite arm state ends up in both.
__device__ __noinline__ void record_contacts(const WS& w, float* rec, int ncon, int tid) {
  const bool zero = !isfinite(rd(w.rq, 0)) || !isfinite(rd(w.rg, 6) + rd(w.rg, 7) + rd(w.rg, 8));
#pragma unroll 1
  for (int c = tid; c < ncon; c += NT) {
    int zone;
    float fr, mu, Dn = w.cD[c];
    contact_params(w.ctype[c], fr, mu);
    const v3 nn = mk(w.cn[0][c], w.cn[1][c], w.cn[2][c]);
    const v3 Fw = zero ? mk(0, 0, 0) : cone_force(mk(w.cjar[0][c], w.cjar[1][c], w.cjar[2][c]), nn, Dn, Dn * dm.impratio, mu, fr, zone);
    float* r = rec + (size_t)c * CREC_DIM;
    r[0] = w.cpos[0][c]; r[1] = w.cpos[1][c]; r[2] = w.cpos[2][c];
    r[3] = nn.x; r[4] = nn.y; r[5] = nn.z;
    r[6] = Fw.x; r[7] = Fw.y; r[8] = Fw.z;
  }
}

__global__ void __launch_bounds__(NT, MINB) solve_kernel(const SolveArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
  const int n = a.n, mode = a.mode;
  const PartTables pt = a.pt;
  const int2* __restrict__ eq_pairs = a.eq_pairs;
  WS& w = *reinterpret_cast<WS*>(smem_raw);
  static_assert(offsetof(WS, qrow) % 16 == 0 && offsetof(WS, x) % 16 == 0 && offsetof(WS, hs) % 16 == 0 && offsetof(WS, ab) % 16 == 0 &&
                    offsetof(WS, ts) % 16 == 0 && (QPAD * 4) % 16 == 0 && (ARMBUF * 4) % 16 == 0 && (USIM_TASK_DIM * 4) % 16 == 0,
                "TMA bulk copies need 16-byte aligned rows");
  if (tid == 0) mbar_init(&w.bar, 1);
  env_sync();
  unsigned phase = 0;
  const int nitems = a.prep ? *a.prep_n : n;
  // one trip per CTA for the env step (grid = n); the prepare launch walks its request list with a small fixed grid
#pragma unroll 1
  for (int item = blockIdx.x;; item += gridDim.x) {
  if (a.queue) { // dynamic hand-out in launch order (longest solves first): a CTA that finishes early takes the next slot
    if (tid == 0) w.item = atomicAdd(a.queue, 1);
    env_sync();
    item = w.item;
  }
  if (item >= nitems) break;
#if USIM_TRACE
  if (a.trace && tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(w.t0));
#endif
  int env = item;
  float *qp_g, *qv_g, *wm_g, *ts_g, *obs_row;
  const float* ab_g;
  if (a.prep) {
    env = a.prep_items[2 * item];
    const size_t row = (size_t)(a.prep_items[2 * item + 1] & 1) * n + env;
    qp_g = a.slot_qpos + row * QPAD; qv_g = nullptr; wm_g = nullptr; // a reset state is at rest: velocity and warm start are zero
    ts_g = a.slot_task + row * USIM_TASK_DIM;
    ab_g = a.armbuf + (size_t)item * ARMBUF;
    obs_row = a.slot_obs + row * SLOT_OBS;
  } else {
    if (a.order) env = a.order[item];
    if (a.mask && !a.mask[env]) continue;
    qp_g = a.qpos + (size_t)env * QPAD; qv_g = a.qvel + (size_t)env * QPAD; wm_g = a.warm + (size_t)env * QPAD;
    ts_g = a.task + (size_t)env * USIM_TASK_DIM;
    ab_g = a.armbuf + (size_t)env * ARMBUF;
    obs_row = a.obs ? a.obs + (size_t)env * USIM_OBS_DIM : nullptr;
  }
  if (mode != 1 && ts_g[USIM_TS_DONE] != 0.f) { // terminated env: frozen until reset; it keeps its place in the launch order
    if (tid == 0 && a.bin_cnt) a.bin_items[atomicAdd(a.bin_cnt, 1)] = env;
    continue;
  }
  const int np = dm.soft ? dm.npart : 0;
  const int nv = 7 + (dm.soft ? 6 + np : 0);
  const float h = dm.h;

  // ------------------------------------------------------------------ load: five TMA bulk copies, one mbarrier
  if (tid == 0) {
    mbar_expect_tx(&w.bar, ((qv_g ? 3 : 1) * QPAD + ARMBUF + USIM_TASK_DIM) * 4);
    tma_load_row(w.qrow, qp_g, QPAD * 4, &w.bar);
    if (qv_g) {
      tma_load_row(w.x, wm_g, QPAD * 4, &w.bar);
      tma_load_row(w.hs, qv_g, QPAD * 4, &w.bar);
    }
    tma_load_row(w.ab, ab_g, ARMBUF * 4, &w.bar);
    tma_load_row(w.ts, ts_g, USIM_TASK_DIM * 4, &w.bar);
  }
  // (overlapped with the copies)
  for (int i = tid; i < QPAD; i += NT) { w.grad[i] = 0.f; w.pg[i] = 0.f; w.s[i] = 0.f; }
  if (!qv_g)
    for (int i = tid; i < QPAD; i += NT) { w.x[i] = 0.f; w.hs[i] = 0.f; }
  for (int i = tid; i < np; i += NT) { w.cslot[i] = -1; w.cslot2[i] = -1; }
  for (int i = tid; i < 49; i += NT) w.Sf[i] = (i % 8 == 0) ? 1.f : 0.f; // identity: row/col 6 of the padded 6x6 stay like this
  mbar_wait(&w.bar, phase);
  phase ^= 1;
  if (!qv_g) env_sync(); // the zero rows above were written by plain stores of other threads (racecheck), not by the bulk copies the wait orders
  for (int i = nv + tid; i < QPAD; i += NT) w.x[i] = 0.f; // the solver vectors are zero beyond nv
  if (tid < 7) {
    w.qdarm[tid] = w.hs[tid];
#if ARM_SHIFT
#ifdef ARM_SHIFT_SCALE // developer knob: damped shift (in contact M^-1 over-estimates the response of the arm)
    if (mode != 1) w.x[tid] += ARM_SHIFT_SCALE * w.ab[AB_DX + tid];
#else
    if (mode != 1) w.x[tid] += w.ab[AB_DX + tid]; // warm start of the arm follows the change of its applied force (arm kernel)
#endif
#endif
  }
  float quat[4] = {1, 0, 0, 0};
  if (dm.soft) {
    if (tid < 6) w.vf[tid] = w.hs[7 + tid];
    if (tid < 3) w.p[tid] = w.qrow[7 + tid];
    quat[0] = w.qrow[10]; quat[1] = w.qrow[11]; quat[2] = w.qrow[12]; quat[3] = w.qrow[13];
    float nq = rsqrtf(quat[0] * quat[0] + quat[1] * quat[1] + quat[2] * quat[2] + quat[3] * quat[3]);
    quat[0] *= nq; quat[1] *= nq; quat[2] *= nq; quat[3] *= nq;
    if (tid == 0) quat2mat(quat, w.R);
  }
  env_sync();
  const float off = dm.cap_r + dm.cap_hl;
  const v3 site = ld3(w.ab + AB_EEFPOS), ptip = ld3(w.ab + AB_PTIP), pback = ld3(w.ab + AB_PBACK);
  float R[9];
  v3 P = mk(0, 0, 0), vlin = mk(0, 0, 0), wl = mk(0, 0, 0), ww = mk(0, 0, 0);
  if (dm.soft) {
#pragma unroll
    for (int i = 0; i < 9; i++) R[i] = w.R[i];
    P = ld3(w.p); vlin = ld3(w.vf); wl = ld3(w.vf + 3); ww = mv(R, wl);
  }
  const float mp = dm.part_mass;
  // slider sums of the current search direction (or of x for the warm-start pass): sum_i v_i and m sum_i a_i v_i (torso frame)
  float S4[4] = {0.f, 0.f, 0.f, 0.f};

  // ------------------------------------------------------------------ K3: torso inertia + bias, equality parameters
  const float ksm = -w.ts[USIM_TS_STIFFNESS], bsm = -w.ts[USIM_TS_DAMPING];
  if (dm.soft) {
    v3 gl = mtv(R, ld3(dm.g));
    // [0..2] m c, [3..5] F, [6..8] T, [9..14] parallel-axis inertia, [15] sum q, [16] sum qdot, [17] sum x, [18..20] m sum a x
    float a[21];
#pragma unroll
    for (int k = 0; k < 21; k++) a[k] = 0.f;
    for (int i = tid; i < np; i += NT) {
      const float4 a4 = pt.ax4[i];
      v3 ah = xyz(a4), r0 = xyz(pt.ps4[i]);
      float q = w.qrow[14 + i], sd = w.hs[13 + i], xi = w.x[13 + i];
      v3 c = r0 + (q - off) * ah;
      a[0] += mp * c.x; a[1] += mp * c.y; a[2] += mp * c.z;
      float cc = dot(c, c);
      a[9] += mp * (cc - c.x * c.x); a[10] += mp * (cc - c.y * c.y); a[11] += mp * (cc - c.z * c.z);
      a[12] -= mp * c.x * c.y; a[13] -= mp * c.x * c.z; a[14] -= mp * c.y * c.z;
      v3 avp = cross(wl, cross(wl, c)) + 2.f * sd * cross(wl, ah);
      v3 F = mp * (avp - gl);
      v3 T = cross(c, F);
      a[3] += F.x; a[4] += F.y; a[5] += F.z; a[6] += T.x; a[7] += T.y; a[8] += T.z;
      a[15] += q; a[16] += sd;
      a[17] += xi; a[18] += mp * ah.x * xi; a[19] += mp * ah.y * xi; a[20] += mp * ah.z * xi;
      // "fix" equality of this slider
      float K, B, imp;
      kbi(dm.solref[0], dm.solref[1], q, &K, &B, &imp);
      float D = 1.f / fmaxf(1e-15f, (1.f - imp) / imp * a4.w);
      w.dgm[i] = mp + D;
      w.grad[13 + i] = -dot(ah, F) + D * (-B * sd - K * imp * q);
    }
    tsum_to(a, lane, w.r3[wrp]);
    env_sync();
    // tendon equality: sum q = 0
    const float a_q = rd(w.r3, 15), a_v = rd(w.r3, 16);
    S4[0] = rd(w.r3, 17); S4[1] = rd(w.r3, 18); S4[2] = rd(w.r3, 19); S4[3] = rd(w.r3, 20);
    float K, B, imp;
    kbi(dm.solref[0], dm.solref[1], a_q, &K, &B, &imp);
    const float Dt = 1.f / fmaxf(1e-15f, (1.f - imp) / imp * dm.tendon_iw);
    const float areft = -B * a_v - K * imp * a_q;
    if (tid == 0) {
      const float mtot = np * mp + dm.center_mass;
      float t15[15];
#pragma unroll
      for (int k = 0; k < 15; k++) t15[k] = rd(w.r3, k);
      const v3 mc = ld3(t15);
      w.Dt = Dt; w.areft = areft;
      // M_ff: [v (world); omega (body)]
      // rotational inertia: parallel-axis part (depends on q) + constant part (capsules about their COM, centre geom)
      float It[9] = {t15[9] + dm.rot_I[0],  t15[12] + dm.rot_I[3], t15[13] + dm.rot_I[4], t15[12] + dm.rot_I[3], t15[10] + dm.rot_I[1],
                     t15[14] + dm.rot_I[5], t15[13] + dm.rot_I[4], t15[14] + dm.rot_I[5], t15[11] + dm.rot_I[2]};
      for (int k = 0; k < 36; k++) w.Mff[k] = 0.f;
      for (int k = 0; k < 3; k++) w.Mff[k * 6 + k] = mtot;
      // M_v,omega = -R [mc]x  ;  [mc]x = [[0,-z,y],[z,0,-x],[-y,x,0]]
      float X[9] = {0, -mc.z, mc.y, mc.z, 0, -mc.x, -mc.y, mc.x, 0}, RX[9];
      mm3(R, X, RX);
      for (int r = 0; r < 3; r++)
        for (int b = 0; b < 3; b++) { w.Mff[r * 6 + 3 + b] = -RX[3 * r + b]; w.Mff[(3 + b) * 6 + r] = -RX[3 * r + b]; }
      for (int r = 0; r < 3; r++)
        for (int b = 0; b < 3; b++) w.Mff[(3 + r) * 6 + 3 + b] = It[3 * r + b];
      // the same block with a WORLD-frame angular velocity (what the preconditioner works in): -[R mc]x and R I R^T
      {
        v3 rm = mv(R, mc);
        float RI[9], Iw[9], Rt[9] = {R[0], R[3], R[6], R[1], R[4], R[7], R[2], R[5], R[8]};
        mm3(R, It, RI);
        mm3(RI, Rt, Iw);
        float* M = w.Mfw;
        M[tri6(0, 0)] = mtot; M[tri6(0, 1)] = 0.f; M[tri6(0, 2)] = 0.f; M[tri6(1, 1)] = mtot; M[tri6(1, 2)] = 0.f; M[tri6(2, 2)] = mtot;
        M[tri6(0, 3)] = 0.f;   M[tri6(0, 4)] = rm.z;  M[tri6(0, 5)] = -rm.y;
        M[tri6(1, 3)] = -rm.z; M[tri6(1, 4)] = 0.f;   M[tri6(1, 5)] = rm.x;
        M[tri6(2, 3)] = rm.y;  M[tri6(2, 4)] = -rm.x; M[tri6(2, 5)] = 0.f;
        M[tri6(3, 3)] = Iw[0]; M[tri6(3, 4)] = Iw[1]; M[tri6(3, 5)] = Iw[2]; M[tri6(4, 4)] = Iw[4]; M[tri6(4, 5)] = Iw[5]; M[tri6(5, 5)] = Iw[8];
      }
      // bias of the free body
      v3 sF = ld3(t15 + 3), sT = ld3(t15 + 6);
      v3 bv = mv(R, sF) - dm.center_mass * ld3(dm.g);
      v3 Iw = symv(dm.rot_I, wl);
      v3 bw = sT + cross(wl, Iw);
      w.grad[7] = -bv.x - dm.free_damp * vlin.x; w.grad[8] = -bv.y - dm.free_damp * vlin.y; w.grad[9] = -bv.z - dm.free_damp * vlin.z;
      w.grad[10] = -bw.x - dm.free_damp * wl.x; w.grad[11] = -bw.y - dm.free_damp * wl.y; w.grad[12] = -bw.z - dm.free_damp * wl.z;
    }
    env_sync();
    // "smooth" pair equalities (carry solrefsmooth = (-stiffness, -damping) of this episode); scratch: pg|s (contiguous, unused so far)
    float* arp = w.pg;
    for (int pr = tid; pr < dm.npair; pr += NT) {
      const int2 pr2 = eq_pairs[pr];
      const int ia = pr2.x, ib = pr2.y;
      float pos = w.qrow[14 + ia] - w.qrow[14 + ib], vel = w.hs[13 + ia] - w.hs[13 + ib], K2, B2, imp2;
      kbi(ksm, bsm, pos, &K2, &B2, &imp2);
      float D = 1.f / fmaxf(1e-15f, (1.f - imp2) / imp2 * (pt.ax4[ia].w + pt.ax4[ib].w));
      w.Dp[pr] = D;
      arp[pr] = D * (-B2 * vel - K2 * imp2 * pos); // D aref of the pair row: + on its first slider, - on its second
      if (pr == 0) { w.Dp[dm.npair] = 0.f; arp[dm.npair] = 0.f; } // the slot empty neighbour entries point at
    }
    env_sync();
    // every slider gathers its (at most 4) pair rows in table order: no atomics, the same sum in any thread arrangement
    for (int i = tid; i < np; i += NT) {
      const int4 e = pt.nb4[i];
      float sd = w.Dp[e.x >> 16] + w.Dp[e.y >> 16] + w.Dp[e.z >> 16] + w.Dp[e.w >> 16];
      float sa = ((e.x & 0x8000) ? -arp[e.x >> 16] : arp[e.x >> 16]) + ((e.y & 0x8000) ? -arp[e.y >> 16] : arp[e.y >> 16]) +
                 ((e.z & 0x8000) ? -arp[e.z >> 16] : arp[e.z >> 16]) + ((e.w & 0x8000) ? -arp[e.w >> 16] : arp[e.w >> 16]);
      w.grad[13 + i] += Dt * areft + sa;
      w.dgm[i] += sd;
    }
    env_sync();
    for (int i = tid; i < 2 * QPAD; i += NT) arp[i] = 0.f; // pg and s start the solve as zero vectors
  }
  if (tid < 7) {
    w.grad[lane] = w.ab[AB_QS + lane];
    // joint limits (margin 0)
    float q = w.qrow[lane], lo = dm.jnt_lo[lane], hi = dm.jnt_hi[lane], dist = 0.f, sg = 0.f;
    if (q - lo < 0.f) { dist = q - lo; sg = 1.f; } else if (hi - q < 0.f) { dist = hi - q; sg = -1.f; }
    float K, B, imp;
    kbi(dm.solref[0], dm.solref[1], dist, &K, &B, &imp);
    w.lsign[lane] = sg;
    w.lD[lane] = 1.f / fmaxf(1e-15f, (1.f - imp) / imp * dm.iw_arm[lane]);
    w.laref[lane] = -B * sg * w.qdarm[tid] - K * imp * dist;
  }
  env_sync();

  // ------------------------------------------------------------------ K4: collision, MuJoCo contact order
  int ncon = 0;
  { // (table, probe): geom1 = table, geom2 = probe
    if (tid == 0) {
      v3 ends[2] = {ptip, pback};
      for (int e = 0; e < 2; e++) {
        float dist = ends[e].z - dm.probe_r - dm.table_z;
        if (dist < 0.f && fabsf(ends[e].x) <= dm.table_half && fabsf(ends[e].y) <= dm.table_half) {
          w.cpos[0][ncon] = ends[e].x; w.cpos[1][ncon] = ends[e].y; w.cpos[2][ncon] = dm.table_z + 0.5f * dist;
          w.cn[0][ncon] = 0.f; w.cn[1][ncon] = 0.f; w.cn[2][ncon] = 1.f;
          w.cfs[ncon] = dist; w.cpart[ncon] = -1; w.ctype[ncon] = 2;
          ncon++;
        }
      }
    }
    if (tid == 0) w.ncon = ncon;
    env_sync();
    ncon = w.ncon;
  }
  if (dm.soft) {
    const unsigned lt = (1u << lane) - 1u;
    int cphase = 0;
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) { // pass 0: (table, particle k); pass 1: (probe, particle k)
      for (int base = 0; base < np; base += NT) {
        int i = base + tid;
        bool h0 = false, h1 = false;
        v3 p0 = mk(0, 0, 0), p1 = mk(0, 0, 0), n0 = mk(0, 0, -1);
        float d0 = 0.f, d1 = 0.f;
        if (i < np) {
          v3 ah = xyz(pt.ax4[i]), r0 = xyz(pt.ps4[i]);
          float q = w.qrow[14 + i];
          v3 eo = P + mv(R, r0 + (q - dm.cap_r) * ah), ei = P + mv(R, r0 + (q - dm.cap_r - 2.f * dm.cap_hl) * ah);
          if (pass == 0) {
            d0 = eo.z - dm.cap_r - dm.table_z;
            h0 = d0 < 0.f && fabsf(eo.x) <= dm.table_half && fabsf(eo.y) <= dm.table_half;
            p0 = mk(eo.x, eo.y, dm.table_z + 0.5f * d0);
            d1 = ei.z - dm.cap_r - dm.table_z;
            h1 = d1 < 0.f && fabsf(ei.x) <= dm.table_half && fabsf(ei.y) <= dm.table_half;
            p1 = mk(ei.x, ei.y, dm.table_z + 0.5f * d1);
          } else {
            v3 c1, c2;
            seg_seg(eo, ei, ptip, pback, c1, c2);
            v3 d = c2 - c1;
            float len = norm(d);
            d0 = len - dm.cap_r - dm.probe_r;
            h0 = d0 < 0.f;
            n0 = len > 1e-12f ? (1.f / len) * d : mk(0, 0, 1);
            p0 = c1 + (dm.cap_r + 0.5f * d0) * n0;
          }
        }
        unsigned b0 = __ballot_sync(0xffffffffu, h0), b1 = __ballot_sync(0xffffffffu, h1);
        int before = 0, total = __popc(b0) + __popc(b1);
        if (WPE > 1) { // cross-warp exclusive prefix of the per-warp hit counts (keeps the particle order)
          int* cb = w.cnt[cphase];
          cphase ^= 1;
          if (lane == 0) cb[wrp] = total;
          __syncthreads();
          total = 0;
#pragma unroll
          for (int q = 0; q < WPE; q++) { if (q < wrp) before += cb[q]; total += cb[q]; }
        }
        int slot = ncon + before + __popc(b0 & lt) + __popc(b1 & lt);
        // owner slot of the slider: its first contact (the same thread handles slider i in both passes)
        if ((h0 || h1) && slot < DEV_MAXC && w.cslot[i] < 0) w.cslot[i] = (short)slot;
        if (pass == 1 && h0 && slot < DEV_MAXC) w.cslot2[i] = (short)slot;
        if (h0 && slot < DEV_MAXC) {
          w.cpos[0][slot] = p0.x; w.cpos[1][slot] = p0.y; w.cpos[2][slot] = p0.z;
          w.cn[0][slot] = n0.x; w.cn[1][slot] = n0.y; w.cn[2][slot] = n0.z;
          w.cfs[slot] = d0; w.cpart[slot] = (short)i; w.ctype[slot] = (unsigned char)pass;
        }
        if (h0) slot++;
        if (h1 && slot < DEV_MAXC) {
          w.cpos[0][slot] = p1.x; w.cpos[1][slot] = p1.y; w.cpos[2][slot] = p1.z;
          w.cn[0][slot] = 0.f; w.cn[1][slot] = 0.f; w.cn[2][slot] = -1.f;
          w.cfs[slot] = d1; w.cpart[slot] = (short)i; w.ctype[slot] = 0;
        }
        ncon += total;
      }
    }
  }
  const int ncon_found = ncon;
  if (ncon > DEV_MAXC) { // contacts beyond the cap are dropped: counted, never silent (usim_contact_overflow_count)
    ncon = DEV_MAXC;
    if (tid == 0 && a.counters) atomicAdd(a.counters + 1, 1);
  }
  env_sync();

  // ------------------------------------------------------------------ K5: contact parameters (aref, D)
  v3 Vs, Ws; // site velocity (linear, angular)
  {
    float s6[6];
#pragma unroll
    for (int r = 0; r < 6; r++) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 7; j++) s += w.ab[AB_JSITE + r * 7 + j] * w.qdarm[j];
      s6[r] = s;
    }
    Vs = mk(s6[0], s6[1], s6[2]); Ws = mk(s6[3], s6[4], s6[5]);
  }
  for (int c = tid; c < ncon; c += NT) {
    int type = w.ctype[c], i = w.cpart[c];
    v3 pos = mk(w.cpos[0][c], w.cpos[1][c], w.cpos[2][c]), nn = mk(w.cn[0][c], w.cn[1][c], w.cn[2][c]);
    v3 rel = mk(0, 0, 0);
    float diagA = 0.f;
    if (type != 2) {
      v3 aw = mv(R, xyz(pt.ax4[i]));
      rel = rel - (vlin + cross(ww, pos - P) + w.hs[13 + i] * aw);
      diagA += pt.ps4[i].w;
    }
    if (type != 0) { rel = rel + Vs + cross(Ws, pos - site); diagA += dm.iw_probe; }
    float K, B, imp;
    kbi(dm.solref[0], dm.solref[1], w.cfs[c], &K, &B, &imp);
    w.cD[c] = 1.f / fmaxf(1e-15f, (1.f - imp) / imp * diagA);
    // aref = -B v_rel - K imp dist n: the normal row carries the position term, the tangential rows only damping
    v3 ar = (-B) * rel - (K * imp * w.cfs[c]) * nn;
    w.cjv[0][c] = ar.x; w.cjv[1][c] = ar.y; w.cjv[2][c] = ar.z;
    w.czone[c] = 255; // "unknown": the first gradient evaluation always reports a change
    if (a.dist_out) a.dist_out[(size_t)env * DEV_MAXC + c] = w.cfs[c]; // the depth leaves here: cfs becomes scratch
  }
  env_sync();

  float gnorm = 0.f, rhsn = 0.f, hxn = 0.f; // |grad|, |rhs|, |Hx| of the current iterate
  // ------------------------------------------------------------------ helpers (lambdas over the warp)
  // out = (M + E) in, in ONE pass: the two slider sums of `in` it needs (S4) are produced by whoever produced `in`.
  // With q != nullptr also accumulates q[0] += in.Hx, q[1] += in.out (this lane's share).
  auto applyH = [&](const float* in, float* out, float* q) {
    if (dm.soft) {
      const v3 ivl = mtv(R, ld3(in + 7)); // R^T in_v
      const float Dt = w.Dt, dts = Dt * S4[0];
      PRAGMA_HOT_S
      for (int i = tid; i < np; i += NT) {
        float xi = in[13 + i];
        v3 ah = xyz(pt.ax4[i]);
        // 4 packed (pair << 16 | neighbour) entries in one 16-byte load, no data-dependent branch
        const int4 e = pt.nb4[i];
        float acc = mp * dot(ah, ivl) + w.dgm[i] * xi + dts;
        acc -= w.Dp[e.x >> 16] * in[13 + (e.x & 0x7fff)]; acc -= w.Dp[e.y >> 16] * in[13 + (e.y & 0x7fff)];
        acc -= w.Dp[e.z >> 16] * in[13 + (e.z & 0x7fff)]; acc -= w.Dp[e.w >> 16] * in[13 + (e.w & 0x7fff)];
        out[13 + i] = acc;
        if (q) { q[0] += xi * w.Hx[13 + i]; q[1] += xi * acc; }
      }
    }
    if (tid < 13) {
      float s = 0.f;
      if (tid < 7) {
#pragma unroll
        for (int j = 0; j < 7; j++) s += w.ab[AB_M + lane * 7 + j] * in[j];
      } else if (dm.soft) {
        int r = lane - 7;
#pragma unroll
        for (int c = 0; c < 6; c++) s += w.Mff[r * 6 + c] * in[7 + c];
        if (r < 3) s += w.R[3 * r] * S4[1] + w.R[3 * r + 1] * S4[2] + w.R[3 * r + 2] * S4[3];
      }
      if (tid < 7 || dm.soft) {
        out[lane] = s;
        if (q) { q[0] += in[lane] * w.Hx[lane]; q[1] += in[lane] * s; }
      }
    }
    // dv[0..5] = Jsite in_arm ; dv[6..8] = in_v ; dv[9..11] = R in_omega
    // (done by the LAST warp of the env: the dense rows above belong to the first)
    const int dl = tid - (NT - 16);
    if (dl >= 0 && dl < 6) {
      int r = dl;
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 7; j++) s += w.ab[AB_JSITE + r * 7 + j] * in[j];
      w.dv[r] = s;
    } else if (dl >= 6 && dl < 9) {
      w.dv[dl] = dm.soft ? in[7 + dl - 6] : 0.f;
    } else if (dl >= 9 && dl < 12) {
      int r = dl - 9;
      w.dv[9 + r] = dm.soft ? w.R[3 * r] * in[10] + w.R[3 * r + 1] * in[11] + w.R[3 * r + 2] * in[12] : 0.f;
    }
    env_sync();
  };
  // out[.][c] = relative acceleration of the contact point pair (geom2 - geom1) as a WORLD vector, i.e. the 3 rows of J in
  // before projection on the contact frame (needs dv of `in`, written by applyH)
  auto contactJ = [&](const float* in, float (*out)[DEV_MAXC], bool sub_aref) {
    v3 V = ld3(w.dv), W = ld3(w.dv + 3), iv = ld3(w.dv + 6), iw = ld3(w.dv + 9);
    PRAGMA_HOT
    for (int c = tid; c < ncon; c += NT) {
      int type = w.ctype[c], i = w.cpart[c];
      v3 pos = mk(w.cpos[0][c], w.cpos[1][c], w.cpos[2][c]);
      v3 rel = mk(0, 0, 0);
      if (type != 2) rel = rel - (iv + cross(iw, pos - P) + in[13 + i] * mv(R, xyz(pt.ax4[i])));
      if (type != 0) rel = rel + V + cross(W, pos - site);
      if (sub_aref) rel = rel - mk(w.cjv[0][c], w.cjv[1][c], w.cjv[2][c]);
      out[0][c] = rel.x; out[1][c] = rel.y; out[2][c] = rel.z;
    }
    // (no barrier: every per-contact loop of the solve maps contact c to the same thread, which is the only reader of out[.][c]
    // until the next one)
  };
  // sum of a per-contact quantity over the contacts of slider i, called by its owner slot c: the second table contact sits in
  // the next slot, the probe contact (if any, and if it is not the owner itself) in cslot2
  auto slider_gather = [&](const float* v, int c, int i) -> float {
    float f = v[c];
    if (w.ctype[c] == 0 && c + 1 < ncon && w.cpart[c + 1] == i && w.ctype[c + 1] == 0) f += v[c + 1];
    const int c2 = w.cslot2[i];
    if (c2 >= 0 && c2 != c) f += v[c2];
    return f;
  };
  // grad (= Hx on entry) -= J^T f(jar).  Lands in w.rg: [0..5] torso wrench about P, [6..11] probe wrench about the site,
  // [12] zone changes, [13] hx2, [14] rhs2 (the caller's two riders).
  auto update_grad = [&](float hx2, float rhs2) {
    float g[15];
#pragma unroll
    for (int k = 0; k < 15; k++) g[k] = 0.f;
    g[13] = hx2; g[14] = rhs2;
    PRAGMA_HOT
    for (int c = tid; c < ncon; c += NT) {
      int type = w.ctype[c], i = w.cpart[c], zone;
      float fr, mu, Dn = w.cD[c];
      contact_params(type, fr, mu);
      const v3 nn = mk(w.cn[0][c], w.cn[1][c], w.cn[2][c]);
      const v3 Fw = cone_force(mk(w.cjar[0][c], w.cjar[1][c], w.cjar[2][c]), nn, Dn, Dn * dm.impratio, mu, fr, zone); // force on geom2
      if (zone != (int)w.czone[c]) g[12] += 1.f;
      w.czone[c] = (unsigned char)zone;
      w.cfs[c] = 0.f;
      if (zone == 0) continue;
      const v3 pos = mk(w.cpos[0][c], w.cpos[1][c], w.cpos[2][c]);
      if (type != 2) {
        v3 Fp = -Fw, T = cross(pos - P, Fp);
        g[0] += Fp.x; g[1] += Fp.y; g[2] += Fp.z; g[3] += T.x; g[4] += T.y; g[5] += T.z;
        w.cfs[c] = -dot(mv(R, xyz(pt.ax4[i])), Fp); // this contact's share of its slider's row, gathered by the owner below
      }
      if (type != 0) {
        v3 T = cross(pos - site, Fw);
        g[6] += Fw.x; g[7] += Fw.y; g[8] += Fw.z; g[9] += T.x; g[10] += T.y; g[11] += T.z;
      }
    }
    tsum_to(g, lane, w.rg[wrp]);
    env_sync();
    // slider rows: the owner contact of each slider adds the shares of its (at most 3) contacts in slot order -- no atomics
    PRAGMA_HOT
    for (int c = tid; c < ncon; c += NT) {
      const int i = w.cpart[c];
      if (i >= 0 && w.cslot[i] == c) w.grad[13 + i] += slider_gather(w.cfs, c, i);
    }
    if (tid < 7) {
      float s = 0.f;
#pragma unroll
      for (int r = 0; r < 6; r++) s += w.ab[AB_JSITE + r * 7 + lane] * rd(w.rg, 6 + r);
      // joint limit row
      float sg = w.lsign[lane];
      if (sg != 0.f) {
        float jar = sg * w.x[lane] - w.laref[lane];
        if (jar < 0.f) s += sg * (-w.lD[lane] * jar);
      }
      w.grad[lane] -= s;
    } else if (tid < 10 && dm.soft) {
      w.grad[lane] -= rd(w.rg, lane - 7);
    } else if (tid < 13 && dm.soft) {
      int r = lane - 10; // R^T torque
      w.grad[lane] -= w.R[r] * rd(w.rg, 3) + w.R[3 + r] * rd(w.rg, 4) + w.R[6 + r] * rd(w.rg, 5);
    }
    env_sync();
  };
  // pg = P^-1 grad  (arm: dense 7x7 Cholesky; torso: arrow with the 6x6 Schur complement, solved with a WORLD-frame angular part).
  // A slider without contacts couples to the free body through m a_i only; the few with contacts add their owner slot's (K a, r x K a).
  // Lands in w.rp: [9] = grad.pg_old, [10] = |grad|^2 (the convergence test: returns false when the solve has converged, before
  // the solves and the stencil passes) and in w.rq: [0] grad.pg, [2..5] the slider sums of pg (the next S4).
  auto precond = [&]() -> bool {
    float a[11];
#pragma unroll
    for (int k = 0; k < 11; k++) a[k] = 0.f;
    PRAGMA_HOT_S
    for (int i = tid; i < np; i += NT) {
      float g = w.grad[13 + i], gi = g * w.dg[i];
      v3 ah = xyz(pt.ax4[i]);
      a[0] += ah.x * gi; a[1] += ah.y * gi; a[2] += ah.z * gi;
      a[9] += g * w.pg[13 + i];
      a[10] += g * g;
      w.hs[13 + i] = gi; // hs is free between the line search and the next applyH
      int cs = w.cslot[i];
      if (cs >= 0) {
        a[3] += w.sk[0][cs] * gi; a[4] += w.sk[1][cs] * gi; a[5] += w.sk[2][cs] * gi;
        a[6] += w.sc[0][cs] * gi; a[7] += w.sc[1][cs] * gi; a[8] += w.sc[2][cs] * gi;
      }
    }
    if (tid < 13) { a[9] += w.grad[lane] * w.pg[lane]; a[10] += w.grad[lane] * w.grad[lane]; }
    tsum_to(a, lane, w.rp[wrp]);
    env_sync();
    // |grad| is known here: a converged solve stops before the solves, the stencil passes and the second reduction
    // (fp32 floor of the gradient is ~eps * (|Hx| + |rhs|): the terms that cancel in it)
    gnorm = sqrtf(rd(w.rp, 10));
    if (gnorm <= dm.tol * (1.f + rhsn + hxn)) return false;
#if WARP_SOLVE
    // dense blocks: the first warp solves both at once (arm 7x7 in lanes 0-6, torso 6x6 in lanes 8-13); the arm part goes straight to
    // pg, the torso part (world frame) to yS for everybody; the other warp goes ahead with the stencil pass, which needs neither
    if (wrp == 0) {
      const int k = lane & 7;
      float rhs = 0.f;
      if (lane < 7) rhs = w.grad[lane];
      else if (dm.soft && lane >= 8 && lane < 11) // gd[7+k] - (m R t[0:3] + t[3:6])_k
        rhs = w.grad[7 + k] - (mp * (w.R[3 * k] * rd(w.rp, 0) + w.R[3 * k + 1] * rd(w.rp, 1) + w.R[3 * k + 2] * rd(w.rp, 2)) + rd(w.rp, 3 + k));
      else if (dm.soft && lane >= 11 && lane < 14) // (R gd[10:13])_k - t[6:9]_k
        rhs = w.R[3 * (k - 3)] * w.grad[10] + w.R[3 * (k - 3) + 1] * w.grad[11] + w.R[3 * (k - 3) + 2] * w.grad[12] - rd(w.rp, 3 + k);
      const float sol = chol7_solve_warp2(w.Pa, w.Sf, rhs, lane);
      if (lane < 7) w.pg[lane] = sol;
      else if (lane >= 8 && lane < 14) w.yS[k] = dm.soft ? sol : 0.f;
    }
    float b[6] = {0, 0, 0, 0, 0, 0};
#else
    float y[6] = {0, 0, 0, 0, 0, 0};
    v3 yl = mk(0, 0, 0), yb = mk(0, 0, 0);
    float b[6] = {0, 0, 0, 0, 0, 0};
#if SPLIT_DENSE
    if (wrp == 0) { // arm block
      float ga[7], ya[7];
#pragma unroll
      for (int j = 0; j < 7; j++) { ga[j] = w.grad[j]; ya[j] = ga[j]; }
      chol7_solve<7>(w.Pa, ya);
      if (tid == 0) {
#pragma unroll
        for (int j = 0; j < 7; j++) { w.pg[j] = ya[j]; b[0] += ga[j] * ya[j]; }
      }
    } else { // torso block (world frame), for everybody through yS
      if (dm.soft) {
        float gt[6], t9[9];
#pragma unroll
        for (int k = 0; k < 6; k++) gt[k] = w.grad[7 + k];
#pragma unroll
        for (int k = 0; k < 9; k++) t9[k] = rd(w.rp, k);
        v3 tv = mp * mv(R, ld3(t9)) + ld3(t9 + 3), gw = mv(R, mk(gt[3], gt[4], gt[5])) - ld3(t9 + 6);
        y[0] = gt[0] - tv.x; y[1] = gt[1] - tv.y; y[2] = gt[2] - tv.z; y[3] = gw.x; y[4] = gw.y; y[5] = gw.z;
        chol7_solve<6>(w.Sf, y);
        yb = mtv(R, mk(y[3], y[4], y[5])); // back to the body frame
        if (lane == 0) {
          w.pg[7] = y[0]; w.pg[8] = y[1]; w.pg[9] = y[2]; w.pg[10] = yb.x; w.pg[11] = yb.y; w.pg[12] = yb.z;
          b[0] += gt[0] * y[0] + gt[1] * y[1] + gt[2] * y[2] + gt[3] * yb.x + gt[4] * yb.y + gt[5] * yb.z;
        }
      }
      if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) w.yS[k] = y[k];
      }
    }
    env_sync();
#pragma unroll
    for (int k = 0; k < 6; k++) y[k] = w.yS[k];
    yl = mtv(R, mk(y[0], y[1], y[2]));
#else
#if SPLIT_SOLVE
    if (wrp == 0) {
#endif
    float gd[13]; // dense part of the gradient
#pragma unroll
    for (int k = 0; k < 13; k++) gd[k] = w.grad[k];
    float ya[7];
#pragma unroll
    for (int j = 0; j < 7; j++) ya[j] = gd[j];
    chol7_solve<7>(w.Pa, ya);
    if (dm.soft) {
      float t9[9];
#pragma unroll
      for (int k = 0; k < 9; k++) t9[k] = rd(w.rp, k);
      v3 tv = mp * mv(R, ld3(t9)) + ld3(t9 + 3), gw = mv(R, mk(gd[10], gd[11], gd[12])) - ld3(t9 + 6);
      y[0] = gd[7] - tv.x; y[1] = gd[8] - tv.y; y[2] = gd[9] - tv.z; y[3] = gw.x; y[4] = gw.y; y[5] = gw.z;
      chol7_solve<6>(w.Sf, y);
      yl = mtv(R, mk(y[0], y[1], y[2]));
      yb = mtv(R, mk(y[3], y[4], y[5])); // back to the body frame
    }
    if (tid == 0) {
#pragma unroll
      for (int j = 0; j < 7; j++) { w.pg[j] = ya[j]; b[0] += gd[j] * ya[j]; }
      if (dm.soft) {
        w.pg[7] = y[0]; w.pg[8] = y[1]; w.pg[9] = y[2]; w.pg[10] = yb.x; w.pg[11] = yb.y; w.pg[12] = yb.z;
        b[0] += gd[7] * y[0] + gd[8] * y[1] + gd[9] * y[2] + gd[10] * yb.x + gd[11] * yb.y + gd[12] * yb.z;
      }
#if SPLIT_SOLVE
#pragma unroll
      for (int k = 0; k < 6; k++) w.yS[k] = y[k];
#endif
    }
#if SPLIT_SOLVE
    } // (first warp)
#endif
#endif // SPLIT_DENSE
#endif
#if PREC3
#if SPLIT_Z1
    if (wrp == 1) { // (the whole pass by the second warp, while the first one solves)
      PRAGMA_HOT_S
      for (int i = lane; i < np; i += 32) {
        const int4 e = pt.nb4[i];
        float nb = w.Dp[e.x >> 16] * w.hs[13 + (e.x & 0x7fff)] + w.Dp[e.y >> 16] * w.hs[13 + (e.y & 0x7fff)] +
                   w.Dp[e.z >> 16] * w.hs[13 + (e.z & 0x7fff)] + w.Dp[e.w >> 16] * w.hs[13 + (e.w & 0x7fff)];
        w.pg[13 + i] = nb * w.dg[i];
      }
    }
#else
    PRAGMA_HOT_S
    for (int i = tid; i < np; i += NT) {
      const int4 e = pt.nb4[i];
      float nb = w.Dp[e.x >> 16] * w.hs[13 + (e.x & 0x7fff)] + w.Dp[e.y >> 16] * w.hs[13 + (e.y & 0x7fff)] +
                 w.Dp[e.z >> 16] * w.hs[13 + (e.z & 0x7fff)] + w.Dp[e.w >> 16] * w.hs[13 + (e.w & 0x7fff)];
      w.pg[13 + i] = nb * w.dg[i];
    }
#endif
#endif
#if WARP_SOLVE || PREC3
    env_sync();
#endif
#if SPLIT_SOLVE
    // the dense solution of the first warp, for everybody
#pragma unroll
    for (int k = 0; k < 6; k++) y[k] = w.yS[k];
    yl = mtv(R, mk(y[0], y[1], y[2]));
#endif
#if WARP_SOLVE
    float y[6];
#pragma unroll
    for (int k = 0; k < 6; k++) y[k] = w.yS[k];
    const v3 yl = mtv(R, mk(y[0], y[1], y[2]));
    if (tid < 13) { // dense part of pg (the torso rotation goes back to the body frame) and its share of grad.pg
      float pgk;
      if (tid < 7) pgk = w.pg[tid];
      else if (tid < 10) pgk = y[0] * (tid == 7) + y[1] * (tid == 8) + y[2] * (tid == 9);
      else { const int c = tid - 10; pgk = w.R[c] * y[3] + w.R[3 + c] * y[4] + w.R[6 + c] * y[5]; }
      if (tid >= 7) w.pg[tid] = dm.soft ? pgk : 0.f;
      if (tid < 7 || dm.soft) b[0] += w.grad[tid] * pgk;
    }
#endif
    PRAGMA_HOT_S
    for (int i = tid; i < np; i += NT) {
      float g = w.grad[13 + i];
      v3 ah = xyz(pt.ax4[i]);
      float by = mp * dot(ah, yl);
      int cs = w.cslot[i];
      if (cs >= 0)
        by += w.sk[0][cs] * y[0] + w.sk[1][cs] * y[1] + w.sk[2][cs] * y[2] + w.sc[0][cs] * y[3] + w.sc[1][cs] * y[4] + w.sc[2][cs] * y[5];
      // slider block D - W (W: the pair couplings) inverted to second order, D^-1 + D^-1 W D^-1: hs holds D^-1 grad
      const int4 e = pt.nb4[i];
#if PREC3
      // third order with Chebyshev weights: z0 + c (z1 + z2), z1 = D^-1 W z0 (in pg), z2 = D^-1 W z1
      float nb = w.Dp[e.x >> 16] * w.pg[13 + (e.x & 0x7fff)] + w.Dp[e.y >> 16] * w.pg[13 + (e.y & 0x7fff)] +
                 w.Dp[e.z >> 16] * w.pg[13 + (e.z & 0x7fff)] + w.Dp[e.w >> 16] * w.pg[13 + (e.w & 0x7fff)];
      float p = w.hs[13 + i] + CHEB_C * (w.pg[13 + i] + nb * w.dg[i]) - by * w.dg[i];
      w.hs[13 + i] = p; // neighbours read pg in this pass, not hs
#else
#ifdef PREC_JACOBI // developer knob: diagonal slider block (no stencil pass at all)
      float nb = 0.f;
#else
      float nb = w.Dp[e.x >> 16] * w.hs[13 + (e.x & 0x7fff)] + w.Dp[e.y >> 16] * w.hs[13 + (e.y & 0x7fff)] +
                 w.Dp[e.z >> 16] * w.hs[13 + (e.z & 0x7fff)] + w.Dp[e.w >> 16] * w.hs[13 + (e.w & 0x7fff)];
#endif
#ifdef PREC2_C // developer knob: weight of the first-order term of the second-order slider block
      float p = w.hs[13 + i] + (PREC2_C * nb - by) * w.dg[i];
#else
      float p = w.hs[13 + i] + (nb - by) * w.dg[i];
#endif
      w.pg[13 + i] = p;
#endif
      b[0] += g * p; b[2] += p;
      b[3] += mp * ah.x * p; b[4] += mp * ah.y * p; b[5] += mp * ah.z * p;
    }
    tsum_to(b, lane, w.rq[wrp]);
    env_sync();
    return true;
  };

  // preconditioner from the current active set (contact zones); rebuilt when the zones change.  Runs 1-3 times per solve.
  auto build_precond = [&]() {
#pragma unroll 1
    for (int i = tid; i < np; i += NT) w.dg[i] = w.dgm[i] + w.Dt;
    // Packed upper triangles of the 6x6 wrench-space Hessians: side 0 = torso (about P), side 1 = probe (about the site).  The two
    // sides are two trips of ONE rolled loop (one copy of the body in the instruction cache; only the few probe-particle contacts
    // are visited by both trips).  Entry l of a triangle lands in lane l of every warp, then in row `wrp` of rb1 / rb2.
#pragma unroll 1
    for (int side = 0; side < 2; side++) {
    float acc[21];
#pragma unroll
    for (int k = 0; k < 21; k++) acc[k] = 0.f;
#pragma unroll 1
    for (int c = tid; c < ncon; c += NT) {
      int zone = w.czone[c], type = w.ctype[c], i = w.cpart[c];
      if (side == 0) { w.sc[0][c] = 0.f; w.sc[1][c] = 0.f; w.sc[2][c] = 0.f; w.cfs[c] = 0.f; } // this contact's share of its slider's (K a, a^T K a)
      if (zone == 0 || type == (side == 0 ? 2 : 0)) continue;
      const float Dn = w.cD[c], Dtn = Dn * dm.impratio;
      const v3 pos = mk(w.cpos[0][c], w.cpos[1][c], w.cpos[2][c]), nn = mk(w.cn[0][c], w.cn[1][c], w.cn[2][c]);
      // World Hessian of the cone cost wrt the contact-point acceleration, K = c_i I + c_n n n^T + c_u u u^T + c_g g g^T
      // (u: unit tangential direction of j, g = mu n - mu fr u the gradient direction of the middle zone)
      float ci, cnn, cu = 0.f, cg = 0.f;
      v3 u = mk(0, 0, 0), gv = mk(0, 0, 0);
      if (zone == 2) { // bottom zone: quadratic, Dn along n and Dt in the tangent plane
        ci = Dtn; cnn = Dn - Dtn;
      } else { // middle zone: exact Hessian of 0.5 Dm (N - mu T)^2
        float fr, mu;
        contact_params(type, fr, mu);
        const v3 j = mk(w.cjar[0][c], w.cjar[1][c], w.cjar[2][c]);
        const float jn = dot(j, nn);
        const v3 jt = j - jn * nn;
        const float tn = fmaxf(norm(jt), 1e-20f), T = fr * tn, Dm = Dn / (mu * mu * (1.f + mu * mu)), NmT = jn * mu - mu * T;
        u = (1.f / tn) * jt;
        gv = mu * nn - (mu * fr) * u;
        const float kk = -Dm * mu * NmT / T * fr * fr; // curvature of the cone surface, acts on the tangent plane minus u
        ci = kk; cnn = -kk; cu = -kk; cg = Dm;
      }
      float Ks[6]; // xx, xy, xz, yy, yz, zz
      Ks[0] = ci + cnn * nn.x * nn.x + cu * u.x * u.x + cg * gv.x * gv.x;
      Ks[1] = cnn * nn.x * nn.y + cu * u.x * u.y + cg * gv.x * gv.y;
      Ks[2] = cnn * nn.x * nn.z + cu * u.x * u.z + cg * gv.x * gv.z;
      Ks[3] = ci + cnn * nn.y * nn.y + cu * u.y * u.y + cg * gv.y * gv.y;
      Ks[4] = cnn * nn.y * nn.z + cu * u.y * u.z + cg * gv.y * gv.z;
      Ks[5] = ci + cnn * nn.z * nn.z + cu * u.z * u.z + cg * gv.z * gv.z;
      const v3 K0 = mk(Ks[0], Ks[1], Ks[2]), K1 = mk(Ks[1], Ks[3], Ks[4]), K2 = mk(Ks[2], Ks[4], Ks[5]);
      if (side == 0) { // slider of this particle: K a_i and a_i^T K a_i, gathered per slider by its owner slot below
        v3 aw = mv(R, xyz(pt.ax4[i]));
        v3 ka = mk(dot(K0, aw), dot(K1, aw), dot(K2, aw));
        w.sc[0][c] = ka.x; w.sc[1][c] = ka.y; w.sc[2][c] = ka.z;
        w.cfs[c] = dot(aw, ka);
      }
      // wrench-space Hessian [I; [r]x] K [I, [r]x^T] (force; torque about the reference point), packed upper triangle:
      // upper-right block rows r x K_i, lower-right block columns r x (column of the upper-right block)
      {
        const v3 r = pos - (side == 0 ? P : site);
        const v3 B0 = cross(r, K0), B1 = cross(r, K1), B2 = cross(r, K2); // rows of K [r]x^T
        const v3 C0 = cross(r, mk(B0.x, B1.x, B2.x)), C1 = cross(r, mk(B0.y, B1.y, B2.y)), C2 = cross(r, mk(B0.z, B1.z, B2.z)); // columns of [r]x K [r]x^T
        acc[tri6(0, 0)] += Ks[0]; acc[tri6(0, 1)] += Ks[1]; acc[tri6(0, 2)] += Ks[2]; acc[tri6(1, 1)] += Ks[3]; acc[tri6(1, 2)] += Ks[4]; acc[tri6(2, 2)] += Ks[5];
        acc[tri6(0, 3)] += B0.x; acc[tri6(0, 4)] += B0.y; acc[tri6(0, 5)] += B0.z;
        acc[tri6(1, 3)] += B1.x; acc[tri6(1, 4)] += B1.y; acc[tri6(1, 5)] += B1.z;
        acc[tri6(2, 3)] += B2.x; acc[tri6(2, 4)] += B2.y; acc[tri6(2, 5)] += B2.z;
        acc[tri6(3, 3)] += C0.x; acc[tri6(3, 4)] += C1.x; acc[tri6(3, 5)] += C2.x; acc[tri6(4, 4)] += C1.y; acc[tri6(4, 5)] += C2.y; acc[tri6(5, 5)] += C2.z;
      }
    }
    tsum_to(acc, lane, side == 0 ? w.rb1[wrp] : w.rb2[wrp]);
    }
    env_sync();
    const float kf = lane < 21 ? rd(w.rb1, lane) : 0.f;
    // owner slots: sk <- sum of the slider's K a, diagonal += sum of a^T K a (fixed slot order, no atomics)
#pragma unroll 1
    for (int c = tid; c < ncon; c += NT) {
      const int i = w.cpart[c];
      if (i >= 0 && w.cslot[i] == c) {
        w.sk[0][c] = slider_gather(w.sc[0], c, i); w.sk[1][c] = slider_gather(w.sc[1], c, i); w.sk[2][c] = slider_gather(w.sc[2], c, i);
        w.dg[i] += slider_gather(w.cfs, c, i);
      }
    }
    env_sync();
    // arm block: Pa = M + Jsite^T Kp Jsite + limits   (lanes 0..6, column `lane`)
    float pa_col[7] = {0, 0, 0, 0, 0, 0, 0};
    if (tid < 7) {
      float KJ[6]; // (Kp Jsite)[:, lane]
#pragma unroll
      for (int a2 = 0; a2 < 6; a2++) {
        float sacc = 0.f;
#pragma unroll
        for (int b2 = 0; b2 < 6; b2++) sacc += rd(w.rb2, tri6(a2, b2)) * w.ab[AB_JSITE + b2 * 7 + lane];
        KJ[a2] = sacc;
      }
#pragma unroll
      for (int r2 = 0; r2 < 7; r2++) {
        float sacc = w.ab[AB_M + r2 * 7 + lane];
#pragma unroll
        for (int a2 = 0; a2 < 6; a2++) sacc += w.ab[AB_JSITE + a2 * 7 + r2] * KJ[a2];
        if (r2 == lane && w.lsign[lane] != 0.f) sacc += w.lD[lane];
        pa_col[r2] = sacc;
        w.Pa[r2 * 7 + lane] = sacc;
      }
    }
    // torso block (world-frame omega): Sf = Mfw + Kf - sum_i b_i b_i^T / dg_i,  b_i = [m a_i + K a_i ; r_i x K a_i]
    if (dm.soft) {
      float sb[21];
#pragma unroll
      for (int k = 0; k < 21; k++) sb[k] = 0.f;
#pragma unroll 1
      for (int i = tid; i < np; i += NT) {
        v3 ah = xyz(pt.ax4[i]), aw = mv(R, ah);
        float inv = 1.f / w.dg[i];
        w.dg[i] = inv;
        v3 bv = mp * aw;
        int cs = w.cslot[i];
        if (cs >= 0) {
          v3 kk = mk(w.sk[0][cs], w.sk[1][cs], w.sk[2][cs]);
          v3 cr = mv(R, xyz(pt.ps4[i]) + (w.qrow[14 + i] - dm.cap_r) * ah);
          v3 ck = cross(cr, kk);
          w.sc[0][cs] = ck.x; w.sc[1][cs] = ck.y; w.sc[2][cs] = ck.z;
          bv = bv + kk;
          float b6[6] = {bv.x, bv.y, bv.z, ck.x, ck.y, ck.z};
#pragma unroll
          for (int a2 = 0; a2 < 6; a2++)
#pragma unroll
            for (int c2 = (a2 < 3 ? 3 : a2); c2 < 6; c2++) sb[tri6(a2, c2)] += b6[a2] * b6[c2] * inv;
        }
        sb[tri6(0, 0)] += bv.x * bv.x * inv; sb[tri6(0, 1)] += bv.x * bv.y * inv; sb[tri6(0, 2)] += bv.x * bv.z * inv;
        sb[tri6(1, 1)] += bv.y * bv.y * inv; sb[tri6(1, 2)] += bv.y * bv.z * inv; sb[tri6(2, 2)] += bv.z * bv.z * inv;
      }
      tsum_to(sb, lane, w.rb3[wrp]);
    }
    // both factorisations at once (Sf is a 6x6 padded to 7x7).  If Sf lost positive definiteness (fp32) the second attempt
    // drops the slider coupling: the free block alone is positive definite.
#pragma unroll 1
    for (int attempt = 0; attempt < 2; attempt++) {
      env_sync(); // rb3 (first attempt) / the restored Pa and the cleared slots (second attempt) are in place
      if (dm.soft && tid < 21) {
        int ab2 = c_tri6[tid], a2 = ab2 >> 4, b2 = ab2 & 15;
        float v = w.Mfw[tid] + kf - (attempt == 0 ? rd(w.rb3, tid) : 0.f);
        w.Sf[a2 * 7 + b2] = v; w.Sf[b2 * 7 + a2] = v;
      }
      env_sync();
      if (wrp == 0) {
        const bool ok = chol7_warp2(w.Sf, w.Pa, lane);
        const bool allok = __all_sync(0xffffffffu, ok || lane >= 8);
        if (lane == 0) w.okf = allok;
      }
      env_sync();
      if (w.okf || attempt == 1) break; // (a second failure keeps the clamped factors: the divergence guard ends such an episode)
#pragma unroll 1
      for (int c = tid; c < ncon; c += NT) {
        w.sk[0][c] = 0.f; w.sk[1][c] = 0.f; w.sk[2][c] = 0.f; w.sc[0][c] = 0.f; w.sc[1][c] = 0.f; w.sc[2][c] = 0.f;
      }
      // (Pa was factorised in place by the first attempt: the second one must see the matrix again)
      if (tid < 7) {
#pragma unroll
        for (int r2 = 0; r2 < 7; r2++) w.Pa[r2 * 7 + lane] = pa_col[r2];
      }
    }
  };

  // ------------------------------------------------------------------ K6: nonlinear PCG; pass -1 evaluates the warm start
  float gpg = 1.f;
  int iters = 0, rebuilds = 0, ls_evals = 0;
  const int maxit = mode == 1 ? 2 * dm.iters : dm.iters;
  // every helper has exactly ONE call site (code size: the loop body must stay inside the instruction cache)
#pragma unroll 1
  for (int it = -1; it < maxit; it++) {
    const bool init = it < 0;
    iters = it + 1; // iterations that changed x so far (the convergence test sits in precond(), right after the gradient)
    const float* vin = init ? w.x : w.s;
    float* vout = init ? w.Hx : w.hs;
    float q12[2] = {0.f, 0.f};
    applyH(vin, vout, init ? nullptr : q12);
    contactJ(vin, init ? w.cjar : w.cjv, init);
    float hx2 = 0.f, rhs2 = 0.f;
    if (init) {
      // grad holds rhs until here
      PRAGMA_HOT_S
      for (int i = tid; i < nv; i += NT) {
        float r = w.grad[i], hx = w.Hx[i] - r;
        w.Hx[i] = hx; w.grad[i] = hx;
        rhs2 += r * r; hx2 += hx * hx;
      }
      // (no barrier here: the first pass of update_grad touches per-contact data of this thread only; its own barrier comes before
      // anybody reads the grad rows written above)
    } else {
      // ---- exact line search: Newton on phi'(alpha)
      float q1 = 0.f, q2 = 0.f, alpha = 0.f, lo = 0.f, hi = -1.f, d0abs = 0.f;
#pragma unroll 1
      for (int ls = 0; ls < LS_MAX; ls++) {
        float d1 = 0.f, d2 = 0.f;
        PRAGMA_HOT
        for (int c = tid; c < ncon; c += NT) {
          float fr, mu, a1, a2, Dn = w.cD[c];
          contact_params(w.ctype[c], fr, mu);
          const v3 jv = mk(w.cjv[0][c], w.cjv[1][c], w.cjv[2][c]);
          cone_ls(mk(w.cjar[0][c], w.cjar[1][c], w.cjar[2][c]) + alpha * jv, jv, mk(w.cn[0][c], w.cn[1][c], w.cn[2][c]), Dn, Dn * dm.impratio,
                  mu, fr, a1, a2);
          d1 += a1; d2 += a2;
        }
        if (tid < 7 && w.lsign[lane] != 0.f) {
          float sg = w.lsign[lane], jar = sg * (w.x[lane] + alpha * w.s[lane]) - w.laref[lane], jv = sg * w.s[lane];
          if (jar < 0.f) { d1 += w.lD[lane] * jar * jv; d2 += w.lD[lane] * jv * jv; }
        }
        {
          // the quadratic part (s.Hx, s.Hs) rides on every reduction: constant cost, one call site
          float r4[4] = {d1, d2, q12[0], q12[1]};
          float(*zl)[4] = w.rl[ls & 1]; // alternating landing zones: the next pass may start before every thread has read this one
          tsum_to(r4, lane, zl[wrp]);
          env_sync();
          q1 = rd(zl, 2); q2 = rd(zl, 3);
          d1 = rd(zl, 0) + q1 + alpha * q2;
          d2 = rd(zl, 1) + q2;
        }
        ls_evals++;
        if (ls == 0) d0abs = fabsf(d1);
        if (fabsf(d1) <= LS_TOL * d0abs || !(d2 > 0.f)) break;
        if (d1 < 0.f) lo = alpha; else hi = alpha;
        float an = alpha - d1 / d2;
        if (hi < 0.f) { if (an <= lo) an = 2.f * alpha + 1e-6f; }
        else if (an <= lo || an >= hi) an = 0.5f * (lo + hi);
        if (an == alpha) break;
        alpha = an;
      }
      PRAGMA_HOT_S
      for (int i = tid; i < nv; i += NT) {
        float hx = w.Hx[i] + alpha * w.hs[i];
        w.x[i] += alpha * w.s[i]; w.Hx[i] = hx; w.grad[i] = hx;
        hx2 += hx * hx;
      }
      PRAGMA_HOT
      for (int c = tid; c < ncon; c += NT) {
        w.cjar[0][c] += alpha * w.cjv[0][c]; w.cjar[1][c] += alpha * w.cjv[1][c]; w.cjar[2][c] += alpha * w.cjv[2][c];
      }
      // (no barrier, as above)
    }
    update_grad(hx2, rhs2);
    // Rebuild policy.  A rebuild costs as much as ~0.8 CG passes (two Hessian passes over the contacts, three 21-value reductions, two
    // factorisations) and most zone changes of the first iterations are light contacts flickering: rebuilding on every change
    // (round 1) buys 0.5 iteration for 1.6 rebuilds per solve.  Shipped: no rebuild during the first REBUILD_LATE iterations unless at
    // least REBUILD_MIN contacts changed zone; from then on every change rebuilds (a solve that is still running is a hard one: without
    // the late rebuilds the iteration tail grows, P(>= 20 iterations) 2.5e-4 -> 3.6e-3).  Measured at 4096 envs (kernel ms / iterations /
    // rebuilds per solve / P(>= 40 iterations)):  always 0.481 / 5.33 / 1.63 / 8e-6;  MIN 2, 3, 4, 6 without LATE: 0.468, 0.465, 0.462,
    // 0.460 (6.05 / 0.12 / 7e-5);  never 0.469 / 6.17 / 0 / -;  MIN 4 LATE 5: 0.450;  MIN 6 LATE 5: 0.444;  none before LATE = 6, 5, 4, 3:
    // 0.449, 0.445, 0.442 (5.91 / 0.15 / 1.7e-5), 0.4415 (5.79 / 0.27 / 1.5e-5).
#ifndef REBUILD_MIN
#define REBUILD_MIN 1000
#endif
#ifndef REBUILD_LATE
#define REBUILD_LATE 3
#endif
    const bool changed = rd(w.rg, 12) >= (it < REBUILD_LATE ? (float)REBUILD_MIN : 1.f);
    hxn = sqrtf(rd(w.rg, 13));
    if (init) rhsn = sqrtf(rd(w.rg, 14));
    bool restart = init;
    // soft scene: rebuild when the active set moved; rigid scene (7 unknowns): exact Hessian every iteration = Newton
    if (init || (changed && rebuilds < dm.max_rebuilds) || (!dm.soft && ncon > 0)) {
      build_precond();
      rebuilds += init ? 0 : 1;
      restart = init || !NORESTART;
    }
    if (!precond()) break;
    const float gpo = rd(w.rp, 9), gpn = rd(w.rq, 0); // grad.pg with the previous pg (Polak-Ribiere) and with the new one
#ifdef RESTART_EVERY // developer knob: periodic steepest-descent restart of the nonlinear CG (measured, every 5 / 8 / 12 iterations: 7.82 / 7.68 / 7.86 M against 7.90 M without: long solves are not stalled directions)
    if (it > 0 && it % RESTART_EVERY == 0) restart = true;
#endif
#ifdef BETA_FR // developer knob: Fletcher-Reeves instead of Polak-Ribiere+ (measured: 6.93 instead of 5.79 iterations, 0.655 vs 0.441 ms)
    float beta = restart ? 0.f : gpn / fmaxf(gpg, 1e-30f);
#else
    float beta = restart ? 0.f : fmaxf(0.f, (gpn - gpo) / fmaxf(gpg, 1e-30f));
#endif
    gpg = gpn;
#pragma unroll
    for (int k = 0; k < 4; k++) S4[k] = -rd(w.rq, 2 + k) + beta * S4[k];
    PRAGMA_HOT_S
#if PREC3
    for (int i = tid; i < nv; i += NT) {
      float p = i >= 13 ? w.hs[i] : w.pg[i];
      w.pg[i] = p;
      w.s[i] = -p + beta * w.s[i];
    }
#else
    for (int i = tid; i < nv; i += NT) w.s[i] = -w.pg[i] + beta * w.s[i];
#endif
    env_sync();
  }

  // ------------------------------------------------------------------ K8: probe wrench, F/T torque
  v3 cfrc = mk(rd(w.rg, 6), rd(w.rg, 7), rd(w.rg, 8)), ctq = mk(rd(w.rg, 9), rd(w.rg, 10), rd(w.rg, 11)); // probe wrench of the last gradient evaluation
  v3 ft;
  {
    float t3[3];
#pragma unroll
    for (int r = 0; r < 3; r++) {
      float s = w.ab[AB_TAU0 + r];
#pragma unroll
      for (int j = 0; j < 7; j++) s += w.ab[AB_JFT + r * 7 + j] * w.x[j];
      t3[r] = s;
    }
    ft = mtv(w.ab + AB_EEFR, mk(t3[0], t3[1], t3[2]) - ctq);
  }
  bool in_contact = false;
  for (int c = tid; c < ncon; c += NT) in_contact |= (w.ctype[c] == 1);
  in_contact = WPE == 1 ? __any_sync(0xffffffffu, in_contact) : (bool)__syncthreads_or(in_contact);

  // ------------------------------------------------------------------ K7: integrate (mj_Euler) and write the state back
  if (mode != 1) {
    // arm: implicit joint damping, (M + h D) qacc' = M qacc, through a dense 7x7 Cholesky (w.Pa and w.dv are free again)
    if (tid < 7) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 7; j++) {
        float mj = w.ab[AB_M + lane * 7 + j];
        w.Pa[lane * 7 + j] = mj + (lane == j ? h * dm.arm_damp : 0.f);
        s += mj * w.x[j];
      }
      w.dv[lane] = s;
    }
    env_sync();
    if (wrp == 0) chol7_warp2(w.Pa, nullptr, lane);
    env_sync();
    {
      float b[7];
#pragma unroll
      for (int j = 0; j < 7; j++) b[j] = w.dv[j];
      chol7_solve<7>(w.Pa, b);
      if (tid == 0) {
#pragma unroll
        for (int j = 0; j < 7; j++) w.qdarm[j] += h * b[j];
      }
    }
    env_sync();
    // new state rows are assembled in shared memory (qrow, hs <- qvel, x = qacc_warmstart) and leave as three TMA bulk stores
    if (tid < 7) { w.hs[tid] = w.qdarm[tid]; w.qrow[lane] += h * w.qdarm[tid]; }
    for (int i = 13 + np + tid; i < QPAD; i += NT) w.hs[i] = 0.f;
    if (dm.soft) {
      for (int i = tid; i < np; i += NT) {
        float v = qv_g[13 + i] + h * w.x[13 + i];
        w.hs[13 + i] = v;
        w.qrow[14 + i] += h * v;
      }
      if (tid == 0) {
        v3 vn = vlin + h * ld3(w.x + 7), wn = wl + h * ld3(w.x + 10);
        st3(w.hs + 7, vn); st3(w.hs + 10, wn);
        st3(w.qrow + 7, P + h * vn);
        float wnm = norm(wn), ang = h * wnm;
        if (ang > 0.f) {
          float s = sinf(0.5f * ang) / wnm, qr[4] = {cosf(0.5f * ang), s * wn.x, s * wn.y, s * wn.z}, qn[4];
          quatmul(quat, qr, qn);
          float nq = rsqrtf(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2] + qn[3] * qn[3]);
          w.qrow[10] = qn[0] * nq; w.qrow[11] = qn[1] * nq; w.qrow[12] = qn[2] * nq; w.qrow[13] = qn[3] * nq;
        } else {
          w.qrow[10] = quat[0]; w.qrow[11] = quat[1]; w.qrow[12] = quat[2]; w.qrow[13] = quat[3];
        }
      }
    } else if (tid >= 7 && tid < 13) {
      w.hs[tid] = 0.f;
    }
    // (the new rows stay in shared memory until the task epilogue has decided whether the episode goes on)
  }
  env_sync();

  // ------------------------------------------------------------------ contact list / diagnostics
  if (a.ncon_out) {
    if (tid == 0) a.ncon_out[env] = ncon;
    for (int c = tid; c < ncon; c += NT) {
      int type = w.ctype[c], g1, g2;
      if (type == 2) { g1 = 1; g2 = 2; } else { g1 = 4 + w.cpart[c]; g2 = type == 0 ? 1 : 2; }
      a.geom1_out[(size_t)env * DEV_MAXC + c] = g1;
      a.geom2_out[(size_t)env * DEV_MAXC + c] = g2;
    }
  }

  // divergence guard (MuJoCo resets on bad qacc; SURVEY §5): a non-finite solution ends the episode, the reset wipes the state
  float xnorm2 = 0.f;
  {
    float x1[1] = {0.f};
    for (int i = tid; i < nv; i += NT) x1[0] += w.x[i] * w.x[i];
    tsum_to(x1, lane, w.rq[wrp]);
    env_sync();
    xnorm2 = rd(w.rq, 0);
  }
  // ------------------------------------------------------------------ K9: task epilogue (lane 0)
  if (tid == 0) w.consume = 0;
  if (tid == 0 && mode != 2) {
    float* ts = w.ts;
    v3 hv = mk(0, 0, 0);
    {
      float t3[3];
#pragma unroll
      for (int r = 0; r < 3; r++) {
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 7; j++) s += w.ab[AB_JHAND + r * 7 + j] * w.qdarm[j];
        t3[r] = s;
      }
      hv = mk(t3[0], t3[1], t3[2]);
    }
    v3 eef = ld3(w.ab + AB_EEFPOS);
    const float* quat_e = w.ab + AB_QUAT;
    float reward = 0.f;
    int dn = 0;
    // Task-state channels of the observation.  robosuite samples the observables inside the substep loop, BEFORE _post_action
    // updates the task state, and step() returns the cached values: obs[9..14] of step t carry the task state of step t-1 --
    // the same values reward() uses.  Pinned by the reference's artifacts: in all 192 (old_obs, old_reward) rows of the shipped
    // VecNormalize pickles the reward is reproduced from the observation row to 1e-6 (tests/test_task_golden.py).  A reset
    // force-updates the observables (mode 1: the initialised values below).
    float o_fz = ts[USIM_TS_FZ_MEAN] - 5.f, o_dfz = ts[USIM_TS_DFZ], o_vel = ts[USIM_TS_VEL_MEAN] - 0.04f;
    v3 o_tp = ld3(ts + USIM_TS_TRAJ_PT);
    const bool bad = !isfinite(xnorm2) || !isfinite(cfrc.x + cfrc.y + cfrc.z) || !isfinite(ft.x + ft.y + ft.z) || !isfinite(hv.x + hv.y + hv.z) ||
                     !isfinite(eef.x + eef.y + eef.z);
    if (bad) { // keep the outputs finite; the episode ends below and the reset wipes the state
      cfrc = mk(0, 0, 0); ft = mk(0, 0, 0); hv = mk(0, 0, 0);
      if (!isfinite(eef.x + eef.y + eef.z)) eef = ld3(ts + USIM_TS_TRAJ_PT);
      if (a.counters) atomicAdd(a.counters, 1);
    }
    if (mode == 0) {
      ts[USIM_TS_TIMESTEP] += 1.f;
      if (in_contact) ts[USIM_TS_TOUCHED] = 1.f;
      float pe[2], oe;
      reward = reward_fn(eef, quat_e, ld3(ts + USIM_TS_TRAJ_PT), ts[USIM_TS_VEL_MEAN], ts[USIM_TS_FZ_MEAN], ts[USIM_TS_DFZ], in_contact, pe, &oe);
      ts[USIM_TS_POS_ERR] = pe[0]; ts[USIM_TS_POS_ERR + 1] = pe[1]; ts[USIM_TS_ORI_ERR] = oe;
      float t = ts[USIM_TS_TIMESTEP];
      dn = t >= (float)dm.horizon && !dm.ignore_done; // MujocoEnv._post_action: done = timestep >= horizon and not ignore_done
      float u = fminf(fmaxf(t / (float)dm.horizon + ts[USIM_TS_U0], 0.f), 1.f); // ultrasound.py:528-532
#pragma unroll
      for (int k = 0; k < 3; k++) ts[USIM_TS_TRAJ_PT + k] = ts[USIM_TS_TRAJ_START + k] + u * (ts[USIM_TS_TRAJ_END + k] - ts[USIM_TS_TRAJ_START + k]);
      ts[USIM_TS_VEL_MEAN] += (norm(hv) - ts[USIM_TS_VEL_MEAN]) / t;   // :538
      ts[USIM_TS_DFZ] = (cfrc.z - ts[USIM_TS_FZ_PREV]) * dm.ctrl_freq;  // :542
      ts[USIM_TS_FZ_PREV] = cfrc.z;
      ts[USIM_TS_FZ_MEAN] = 0.1f * cfrc.z + 0.9f * ts[USIM_TS_FZ_MEAN]; // :546
      if (dm.early_term) { // :635-670
        int term = 0;
#pragma unroll
        for (int j = 0; j < 7; j++) {
          float qn = w.qrow[j];
          if (!(dm.jnt_lo[j] + 0.1f < qn && qn < dm.jnt_hi[j] - 0.1f)) term = 1;
        }
        if (sqrtf(pe[0] * pe[0] + pe[1] * pe[1]) > 1.0f) term = 1;
        if (in_contact && oe > 0.10f) term = 1;
        if (ts[USIM_TS_TOUCHED] != 0.f && !in_contact) term = 1;
        dn = dn || term;
      }
      if (bad) dn = 1;
      ts[USIM_TS_DONE] = (float)dn;
    } else {
      ts[USIM_TS_FZ_PREV] = 0.f; ts[USIM_TS_DFZ] = 0.f;
      ts[USIM_TS_VEL_MEAN] = norm(hv);   // :474
      ts[USIM_TS_FZ_MEAN] = cfrc.z;      // :477
      ts[USIM_TS_TOUCHED] = 0.f; ts[USIM_TS_TIMESTEP] = 0.f; ts[USIM_TS_DONE] = 0.f;
      o_fz = ts[USIM_TS_FZ_MEAN] - 5.f; o_dfz = 0.f; o_vel = ts[USIM_TS_VEL_MEAN] - 0.04f;
    }
    ts[USIM_TS_IN_CONTACT] = in_contact ? 1.f : 0.f;
    // auto-reset (SB3 VecEnv semantics): the env takes over its prepared slot below; this step's observation is the terminal one
    const bool consume = mode == 0 && a.auto_reset && dn;
    w.consume = consume;
    { // ultrasound.py:363-401; staged in shared memory, stored by 19 lanes below (one coalesced row: the destination may be
      // page-locked HOST memory, usim_step_host)
      float* o = w.orow;
      o[0] = cfrc.x; o[1] = cfrc.y; o[2] = cfrc.z; o[3] = ft.x; o[4] = ft.y; o[5] = ft.z; o[6] = hv.x; o[7] = hv.y; o[8] = hv.z;
      o[9] = o_fz; o[10] = o_dfz; o[11] = o_vel;
      o[12] = eef.x - o_tp.x; o[13] = eef.y - o_tp.y; o[14] = eef.z - o_tp.z;
      float gq[4] = {GQX, GQY, GQZ, GQW};
      difference_quat(quat_e, gq, o + 15); // xyzw arrays through a wxyz routine (:390)
    }
    if (mode == 0) {
      if (a.rew) a.rew[env] = reward;
      if (a.done) a.done[env] = (uint8_t)dn;
    }
    if (a.diag) {
      float* d = a.diag + (size_t)env * USIM_DIAG_DIM;
      d[0] = cfrc.x; d[1] = cfrc.y; d[2] = cfrc.z; d[3] = ft.x; d[4] = ft.y; d[5] = ft.z; d[6] = eef.x; d[7] = eef.y; d[8] = eef.z;
      d[9] = quat_e[0]; d[10] = quat_e[1]; d[11] = quat_e[2]; d[12] = quat_e[3];
#pragma unroll
      for (int j = 0; j < 7; j++) d[13 + j] = w.ab[AB_TAU + j];
      int nlim = 0;
      for (int j = 0; j < 7; j++) nlim += w.lsign[j] != 0.f;
      d[20] = (float)iters; d[21] = gnorm; d[22] = (float)ncon_found;
      d[23] = (float)(3 * ncon + nlim + (dm.soft ? 2 * 0 + np + dm.npair + 1 : 0));
      d[24] = (float)rebuilds; d[25] = (float)ls_evals; d[26] = 0.f; d[27] = 0.f;
    }
  }
  // file the env for the next launch's order: by the iterations it took; a freshly reset env (cold start) goes first
  if (tid == 0 && a.bin_cnt) {
    const int b = w.consume ? NBIN - 1 : min(iters, NBIN - 1);
    a.bin_items[(size_t)b * n + atomicAdd(a.bin_cnt + b, 1)] = env;
  }
  env_sync();
  // ------------------------------------------------------------------ contact record (opt-in, usim_set_contact_record)
  if (a.crec_out) record_contacts(w, a.crec_out + (size_t)env * DEV_MAXC * CREC_DIM, ncon, tid);
  if (mode != 2 && tid < USIM_OBS_DIM) { // this step's observation: the terminal one if a prepared reset state takes over below
    float* o = w.consume ? (a.tobs ? a.tobs + (size_t)env * USIM_OBS_DIM : nullptr) : obs_row;
    if (o) o[tid] = w.orow[tid];
  }
  if (w.consume) {
    // The episode is over and auto-reset is on: the prepared slot (episode number E = the live record's counter, slot E & 1) becomes
    // the live state.  Velocity and warm start of a reset state are zero.  Then ask for episode E + 2 to be prepared in this slot.
    const int E = (int)w.ts[USIM_TS_EPISODE];
    const size_t row = (size_t)(E & 1) * n + env;
    const float4* sq = reinterpret_cast<const float4*>(a.slot_qpos + row * QPAD);
    const float4* st = reinterpret_cast<const float4*>(a.slot_task + row * USIM_TASK_DIM);
    float4 *dq = reinterpret_cast<float4*>(qp_g), *dvv = reinterpret_cast<float4*>(qv_g), *dw = reinterpret_cast<float4*>(wm_g);
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = tid; i < QPAD / 4; i += NT) { dq[i] = sq[i]; dvv[i] = z4; dw[i] = z4; }
    for (int i = tid; i < USIM_TASK_DIM / 4; i += NT) reinterpret_cast<float4*>(ts_g)[i] = st[i];
    if (obs_row && tid < USIM_OBS_DIM) obs_row[tid] = a.slot_obs[row * SLOT_OBS + tid];
    env_sync(); // every thread has read the slot: it may be overwritten from here on
    if (tid == 0) {
      __threadfence();
      const int p = atomicAdd(a.req_cnt, 1);
      a.req_list[2 * p] = env; a.req_list[2 * p + 1] = E + 2;
    }
  } else {
    // state rows and task record back to HBM (TMA bulk stores out of the shared-memory image), then wait until the stores have
    // finished READING shared memory: the next trip / the exit of the CTA may not come before
    fence_async_smem();
    env_sync();
    if (tid == 0) {
      if (mode != 1) {
        tma_store_row(qp_g, w.qrow, QPAD * 4);
        tma_store_row(qv_g, w.hs, QPAD * 4);
        tma_store_row(wm_g, w.x, QPAD * 4);
      }
      tma_store_row(ts_g, w.ts, USIM_TASK_DIM * 4);
      tma_store_commit_wait();
    }
  }
  env_sync();
#if USIM_TRACE
  if (a.trace && tid == 0) {
    unsigned long long t_end;
    unsigned smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    a.trace[3 * (size_t)env] = w.t0; a.trace[3 * (size_t)env + 1] = t_end; a.trace[3 * (size_t)env + 2] = smid;
  }
#endif
  } // work items
}
