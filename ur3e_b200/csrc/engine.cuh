// Fused per-environment simulation step for the UR3e + 2F85 (+ mug) scenes: one environment per warp,
// all per-substep state in a shared-memory arena (see DESIGN.md "kernel").
//
// Replaces, for one environment, the reference's  controller -> mj_step x frame_skip -> obs/reward/done
// path (reference gymnasium_env/envs/ur3e_env2.py:72-99; controller/controller_func.py:68-117,128-167;
// mujoco mj_step restated in SURVEY App. B).  This file is written against warp_model.cuh and contains
// no CUDA-only constructs, so tests/hostcheck can compile it on the CPU to debug the mathematics.
#pragma once
#include "dev_model.h"
#include "warp_model.cuh"

namespace ur3e {

template <int NB_, int NV_, int NQ_, int NU_, int NG_, int NPAIR_, int MAXCON_, int MAXEFC_, int SPLIT_ = NV_, bool EXACT_ = false>
struct Dims {
  // EXACT: the kernel is only ever launched for a model whose sizes equal NB / NV / NQ / NU / NG / NPAIR (checked at batch
  // creation), so those loop bounds are compile-time constants: WARP_FOR over <= 32 items becomes a predicate, no loop
  static constexpr bool EXACT = EXACT_;
  // dofs [SPLIT, NV) belong to the model's last kinematic tree (the mug's free joint): M never couples them to the dofs
  // before, and the Newton matrix only does while a constraint spans both (a pad touching the mug) -- see chol_solve_reg_body
  static constexpr int SPLIT = SPLIT_;
  static constexpr int NB = NB_, NV = NV_, NQ = NQ_, NU = NU_, NG = NG_ > 0 ? NG_ : 1, NPAIR = NPAIR_ > 0 ? NPAIR_ : 1;
  static constexpr int MAXCON = MAXCON_ > 0 ? MAXCON_ : 1, MAXEFC = MAXEFC_ > 0 ? MAXEFC_ : 1;
  static constexpr bool HAS_CONTACT = MAXCON_ > 0;
  static constexpr int NS = MAXSITE;
  // candidate pairs that survive the broad phase get a narrow-phase slot; more than MAXACT at once counts as an overflow
  static constexpr int ACT_CAP = MAXCON_ <= 8 ? 16 : (MAXCON_ <= 16 ? 20 : 24);
  static constexpr int MAXACT = !HAS_CONTACT ? 1 : (NPAIR < ACT_CAP ? NPAIR : ACT_CAP);
  static constexpr int NGRP = MAXEQ + (NPAIR < MAXCON ? NPAIR : MAXCON);   // one row group per connect equality / pair with contacts
  static constexpr int MAXCONNECT = 2;   // connect equalities a size class stores rows for (the 2F85 has two; checked at batch creation)
  static constexpr int MAXDENSE = HAS_CONTACT ? 3 * MAXCONNECT + 3 * MAXCON : 1;   // stored Jacobian rows
};
using DimsRaw = Dims<8, 6, 6, 6, 1, 0, 0, 12>;          // body counts are after fixed-body merging (merge_bodies.h)          // assets/ur3e_raw.xml
using DimsGrip = Dims<17, 14, 14, 7, 6, 12, 12, 56>;    // assets/ur3e_2f85.xml
using DimsGripExact = Dims<17, 14, 14, 7, 6, 12, 12, 56, 14, true>;   // the same caps, compiled for exactly ur3e_2f85.xml's sizes (float32 only)
using DimsMain = Dims<19, 20, 21, 7, 14, 48, 24, 92, 14>;   // assets/main.xml (collidable geoms: four pad boxes, the mug, the table plane, eight link hulls)
using DimsMainLite = Dims<19, 20, 21, 7, 14, 48, 8, 44, 14, true>;   // same model, caps for the common case (<= 8 contacts, <= 44 rows)
using DimsMainMid = Dims<19, 20, 21, 7, 14, 48, 16, 68, 14, true>;   // the grasp tier: both pads on the lifted mug are 16 contacts / ~62 rows (float32 only)

constexpr int STAGE_PTS = 8;  // contact points a pair can emit
constexpr int STAGE_W = 3 + 4 * STAGE_PTS;

// row kinds; the rows of a launch are ordered [connect equalities | contacts] (dense: these have a stored Jacobian row)
// then [joint equalities | friction loss | joint limits] (sparse: one or two +-1 / polynomial entries, never stored)
enum RowType { ROW_EQ = 0, ROW_EQJ = 1, ROW_FRICTION = 2, ROW_LIMIT_LO = 3, ROW_LIMIT_HI = 4, ROW_CON_N = 5, ROW_CON_T1 = 6, ROW_CON_T2 = 7 };

// Persistent per-environment record (lives in HBM between launches, one contiguous 16-byte aligned block per
// environment so that a warp loads/stores it with coalesced 128-bit accesses).
constexpr int NSTAT = 16;
constexpr int MAX_FRAME_SKIP = 256;   // 256 substeps x 112 rows < 2^15: the per-step row / contact / iteration sums are 16-bit
enum StatSlot { ST_EPISODES = 0, ST_RETURN, ST_LENGTH, ST_SUCCESS, ST_TERM_REACH, ST_TERM_TOPPLE, ST_TERM_COLLISION, ST_TRUNC, ST_UNSTABLE,
                ST_NEFC, ST_NCON, ST_ITER, ST_SUBSTEPS, ST_OVERFLOW,
                ST_PADCON /* env-steps that ended with at least one pad-mug contact */, ST_STEPS /* env-steps */ };
template <typename Real, typename D>
struct alignas(16) EnvState {
  Real qpos[D::NQ], qvel[D::NV], qacc_ws[D::NV];
  Real cache[CACHE_SIZE];   // stale-kinematics cache read by the next step's controller (SURVEY F9)
  Real ep_return;
  union { int i; float f; } stat[NSTAT];   // counters since the last ur3e_batch_stats(reset): 32-bit integers (exact), except ST_RETURN (a float sum)
  int t, episode;
  int tier;   // two-tier stepping: > 0 = steps this environment still goes straight to the full size class (set by the full tier when a
              // step needed more contacts / rows than the lite caps; counts down otherwise).  A function of the environment's own history
              // only, so which kernel steps an environment never depends on the batch size, the chunking or the host's timing.
};

// Debug build (-DUR3E_CANARY, tools/canary_check.sh): guard words between the arena's arrays, set when a warp claims its arena and checked
// after every environment step; a clobbered word is reported with printf and counted as an unstable step.  compute-sanitizer is closed
// on the GPU pool, so this is the memory-safety net for the phase-aliased storage below (the aliases themselves are covered by the
// bit-exactness tests: a premature overwrite of a live alias changes results).
#ifdef UR3E_CANARY
#define UR3E_GUARD(n) unsigned guard##n;
constexpr unsigned CANARY_WORD = 0xC0FFEE5Au;
#else
#define UR3E_GUARD(n)
#endif

template <typename Real, typename D>
struct Arena {
  EnvState<Real, D> st;
  UR3E_GUARD(0)
  Real qacc[D::NV], ctrl[D::NU], act_force[D::NU];
  Real xpos[D::NB][3];
  union alignas(8) {   // body frames are dead once the constraint rows exist; the Newton / Euler matrix reuses their storage
    struct { Real xmat[D::NB][9], xipos[D::NB][3]; } k;
    struct { Real H[(D::NV + 1) * (D::NV + 2) / 2]; } n;   // augmented Newton / Euler matrix, packed lower triangle: (i,j) at i(i+1)/2 + j
  } fr;
  union { alignas(16) Real colbuf[1][32]; Real obs[32]; };   // solver scratch / the step's observation (written after the last solve)
  Real cdof[D::NV][6];
  UR3E_GUARD(1)
  alignas(8) Real M[D::NV * (D::NV + 1) / 2];   // packed lower triangle, M(i,j) at i(i+1)/2 + j for j <= i
  UR3E_GUARD(2)
  Real qfrc_smooth[D::NV], qfrc_bias[D::NV], qfrc_constraint[D::NV], grad[D::NV], search[D::NV], Ma[D::NV];
  union { Real Mv[D::NV]; Real dinv[D::NV]; };   // M * search (line search) / reciprocal pivots of the shared-memory factorisations (host build, tree LDL)
  Real site_xpos[D::NS][3], site_xmat[1][9] /* tcp only */, site_velp[D::NS][3];
  Real con_pos[D::MAXCON][3], con_dist[D::MAXCON], con_mu[D::MAXCON];
  union {
    Real frame[D::MAXCON][9];   // contact frames: normal, two tangents.  The solver keeps each contact's cone Hessian (6 values)
                                // in the tangents' storage (frame[c] + 3); the normal survives for the touch sensors
    Real gpos[D::NG][3];        // broad phase only (before any contact frame exists): world positions of the collidable geoms
  } cu;
  static_assert(D::MAXCON * 9 >= D::NG * 3 || !D::HAS_CONTACT, "geom positions alias the contact frames");
  Real efc_aref[D::MAXEFC], efc_D[D::MAXEFC], efc_jv[D::MAXEFC], efc_Dact[D::MAXEFC];
  UR3E_GUARD(3)
  Real efc_force[D::MAXEFC], efc_jar[D::MAXEFC];
  UR3E_GUARD(4)
  uint8_t con_pair[D::MAXCON], con_row[D::MAXCON];
  uint8_t efc_type[D::MAXEFC], efc_id[D::MAXEFC];
  // row groups sharing one column set (a connect equality, the joint equality, the contacts of one geom pair)
  int grp_mask[D::NGRP];
  uint8_t grp_row0[D::NGRP], grp_nrow[D::NGRP];
  uint8_t stage_n[D::MAXACT], stage_off[D::MAXACT], act_pair[D::MAXACT];   // narrow-phase slots: contacts found, offset in the contact list, candidate pair
  Real eqj_deriv[MAXEQ];
  // per dof: its sparse rows (255 = none) so that the solver's inner loops never touch the model tables
  uint8_t sp_fl[D::NV], sp_lo[D::NV], sp_hi[D::NV], sp_ej[D::NV];
  int lim_lo, lim_hi;
  short nd, rf0, rl0;   // dense rows [0, nd); friction rows from rf0, limit rows from rl0
  short ncon, nefc, ne, nf, nl, ngrp, overflow, solver_iter, bad, max_ncon, max_nefc, cap_con, cap_efc;
  short sum_ncon, sum_nefc, sum_iter, warn;   // accumulated over the substeps of one env step (frame_skip <= MAX_FRAME_SKIP keeps them in range)
  short coupled;   // some constraint of this substep has entries on both sides of Dims::SPLIT
  UR3E_GUARD(5)
  union alignas(16) {
    struct { Real cinert[D::NB][10], cdof_dot[D::NV][6], cvel[D::NB][6], cfrc[D::NB][6]; } dyn;   // cinert becomes the composite inertia, cdof_dot the crb*cdof buffer
    struct { Real lmat[D::NB][9], lpos[D::NB][3]; } kin;   // kinematics only: each body's frame relative to its parent
    Real stage[D::MAXACT][STAGE_W];   // per narrow-phase slot: shared normal (3), then up to STAGE_PTS x (pos 3, dist 1)
    Real efc_J[D::MAXDENSE][D::NV];   // dense rows only
  } u;
  UR3E_GUARD(6)
};

#ifdef UR3E_CANARY
template <typename Real, typename D> UR3E_HD void canary_set(Arena<Real, D>& s) {
  IF_LANE0 { s.guard0 = s.guard1 = s.guard2 = s.guard3 = s.guard4 = s.guard5 = s.guard6 = CANARY_WORD; }
}
template <typename Real, typename D> UR3E_HD int canary_bad(const Arena<Real, D>& s) {
  return (s.guard0 != CANARY_WORD) | ((s.guard1 != CANARY_WORD) << 1) | ((s.guard2 != CANARY_WORD) << 2) | ((s.guard3 != CANARY_WORD) << 3) |
         ((s.guard4 != CANARY_WORD) << 4) | ((s.guard5 != CANARY_WORD) << 5) | ((s.guard6 != CANARY_WORD) << 6);
}
#endif

// Further model constants of an exact-fit size class (tree depth, nnz of M, friction-loss dofs, equalities, tracked sites):
// specialised for the class, checked against the loaded model at batch creation like the Dims sizes.
template <typename D> struct StaticModel { static constexpr int NLEVEL = 0, NM = 0, NFL = 0, NEQ = 0, NSITE = 0, NDEQ = 0, NEJ = 0; static constexpr bool DAMPING = false; };
template <> struct StaticModel<DimsGripExact> { static constexpr int NLEVEL = 10, NM = 81, NFL = 6, NEQ = 3, NSITE = 1, NDEQ = 6, NEJ = 1; static constexpr bool DAMPING = true; };
template <> struct StaticModel<DimsMainLite> { static constexpr int NLEVEL = 10, NM = 102, NFL = 6, NEQ = 3, NSITE = 4, NDEQ = 6, NEJ = 1; static constexpr bool DAMPING = true; };
template <> struct StaticModel<DimsMainMid> : StaticModel<DimsMainLite> {};
#define UR3E_MODEL_CONST(fn, STATIC, field) \
  template <typename D, typename Real> UR3E_HD auto fn(const DevModel<Real>& m) { if constexpr (D::EXACT) return StaticModel<D>::STATIC; else return m.field; }
UR3E_MODEL_CONST(nlevel_, NLEVEL, nlevel) UR3E_MODEL_CONST(nM_, NM, nM) UR3E_MODEL_CONST(nfl_, NFL, nfl) UR3E_MODEL_CONST(neq_, NEQ, neq)
UR3E_MODEL_CONST(nsite_, NSITE, nsite) UR3E_MODEL_CONST(ndeq_, NDEQ, ndeq) UR3E_MODEL_CONST(nej_, NEJ, nej)
template <typename D, typename Real> UR3E_HD bool has_damping_(const DevModel<Real>& m) { if constexpr (D::EXACT) return StaticModel<D>::DAMPING; else return m.has_damping != 0; }
template <typename D, typename Real> UR3E_HD int split_(const DevModel<Real>& m) { if constexpr (D::EXACT) return D::SPLIT; else return m.split; }

// model sizes as seen by a kernel of size class D (see Dims::EXACT)
template <typename D, typename Real> UR3E_HD int nv_(const DevModel<Real>& m) { if constexpr (D::EXACT) return D::NV; else return m.nv; }
template <typename D, typename Real> UR3E_HD int nb_(const DevModel<Real>& m) { if constexpr (D::EXACT) return D::NB; else return m.nbody; }
template <typename D, typename Real> UR3E_HD int nq_(const DevModel<Real>& m) { if constexpr (D::EXACT) return D::NQ; else return m.nq; }
template <typename D, typename Real> UR3E_HD int nu_(const DevModel<Real>& m) { if constexpr (D::EXACT) return D::NU; else return m.nu; }
template <typename D, typename Real> UR3E_HD int ng_(const DevModel<Real>& m) { if constexpr (D::EXACT) return D::NG; else return m.ngeom; }
template <typename D, typename Real> UR3E_HD int np_(const DevModel<Real>& m) { if constexpr (D::EXACT) return D::NPAIR; else return m.npair; }

// ---------------------------------------------------------------- scalar math
template <typename Real> struct Num;
template <> struct Num<float> {
  static UR3E_HD float sqrt(float x) { return ::sqrtf(x); }
  static UR3E_HD float sin(float x) { return ::sinf(x); }
  // branch-free sincos: Cody-Waite reduction by pi/2 + the classic single-precision minimax polynomials (error ~1 ulp for
  // |x| < 1e4); replaces the library calls whose slow paths dominate the kinematics code size
  static UR3E_HD void sincos(float x, float* sn, float* cs) {
    float q = ::rintf(x * 0.636619772f);
    int n = (int)q;
    float r = ::fmaf(q, -1.5707963109016418f, x); r = ::fmaf(q, -1.5893254712295857e-8f, r);
    float r2 = r * r;
    float sp = r + r * r2 * (-1.6666654611e-1f + r2 * (8.3321608736e-3f + r2 * -1.9515295891e-4f));
    float cp = 1.0f + r2 * (-0.5f + r2 * (4.166664568298827e-2f + r2 * (-1.388731625493765e-3f + r2 * 2.443315711809948e-5f)));
    float s0 = (n & 1) ? cp : sp, c0 = (n & 1) ? sp : cp;
    *sn = (n & 2) ? -s0 : s0;
    *cs = ((n + 1) & 2) ? -c0 : c0;
  }
  static UR3E_HD float cos(float x) { return ::cosf(x); }
  static UR3E_HD float atan2(float y, float x) { return ::atan2f(y, x); }
  static UR3E_HD float pow(float x, float y) { return ::powf(x, y); }
#if defined(__CUDA_ARCH__)
  static UR3E_HD float pow_pos(float x, float y) { return x > 0 ? __powf(x, y) : 0.f; }   // x in [0, 1]
#else
  static UR3E_HD float pow_pos(float x, float y) { return x > 0 ? ::powf(x, y) : 0.f; }
#endif
  static UR3E_HD float exp(float x) { return ::expf(x); }
  static UR3E_HD float tanh(float x) { return ::tanhf(x); }
  static UR3E_HD float abs(float x) { return ::fabsf(x); }
  static constexpr float minval = 1e-15f, big = 1e30f;
};
template <> struct Num<double> {
  static UR3E_HD double sqrt(double x) { return ::sqrt(x); }
  static UR3E_HD double sin(double x) { return ::sin(x); }
  static UR3E_HD void sincos(double x, double* sn, double* cs) { *sn = ::sin(x); *cs = ::cos(x); }
  static UR3E_HD double cos(double x) { return ::cos(x); }
  static UR3E_HD double atan2(double y, double x) { return ::atan2(y, x); }
  static UR3E_HD double pow(double x, double y) { return ::pow(x, y); }
  static UR3E_HD double pow_pos(double x, double y) { return x > 0 ? ::pow(x, y) : 0.0; }
  static UR3E_HD double exp(double x) { return ::exp(x); }
  static UR3E_HD double tanh(double x) { return ::tanh(x); }
  static UR3E_HD double abs(double x) { return ::fabs(x); }
  static constexpr double minval = 1e-15, big = 1e300;
};
template <typename Real> UR3E_HD Real rmax(Real a, Real b) { return a > b ? a : b; }
template <typename Real> UR3E_HD Real rmin(Real a, Real b) { return a < b ? a : b; }
template <typename Real> UR3E_HD Real dot3(const Real* a, const Real* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
template <typename Real> UR3E_HD void cross3(Real* r, const Real* a, const Real* b) {
  Real x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
template <typename Real> UR3E_HD void quat_mul(Real* r, const Real* a, const Real* b) {
  Real w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  Real y = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], z = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = w; r[1] = x; r[2] = y; r[3] = z;
}
template <typename Real> UR3E_HD void quat_normalize(Real* q) {
  Real n = Num<Real>::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < Num<Real>::minval) { q[0] = 1; q[1] = q[2] = q[3] = 0; } else { Real s = Real(1) / n; q[0] *= s; q[1] *= s; q[2] *= s; q[3] *= s; }
}
template <typename Real> UR3E_HD void quat2mat(Real* m, const Real* q) {
  Real w = q[0], x = q[1], y = q[2], z = q[3];
  m[0] = w * w + x * x - y * y - z * z; m[1] = 2 * (x * y - w * z); m[2] = 2 * (x * z + w * y);
  m[3] = 2 * (x * y + w * z); m[4] = w * w - x * x + y * y - z * z; m[5] = 2 * (y * z - w * x);
  m[6] = 2 * (x * z - w * y); m[7] = 2 * (y * z + w * x); m[8] = w * w - x * x - y * y + z * z;
}
template <typename Real> UR3E_HD void mat_vec3(Real* r, const Real* m, const Real* v) {
  Real x = m[0] * v[0] + m[1] * v[1] + m[2] * v[2], y = m[3] * v[0] + m[4] * v[1] + m[5] * v[2], z = m[6] * v[0] + m[7] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
template <typename Real> UR3E_HD Real normalize3(Real* a) {
  Real n = Num<Real>::sqrt(dot3(a, a));
  if (n < Num<Real>::minval) { a[0] = 1; a[1] = 0; a[2] = 0; } else { Real s = Real(1) / n; a[0] *= s; a[1] *= s; a[2] *= s; }
  return n;
}
// spatial vectors: [rotational(3); translational(3)] about the tree reference point, world axes
template <typename Real> UR3E_HD void mul_inert(Real* r, const Real* i, const Real* v) {
  Real r0 = i[0] * v[0] + i[3] * v[1] + i[4] * v[2] - i[8] * v[4] + i[7] * v[5];
  Real r1 = i[3] * v[0] + i[1] * v[1] + i[5] * v[2] + i[8] * v[3] - i[6] * v[5];
  Real r2 = i[4] * v[0] + i[5] * v[1] + i[2] * v[2] - i[7] * v[3] + i[6] * v[4];
  Real r3 = i[8] * v[1] - i[7] * v[2] + i[9] * v[3];
  Real r4 = i[6] * v[2] - i[8] * v[0] + i[9] * v[4];
  Real r5 = i[7] * v[0] - i[6] * v[1] + i[9] * v[5];
  r[0] = r0; r[1] = r1; r[2] = r2; r[3] = r3; r[4] = r4; r[5] = r5;
}
template <typename Real> UR3E_HD void cross_motion(Real* r, const Real* vel, const Real* v) {
  Real a[3], b[3], c[3];
  cross3(a, vel, v); cross3(b, vel, v + 3); cross3(c, vel + 3, v);
  r[0] = a[0]; r[1] = a[1]; r[2] = a[2]; r[3] = b[0] + c[0]; r[4] = b[1] + c[1]; r[5] = b[2] + c[2];
}
template <typename Real> UR3E_HD void cross_force(Real* r, const Real* vel, const Real* f) {
  Real a[3], b[3], c[3];
  cross3(a, vel, f); cross3(b, vel + 3, f + 3); cross3(c, vel, f + 3);
  r[0] = a[0] + b[0]; r[1] = a[1] + b[1]; r[2] = a[2] + b[2]; r[3] = c[0]; r[4] = c[1]; r[5] = c[2];
}

// row i of (symmetric, packed lower-triangular) A times x
template <typename Real> UR3E_HD Real sym_matvec_row(const Real* A, const Real* x, int i, int n) {
  Real v = 0;
  const Real* row = A + i * (i + 1) / 2;
  for (int k = 0; k <= i; ++k) v += row[k] * x[k];
  for (int k = i + 1; k < n; ++k) v += A[k * (k + 1) / 2 + i] * x[k];
  return v;
}
// generic-size fall-back (model smaller than the size class): rolled, inline -- a call here would cost the hot path registers
template <typename Real> UR3E_HD Real sym_matvec_row_cold(const Real* A, const Real* x, int i, int n) {
  Real v = 0;
#pragma unroll 1
  for (int k = 0; k < n; ++k) v += (k <= i ? A[i * (i + 1) / 2 + k] : A[k * (k + 1) / 2 + i]) * x[k];
  return v;
}
// the same, fully unrolled for the size class (one address select + load + FMA per column, no loop or index arithmetic)
template <typename Real, int N> UR3E_HD Real sym_matvec_row_n(const Real* A, const Real* x, int i, int n) {
#if defined(__CUDA_ARCH__)
  if (n == N) {
    const Real* row = A + i * (i + 1) / 2;   // entries k <= i
    const Real* col = A + i;                 // entries k > i at col[k (k + 1) / 2]
    Real v = 0;
#pragma unroll
    for (int k = 0; k < N; ++k) { const Real a = *(k <= i ? row + k : col + k * (k + 1) / 2); v += a * x[k]; }
    return v;
  }
#endif
  return sym_matvec_row_cold(A, x, i, n);
}

// ---------------------------------------------------------------- kinematics (SURVEY B.1, B.2)
// r = a b for row-major 3x3 matrices (r must not alias a or b)
template <typename Real> UR3E_HD void mat_mul3(Real* r, const Real* a, const Real* b) {
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) r[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}

// Frames are composed as rotation matrices in three stages, so that the serial part (one step per tree level) is only a
// 3x3 product spread over 12 lanes per body:
//   A. every body in parallel: its frame relative to the parent, (L_b, t_b) = body offset * joint transform
//   B. level by level: R_b = R_p L_b, x_b = x_p + R_p t_b   (lane = one entry of R_b or x_b)
//   C. every body / site in parallel: inertial frame position, joint axis (cdof), site frames (geom frames are built by the
//      collision lanes that need them)
template <typename Real, typename D>
UR3E_HD void kin_frames(const DevModel<Real>& m, Arena<Real, D>& s) {   // stages A and B: xpos, xmat of every body
  auto& kin = s.u.kin;
  WARP_FOR(b, nb_<D>(m)) {
    Real* L = kin.lmat[b]; Real* t = kin.lpos[b];
    const int jk = m.body_jkind[b];
    if (b == 0) {
      for (int k = 0; k < 9; ++k) s.fr.k.xmat[0][k] = (k % 4 == 0) ? Real(1) : Real(0);
      for (int k = 0; k < 3; ++k) { s.xpos[0][k] = 0; s.fr.k.xipos[0][k] = 0; }
    } else if (jk == JK_FREE) {
      const int qa = m.body_qadr[b];
      Real q[4] = {s.st.qpos[qa + 3], s.st.qpos[qa + 4], s.st.qpos[qa + 5], s.st.qpos[qa + 6]};
      quat_normalize(q); quat2mat(L, q);
      for (int k = 0; k < 3; ++k) t[k] = s.st.qpos[qa + k];
    } else if (jk == JK_HINGE) {
      // joint rotation about the (unit) axis a by Rodrigues' formula; the joint anchor stays fixed in the parent frame
      const Real* a = m.jnt_axis[b]; const Real* jp = m.jnt_pos[b]; const Real* Rb = m.body_mat[b];
      Real sn, cs; Num<Real>::sincos(s.st.qpos[m.body_qadr[b]] - m.jnt_q0[b], &sn, &cs);
      const Real v = 1 - cs;
      const Real Rj[9] = {cs + v * a[0] * a[0], v * a[0] * a[1] - sn * a[2], v * a[0] * a[2] + sn * a[1],
                          v * a[0] * a[1] + sn * a[2], cs + v * a[1] * a[1], v * a[1] * a[2] - sn * a[0],
                          v * a[0] * a[2] - sn * a[1], v * a[1] * a[2] + sn * a[0], cs + v * a[2] * a[2]};
      mat_mul3(L, Rb, Rj);
      Real rj[3], d[3]; mat_vec3(rj, Rj, jp);
      for (int k = 0; k < 3; ++k) rj[k] = jp[k] - rj[k];
      mat_vec3(d, Rb, rj);
      for (int k = 0; k < 3; ++k) t[k] = m.body_pos[b][k] + d[k];
    } else {
      for (int k = 0; k < 9; ++k) L[k] = m.body_mat[b][k];
      for (int k = 0; k < 3; ++k) t[k] = m.body_pos[b][k];
    }
  }
  WARP_SYNC();
  for (int lev = 1; lev < nlevel_<D>(m); ++lev) {
    const int b0 = m.lev_start[lev], cnt = m.lev_start[lev + 1] - b0;
    WARP_FOR(i, 12 * cnt) {
      const int slot = i / 12, e = i - 12 * slot, b = m.lev_body[b0 + slot], p = m.body_parent[b];
      if (e < 9) {
        const int r = e / 3, c = e - 3 * r;
        const Real* Rp = s.fr.k.xmat[p] + 3 * r; const Real* L = kin.lmat[b] + c;
        s.fr.k.xmat[b][e] = Rp[0] * L[0] + Rp[1] * L[3] + Rp[2] * L[6];
      } else {
        const int r = e - 9;
        const Real* Rp = s.fr.k.xmat[p] + 3 * r; const Real* t = kin.lpos[b];
        s.xpos[b][r] = s.xpos[p][r] + Rp[0] * t[0] + Rp[1] * t[1] + Rp[2] * t[2];
      }
    }
    WARP_SYNC();
  }
}

template <typename Real, typename D>
UR3E_HD void kinematics(const DevModel<Real>& m, Arena<Real, D>& s) {
  kin_frames(m, s);
  WARP_FOR(i, nb_<D>(m) + nsite_<D>(m)) {
    if (i < nb_<D>(m)) {
      const int b = i;
      if (b > 0) {
        const Real* R = s.fr.k.xmat[b]; const Real* x = s.xpos[b];
        Real v[3]; mat_vec3(v, R, m.body_ipos[b]);
        for (int k = 0; k < 3; ++k) s.fr.k.xipos[b][k] = x[k] + v[k];
        const int jk = m.body_jkind[b];
        if (jk == JK_HINGE) {
          Real axis[3], anchor[3];
          mat_vec3(axis, R, m.jnt_axis[b]); mat_vec3(anchor, R, m.jnt_pos[b]);
          const Real* ref = s.xpos[m.body_root[b]];
          const Real off[3] = {ref[0] - x[0] - anchor[0], ref[1] - x[1] - anchor[1], ref[2] - x[2] - anchor[2]};
          Real* c = s.cdof[m.body_dadr[b]];
          c[0] = axis[0]; c[1] = axis[1]; c[2] = axis[2];
          cross3(c + 3, axis, off);
        } else if (jk == JK_FREE) {
          const int da = m.body_dadr[b];
          for (int a = 0; a < 3; ++a) {
            Real* ct = s.cdof[da + a]; Real* cr = s.cdof[da + 3 + a];
            for (int k = 0; k < 6; ++k) { ct[k] = 0; cr[k] = 0; }
            ct[3 + a] = 1;                                            // translation along world axis a
            cr[0] = R[a]; cr[1] = R[3 + a]; cr[2] = R[6 + a];         // rotation about body axis a, through the reference point
          }
        }
      }
    } else {
      const int j = i - nb_<D>(m), b = m.site_body[j]; Real v[3];
      mat_vec3(v, s.fr.k.xmat[b], m.site_pos[j]);
      for (int k = 0; k < 3; ++k) s.site_xpos[j][k] = s.xpos[b][k] + v[k];
      if (j == 0) mat_mul3(s.site_xmat[0], s.fr.k.xmat[b], m.site_mat[0]);
    }
  }
  WARP_SYNC();
}

// ---------------------------------------------------------------- CRBA + RNE (SURVEY B.3, B.4)
template <typename Real, typename D>
UR3E_HD void dynamics(const DevModel<Real>& m, Arena<Real, D>& s) {
  const int nb = nb_<D>(m), nv = nv_<D>(m);
  auto& y = s.u.dyn;
  // body inertias about the tree reference point + body velocities (sum over the dof chain)
  WARP_FOR(b, nb) {
    Real* ci = y.cinert[b];
    if (b == 0 || m.body_lastdof[b] < 0) { for (int k = 0; k < 10; ++k) ci[k] = 0; for (int k = 0; k < 6; ++k) y.cvel[b][k] = 0; }
    else {
      const Real* ref = s.xpos[m.body_root[b]];
      Real dif[3] = {s.fr.k.xipos[b][0] - ref[0], s.fr.k.xipos[b][1] - ref[1], s.fr.k.xipos[b][2] - ref[2]};
      Real R[9]; mat_mul3(R, s.fr.k.xmat[b], m.body_imat[b]);
      const Real* in = m.body_inertia[b]; Real mass = m.body_mass[b];
      Real t00 = 0, t11 = 0, t22 = 0, t01 = 0, t02 = 0, t12 = 0;
      for (int k = 0; k < 3; ++k) {
        t00 += R[k] * in[k] * R[k]; t11 += R[3 + k] * in[k] * R[3 + k]; t22 += R[6 + k] * in[k] * R[6 + k];
        t01 += R[k] * in[k] * R[3 + k]; t02 += R[k] * in[k] * R[6 + k]; t12 += R[3 + k] * in[k] * R[6 + k];
      }
      ci[0] = t00 + mass * (dif[1] * dif[1] + dif[2] * dif[2]); ci[1] = t11 + mass * (dif[0] * dif[0] + dif[2] * dif[2]);
      ci[2] = t22 + mass * (dif[0] * dif[0] + dif[1] * dif[1]);
      ci[3] = t01 - mass * dif[0] * dif[1]; ci[4] = t02 - mass * dif[0] * dif[2]; ci[5] = t12 - mass * dif[1] * dif[2];
      ci[6] = mass * dif[0]; ci[7] = mass * dif[1]; ci[8] = mass * dif[2]; ci[9] = mass;
      Real cv[6] = {0, 0, 0, 0, 0, 0};
      for (int d = m.body_lastdof[b]; d >= 0; d = m.dof_parent[d]) { Real qd = s.st.qvel[d]; for (int k = 0; k < 6; ++k) cv[k] += s.cdof[d][k] * qd; }
      for (int k = 0; k < 6; ++k) y.cvel[b][k] = cv[k];
    }
  }
  WARP_FOR(i, nv * (nv + 1) / 2) s.M[i] = 0;
  WARP_SYNC();
  // cdof_dot = (velocity before the dof) x cdof   (mj_comVel)
  WARP_FOR(d, nv) {
    int b = m.dof_body[d], fk = m.dof_free_k[d];
    Real* cd = y.cdof_dot[d];
    if (fk >= 0 && fk < 3) { for (int k = 0; k < 6; ++k) cd[k] = 0; }
    else {
      Real vel[6];
      for (int k = 0; k < 6; ++k) vel[k] = y.cvel[m.body_parent[b]][k];
      if (fk >= 3) { int da = m.body_dadr[b]; for (int i = 0; i < 3; ++i) for (int k = 0; k < 6; ++k) vel[k] += s.cdof[da + i][k] * s.st.qvel[da + i]; }
      cross_motion(cd, vel, s.cdof[d]);
    }
  }
  WARP_SYNC();
  // bias wrench of every body: I a + v x* I v, with a = -g + sum cdof_dot qvel over the chain (needs the body's own inertia)
  WARP_FOR(b, nb) {
    Real* f = y.cfrc[b];
    if (b == 0 || m.body_lastdof[b] < 0) { for (int k = 0; k < 6; ++k) f[k] = 0; }
    else {
      Real a[6] = {0, 0, 0, -m.gravity[0], -m.gravity[1], -m.gravity[2]};
      for (int d = m.body_lastdof[b]; d >= 0; d = m.dof_parent[d]) { Real qd = s.st.qvel[d]; for (int k = 0; k < 6; ++k) a[k] += y.cdof_dot[d][k] * qd; }
      Real t1[6], t2[6];
      mul_inert(f, y.cinert[b], a);
      mul_inert(t1, y.cinert[b], y.cvel[b]); cross_force(t2, y.cvel[b], t1);
      for (int k = 0; k < 6; ++k) f[k] += t2[k];
    }
  }
  WARP_SYNC();
  // composite inertias in place (lanes 0-9: one inertia component each) and subtree bias wrenches (lanes 10-15), both serial
  // down the (parent < child) body order
  // (one loop for both: a lane walks its own array with its own stride, so the two groups of lanes do not diverge)
  WARP_FOR(k, 16) {
    Real* const base = k < 10 ? &y.cinert[0][k] : &y.cfrc[0][k - 10];
    const int stride = k < 10 ? 10 : 6;
    for (int b = nb - 1; b > 0; --b) { const int p = m.body_parent[b]; if (p > 0) base[p * stride] += base[b * stride]; }
  }
  WARP_SYNC();
  // M: f_i = crb(body_i) cdof_i (stored over cdof_dot, which is dead) ; M_ij = cdof_j . f_i
  WARP_FOR(i, nv) mul_inert(y.cdof_dot[i], y.cinert[m.dof_body[i]], s.cdof[i]);
  WARP_SYNC();
  WARP_FOR(e, nM_<D>(m)) {
    int i = m.M_i[e], j = m.M_j[e];
    Real v = 0; for (int k = 0; k < 6; ++k) v += s.cdof[j][k] * y.cdof_dot[i][k];
    if (i == j) v += m.dof_armature[i];
    s.M[i * (i + 1) / 2 + j] = v;
  }
  // site linear velocities (mj_objectVelocity, world frame) for the observation
  WARP_FOR(j, nsite_<D>(m)) {
    int b = m.site_body[j];
    if (m.body_lastdof[b] < 0) { s.site_velp[j][0] = s.site_velp[j][1] = s.site_velp[j][2] = 0; }
    else {
      const Real* ref = s.xpos[m.body_root[b]]; const Real* cv = y.cvel[b];
      Real off[3] = {s.site_xpos[j][0] - ref[0], s.site_xpos[j][1] - ref[1], s.site_xpos[j][2] - ref[2]}, t[3];
      cross3(t, cv, off);
      for (int k = 0; k < 3; ++k) s.site_velp[j][k] = cv[3 + k] + t[k];
    }
  }
  // actuator forces (SURVEY B.5)
  WARP_FOR(a, nu_<D>(m)) {
    Real c = s.ctrl[a];
    if (m.act_ctrllimited[a]) c = rmin(rmax(c, m.act_ctrlrange[a][0]), m.act_ctrlrange[a][1]);
    Real len = 0, vel = 0;
    for (int k = 0; k < 2; ++k) { int d = m.act_dof[a][k]; if (d >= 0) { len += m.act_coef[a][k] * s.st.qpos[m.dof_qadr[d]]; vel += m.act_coef[a][k] * s.st.qvel[d]; } }
    Real f = m.act_gain[a] * c + m.act_bias[a][0] + m.act_bias[a][1] * len + m.act_bias[a][2] * vel;
    if (m.act_forcelimited[a]) f = rmin(rmax(f, m.act_forcerange[a][0]), m.act_forcerange[a][1]);
    s.act_force[a] = f;
  }
  WARP_SYNC();
  WARP_FOR(d, nv) {
    Real bias = 0; for (int k = 0; k < 6; ++k) bias += s.cdof[d][k] * y.cfrc[m.dof_body[d]][k];
    s.qfrc_bias[d] = bias;
    Real f = -m.dof_damping[d] * s.st.qvel[d];
    if (m.dof_free_k[d] < 0) f -= m.dof_stiffness[d] * (s.st.qpos[m.dof_qadr[d]] - m.dof_springref[d]);
    for (int k = 0; k < m.dof_nact[d]; ++k) f += m.dof_actcoef[d][k] * s.act_force[m.dof_act[d][k]];
    s.qfrc_smooth[d] = f - bias;
  }
  WARP_SYNC();
}

// ---------------------------------------------------------------- collision (SURVEY B.9)
template <typename Real> UR3E_HD void make_frame(Real* f) {
  normalize3(f);
  Real* y = f + 3;
  y[0] = 0; y[1] = 0; y[2] = 0;
  if (f[1] < Real(0.5) && f[1] > Real(-0.5)) y[1] = 1; else y[2] = 1;
  Real t = dot3(f, y);
  for (int k = 0; k < 3; ++k) y[k] -= t * f[k];
  normalize3(y);
  cross3(f + 6, f, y);
}

template <typename Real>
UR3E_HD int plane_box(const Real* ppos, const Real* pmat, const Real* bpos, const Real* bmat, const Real* size, Real margin, Real* out) {
  Real n[3] = {pmat[2], pmat[5], pmat[8]};
  Real dif[3] = {bpos[0] - ppos[0], bpos[1] - ppos[1], bpos[2] - ppos[2]};
  Real cd = dot3(dif, n);
  int cnt = 0;
  for (int i = 0; i < 8; ++i) {
    Real v[3] = {(i & 1) ? size[0] : -size[0], (i & 2) ? size[1] : -size[1], (i & 4) ? size[2] : -size[2]}, c[3];
    mat_vec3(c, bmat, v);
    Real ld = dot3(n, c);
    if (cd + ld > margin || ld > 0) continue;
    Real dist = cd + ld;
    for (int k = 0; k < 3; ++k) { out[3 + 4 * cnt + k] = c[k] + bpos[k] - n[k] * dist * Real(0.5); out[k] = n[k]; }
    out[3 + 4 * cnt + 3] = dist;
    if (++cnt >= 4) break;
  }
  return cnt;
}

template <typename Real>
UR3E_HD int clip_poly(const Real* px, const Real* py, int n, Real* ox, Real* oy, Real a, Real b, Real c) {
  // clips (px, py)[0..n) by a x + b y <= c into (ox, oy); the caller ping-pongs two buffers (no copy back)
  int k = 0;
  for (int i = 0; i < n; ++i) {
    int j = (i + 1 == n) ? 0 : i + 1;
    Real di = a * px[i] + b * py[i] - c, dj = a * px[j] + b * py[j] - c;
    if (di <= 0) { ox[k] = px[i]; oy[k] = py[i]; ++k; }
    if ((di < 0 && dj > 0) || (di > 0 && dj < 0)) { Real t = di / (di - dj); ox[k] = px[i] + t * (px[j] - px[i]); oy[k] = py[i] + t * (py[j] - py[i]); ++k; }
    if (k >= 15) break;
  }
  return k;
}

// box-box manifold; same rules as the oracle's box_box (oracle/ur3e_oracle.c), normal from box 1 to box 2.
// `out` is the slot's staging row (STAGE_W values, shared memory).  On entry it holds the two world frames (R1 = out[0, 9),
// R2 = out[9, 18)), so that no argument is passed by address from the caller's stack; the frames are dead once the
// clipping starts, and the row then holds one of the two clip polygons until the contact points overwrite it.
template <typename Real>
UR3E_PHASE int box_box(const Real* p1, const Real* s1, const Real* p2, const Real* s2, Real margin, Real* out) {
  const Real* const R1 = out; const Real* const R2 = out + 9;
  Real d[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]}, A1[3][3], A2[3][3];
  for (int i = 0; i < 3; ++i) for (int k = 0; k < 3; ++k) { A1[i][k] = R1[3 * k + i]; A2[i][k] = R2[3 * k + i]; }
  Real AC[3][3];
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) AC[i][j] = Num<Real>::abs(dot3(A1[i], A2[j]));
  Real best = -Num<Real>::big; int code = -1; Real bn[3] = {0, 0, 0};
  for (int i = 0; i < 3; ++i) {
    Real t = dot3(d, A1[i]), ra = s1[i], rb = s2[0] * AC[i][0] + s2[1] * AC[i][1] + s2[2] * AC[i][2];
    Real sep = Num<Real>::abs(t) - ra - rb;
    if (sep > margin) return 0;
    if (sep > best) { best = sep; code = i; Real sg = t < 0 ? Real(-1) : Real(1); for (int k = 0; k < 3; ++k) bn[k] = sg * A1[i][k]; }
  }
  for (int j = 0; j < 3; ++j) {
    Real t = dot3(d, A2[j]), ra = s1[0] * AC[0][j] + s1[1] * AC[1][j] + s1[2] * AC[2][j], rb = s2[j];
    Real sep = Num<Real>::abs(t) - ra - rb;
    if (sep > margin) return 0;
    if (sep > best + Real(1e-6) * (s1[0] + s1[1] + s1[2])) { best = sep; code = 3 + j; Real sg = t < 0 ? Real(-1) : Real(1); for (int k = 0; k < 3; ++k) bn[k] = sg * A2[j][k]; }
  }
  Real ebest = -Num<Real>::big; int ei = -1, ej = -1; Real en[3] = {0, 0, 0};
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) {
    Real ax[3]; cross3(ax, A1[i], A2[j]);
    Real l = Num<Real>::sqrt(dot3(ax, ax));
    if (l < Real(1e-6)) continue;
    for (int k = 0; k < 3; ++k) ax[k] /= l;
    Real t = dot3(d, ax), ra = 0, rb = 0;
    for (int k = 0; k < 3; ++k) { ra += s1[k] * Num<Real>::abs(dot3(A1[k], ax)); rb += s2[k] * Num<Real>::abs(dot3(A2[k], ax)); }
    Real sep = Num<Real>::abs(t) - ra - rb;
    if (sep > margin) return 0;
    if (sep > ebest) { ebest = sep; ei = i; ej = j; Real sg = t < 0 ? Real(-1) : Real(1); for (int k = 0; k < 3; ++k) en[k] = sg * ax[k]; }
  }
  if (ei >= 0 && ebest > best + Real(1e-3) * Num<Real>::abs(best) + Real(1e-9)) {
    Real c1[3] = {p1[0], p1[1], p1[2]}, c2[3] = {p2[0], p2[1], p2[2]};
    for (int a = 0; a < 3; ++a) if (a != ei) { Real sg = dot3(A1[a], en) > 0 ? Real(1) : Real(-1); for (int k = 0; k < 3; ++k) c1[k] += sg * s1[a] * A1[a][k]; }
    for (int a = 0; a < 3; ++a) if (a != ej) { Real sg = dot3(A2[a], en) > 0 ? Real(-1) : Real(1); for (int k = 0; k < 3; ++k) c2[k] += sg * s2[a] * A2[a][k]; }
    const Real u[3] = {R1[ei], R1[3 + ei], R1[6 + ei]}, v[3] = {R2[ej], R2[3 + ej], R2[6 + ej]};   // axes picked at run time: read from the frames (see below)
    Real w[3] = {c1[0] - c2[0], c1[1] - c2[1], c1[2] - c2[2]};
    Real b = dot3(u, v), dd = dot3(u, w), e = dot3(v, w), den = 1 - b * b;
    Real sa = (b * e - dd) / den, sb = (e - b * dd) / den;
    sa = rmin(rmax(sa, -s1[ei]), s1[ei]); sb = rmin(rmax(sb, -s2[ej]), s2[ej]);
    for (int k = 0; k < 3; ++k) { out[3 + k] = Real(0.5) * (c1[k] + sa * u[k] + c2[k] + sb * v[k]); out[k] = en[k]; }
    out[6] = ebest;
    return 1;
  }
  bool ref1 = code < 3; int ra = ref1 ? code : code - 3;
  const Real *rp = ref1 ? p1 : p2, *ip = ref1 ? p2 : p1, *rs = ref1 ? s1 : s2, *is = ref1 ? s2 : s1;
  // Axes chosen at run time are read from the frames themselves (axis a of a box = column a of its matrix): indexing the
  // register copies A1 / A2 dynamically would push them into local memory.
  const Real* RR = ref1 ? R1 : R2; const Real* IR = ref1 ? R2 : R1;
  Real nref[3]; for (int k = 0; k < 3; ++k) nref[k] = ref1 ? bn[k] : -bn[k];
  int ia = 0; Real mind = Num<Real>::big, isg = 1;
  for (int a = 0; a < 3; ++a) { Real t = IR[a] * nref[0] + IR[3 + a] * nref[1] + IR[6 + a] * nref[2]; if (-Num<Real>::abs(t) < mind) { mind = -Num<Real>::abs(t); ia = a; isg = t > 0 ? Real(-1) : Real(1); } }
  int iu = (ia + 1) % 3, iv = (ia + 2) % 3, ru = (ra + 1) % 3, rv = (ra + 2) % 3;
  const Real IAa[3] = {IR[ia], IR[3 + ia], IR[6 + ia]}, IAu[3] = {IR[iu], IR[3 + iu], IR[6 + iu]}, IAv[3] = {IR[iv], IR[3 + iv], IR[6 + iv]};
  const Real RAu[3] = {RR[ru], RR[3 + ru], RR[6 + ru]}, RAv[3] = {RR[rv], RR[3 + rv], RR[6 + rv]};
  const Real hia = is[ia], hiu = is[iu], hiv = is[iv];
  Real fc[3], rc[3];
  for (int k = 0; k < 3; ++k) { fc[k] = ip[k] + isg * hia * IAa[k]; rc[k] = rp[k] + rs[ra] * nref[k]; }
  Real px[16], py[16];
  for (int c = 0; c < 4; ++c) {
    Real su = (c == 0 || c == 3) ? Real(1) : Real(-1), sv = (c < 2) ? Real(1) : Real(-1), r[3];
    for (int k = 0; k < 3; ++k) r[k] = fc[k] + su * hiu * IAu[k] + sv * hiv * IAv[k] - rc[k];
    px[c] = dot3(r, RAu); py[c] = dot3(r, RAv);
  }
  int n = 4;
  static_assert(STAGE_W >= 2 * 16, "the second clip polygon lives in the staging row");
  Real* const qx = out; Real* const qy = out + 16;   // the frames are dead from here on (IAa / RAu / ... hold what is still needed)
  n = clip_poly(px, py, n, qx, qy, Real(1), Real(0), rs[ru]); n = clip_poly(qx, qy, n, px, py, Real(-1), Real(0), rs[ru]);
  n = clip_poly(px, py, n, qx, qy, Real(0), Real(1), rs[rv]); n = clip_poly(qx, qy, n, px, py, Real(0), Real(-1), rs[rv]);
  if (n == 0) return 0;
  Real ni[3]; for (int k = 0; k < 3; ++k) ni[k] = isg * IAa[k];
  Real nn = dot3(ni, nref);
  int cnt = 0;
  for (int c = 0; c < n && cnt < STAGE_PTS; ++c) {
    Real base[3], r[3];
    for (int k = 0; k < 3; ++k) { base[k] = rc[k] + px[c] * RAu[k] + py[c] * RAv[k]; r[k] = fc[k] - base[k]; }
    Real h = Num<Real>::abs(nn) > Real(1e-12) ? dot3(ni, r) / nn : Real(0);
    if (h > margin) continue;
    for (int k = 0; k < 3; ++k) { out[3 + 4 * cnt + k] = base[k] + Real(0.5) * h * nref[k]; out[k] = bn[k]; }
    out[3 + 4 * cnt + 3] = h;
    ++cnt;
  }
  return cnt;
}

// world position of geom g (its body's frame is still alive during the collision phase)
template <typename Real, typename D>
UR3E_HD void geom_world_pos(const DevModel<Real>& m, const Arena<Real, D>& s, int g, Real* x) {
  const int b = m.geom_body[g]; Real v[3];
  mat_vec3(v, s.fr.k.xmat[b], m.geom_pos[g]);
  for (int k = 0; k < 3; ++k) x[k] = s.xpos[b][k] + v[k];
}

// Broad phase over the model's static candidate list (lane = pair; bounding spheres / plane distance), then the narrow phase on
// the survivors only (lane = survivor; plane-box, box-box SAT + clipping), then compaction into the contact list in pair order.
template <typename Real, typename D>
UR3E_HD void collision(const DevModel<Real>& m, Arena<Real, D>& s) {
  if constexpr (!D::HAS_CONTACT) { s.ncon = 0; return; }
  else {
    const int np = np_<D>(m);
    WARP_FOR(g, ng_<D>(m)) geom_world_pos(m, s, g, s.cu.gpos[g]);
    WARP_SYNC();
    int nact = 0;
    for (int base = 0; base < np; base += 32) {
      const int cnt = np - base < 32 ? np - base : 32;
      int bits = 0;
      WARP_FOR(i, cnt) {
        const int p = base + i, code = m.pair_code[p], g1 = code & 255, g2 = (code >> 8) & 255;
        const Real* x1 = s.cu.gpos[g1]; const Real* x2 = s.cu.gpos[g2];
        const Real dd[3] = {x2[0] - x1[0], x2[1] - x1[1], x2[2] - x1[2]}, r = m.pair_rsum[p];
        const bool hit = (code >> 16) ? dot3(dd, m.geom_nrm[g1]) <= r : dot3(dd, dd) <= r * r;
        if (hit) bits |= (int)(1u << i);
      }
      bits = warp_or(bits);
      WARP_FOR(i, cnt) {
        if ((bits >> i) & 1) { const int slot = nact + popcount32(bits & (int)((1u << i) - 1u)); if (slot < D::MAXACT) s.act_pair[slot] = (uint8_t)(base + i); }
      }
      nact += popcount32(bits);
    }
    if (nact > D::MAXACT) { nact = D::MAXACT; IF_LANE0 s.overflow |= 1; }
    WARP_SYNC();
    WARP_FOR(a, nact) {
      const int p = s.act_pair[a], g1 = m.pair_g1[p], g2 = m.pair_g2[p];
      const Real margin = m.pair_margin[p];
      Real R1[9], R2[9];
      mat_mul3(R1, s.fr.k.xmat[m.geom_body[g1]], m.geom_mat[g1]); mat_mul3(R2, s.fr.k.xmat[m.geom_body[g2]], m.geom_mat[g2]);
      Real* st = s.u.stage[a];
      int n;
      if (m.geom_kind[g1] == GK_PLANE) {
        const Real x1[3] = {s.cu.gpos[g1][0], s.cu.gpos[g1][1], s.cu.gpos[g1][2]}, x2[3] = {s.cu.gpos[g2][0], s.cu.gpos[g2][1], s.cu.gpos[g2][2]};
        n = plane_box(x1, R1, x2, R2, m.geom_size[g2], margin, st);
      } else {
        // the out-of-line box_box takes everything through the arena: arrays passed by address would live on the stack
        for (int k = 0; k < 9; ++k) { st[k] = R1[k]; st[9 + k] = R2[k]; }
        n = box_box(s.cu.gpos[g1], m.geom_size[g1], s.cu.gpos[g2], m.geom_size[g2], margin, st);
      }
      int keep = 0;   // MuJoCo keeps a contact only when dist < margin
      for (int c = 0; c < n; ++c) if (st[3 + 4 * c + 3] < margin) { if (keep != c) for (int k = 0; k < 4; ++k) st[3 + 4 * keep + k] = st[3 + 4 * c + k]; ++keep; }
      s.stage_n[a] = (uint8_t)keep;
    }
    WARP_SYNC();
    int total = 0;
    for (int a = 0; a < nact; ++a) { int n = s.stage_n[a]; IF_LANE0 s.stage_off[a] = (uint8_t)total; total += n; }
    const int capc = s.cap_con;   // <= D::MAXCON; smaller only when the caller lowers the cap (ur3e_env_config.lite_max_contacts)
    int ncon = total > capc ? capc : total;
    IF_LANE0 { s.ncon = ncon; if (total > capc) s.overflow |= 1; }
    WARP_SYNC();
    WARP_FOR(i, nact * STAGE_PTS) {
      int a = i / STAGE_PTS, c = i % STAGE_PTS;
      int o = s.stage_off[a] + c;
      if (c < s.stage_n[a] && o < capc) {
        const Real* src = s.u.stage[a];
        for (int k = 0; k < 3; ++k) { s.con_pos[o][k] = src[3 + 4 * c + k]; s.cu.frame[o][k] = src[k]; }
        s.con_dist[o] = src[3 + 4 * c + 3]; s.con_pair[o] = s.act_pair[a];
        make_frame(s.cu.frame[o]);
      }
    }
    WARP_SYNC();
  }
}

// ---------------------------------------------------------------- constraints (SURVEY B.6)
// translational jacobian column of dof d for a world point rigidly attached to `body`
template <typename Real, typename D>
UR3E_HD void jac_col(const DevModel<Real>& m, const Arena<Real, D>& s, int d, const Real* point, int body, Real* out) {
  if ((m.body_dofmask[body] >> d) & 1u) {
    const Real* ref = s.xpos[m.body_root[body]]; const Real* c = s.cdof[d];
    Real off[3] = {point[0] - ref[0], point[1] - ref[1], point[2] - ref[2]}, t[3];
    cross3(t, c, off);
    out[0] = c[3] + t[0]; out[1] = c[4] + t[1]; out[2] = c[5] + t[2];
  } else { out[0] = 0; out[1] = 0; out[2] = 0; }
}

// general solimp power (never taken by the reference scenes, whose power is 2): x^p for x in (0, 1) through exp2(p log2 x), a
// handful of inline instructions in float (powf is ~700 and a call would cost the hot path registers)
template <typename Real> UR3E_HD Real impedance_pow(Real x, Real s3, Real s4) {
  if (x <= s3) return Num<Real>::pow_pos(x, s4) / Num<Real>::pow_pos(s3, s4 - 1);
  return 1 - Num<Real>::pow_pos(1 - x, s4) / Num<Real>::pow_pos(1 - s3, s4 - 1);
}
template <typename Real> UR3E_HD Real impedance(const Real* si, Real pos, Real margin) {
  const Real lo = Real(0.0001), hi = Real(0.9999);
  Real s0 = rmin(rmax(si[0], lo), hi), s1 = rmin(rmax(si[1], lo), hi), s2 = rmax(si[2], Real(0)), s3 = rmin(rmax(si[3], lo), hi), s4 = rmax(si[4], Real(1));
  if (s0 == s1 || s2 <= Num<Real>::minval) return Real(0.5) * (s0 + s1);
  Real x = (pos - margin) / s2; if (x < 0) x = -x;
  if (x >= 1 || x <= 0) return x >= 1 ? s1 : s0;
  Real y;
  if (s4 == 1) y = x;
  else if (s4 == 2) y = x <= s3 ? x * x / s3 : 1 - (1 - x) * (1 - x) / (1 - s3);
  else y = impedance_pow(x, s3, s4);
  return s0 + y * (s1 - s0);
}

template <typename Real> UR3E_HD void kb_params(const Real* solref, const Real* solimp, Real timestep, Real* K, Real* B) {
  Real dmax = rmin(rmax(solimp[1], Real(0.0001)), Real(0.9999));
  if (solref[0] > 0) {
    Real tc = rmax(solref[0], 2 * timestep), dr = solref[1];
    *K = 1 / rmax(Num<Real>::minval, dmax * dmax * tc * tc * dr * dr); *B = 2 / rmax(Num<Real>::minval, dmax * tc);
  } else { *K = -solref[0] / rmax(Num<Real>::minval, dmax * dmax); *B = -solref[1] / rmax(Num<Real>::minval, dmax); }
}

template <typename Real> UR3E_HD Real dense_dot_cold(const Real* J, const Real* x, int n) {
  Real v = 0;
#pragma unroll 1
  for (int k = 0; k < n; ++k) v += J[k] * x[k];
  return v;
}
// J[r] . x for any row (dense rows read the stored Jacobian, sparse rows are one or two entries)
template <typename Real, typename D>
UR3E_HD Real row_dot(const DevModel<Real>& m, const Arena<Real, D>& s, int r, const Real* x) {
  if (r < s.nd) {
    const Real* J = s.u.efc_J[r];
#if defined(__CUDA_ARCH__)
    // float rows of the full size: five 128-bit loads (16-byte aligned rows of 80 bytes are bank-conflict free across lanes)
    if constexpr (sizeof(Real) == 4 && D::NV % 4 == 0) {
      if (nv_<D>(m) == D::NV) {
        const float4* J4 = reinterpret_cast<const float4*>(J);
        float v = 0;
#pragma unroll
        for (int q = 0; q < D::NV / 4; ++q) { const float4 j = J4[q]; v += j.x * x[4 * q] + j.y * x[4 * q + 1] + j.z * x[4 * q + 2] + j.w * x[4 * q + 3]; }
        return v;
      }
    }
#endif
    return dense_dot_cold(J, x, nv_<D>(m));
  }
  const int t = s.efc_type[r], id = s.efc_id[r];
  if (t == ROW_EQJ) { const int d2 = m.eq_o2[id]; Real v = x[m.eq_o1[id]]; if (d2 >= 0) v -= s.eqj_deriv[id] * x[d2]; return v; }
  return t == ROW_LIMIT_HI ? -x[id] : x[id];
}
// entry of joint-equality row r in column d (d is one of the row's two dofs): 1 on the first dof, -polynomial derivative on the second
template <typename Real, typename D>
UR3E_HD Real eqj_coef(const DevModel<Real>& m, const Arena<Real, D>& s, int d, int r) {
  const int id = s.efc_id[r];
  return m.eq_o1[id] == d ? Real(1) : -s.eqj_deriv[id];
}
// sum_r J[r][d] f[r] over all rows
template <typename Real, typename D>
UR3E_HD Real col_dot(const DevModel<Real>& m, const Arena<Real, D>& s, int d, const Real* f) {
  (void)m;
  Real v = 0;
#pragma unroll 4
  for (int r = 0; r < s.nd; ++r) v += s.u.efc_J[r][d] * f[r];
  int r = s.sp_ej[d]; if (r != 255) v += eqj_coef(m, s, d, r) * f[r];
  r = s.sp_fl[d]; if (r != 255) v += f[r];
  r = s.sp_lo[d]; if (r != 255) v += f[r];
  r = s.sp_hi[d]; if (r != 255) v -= f[r];
  return v;
}

template <typename Real, typename D>
UR3E_HD void make_constraint(const DevModel<Real>& m, Arena<Real, D>& s) {
  const int nv = nv_<D>(m);
  // row budget: dense rows = connect equalities + contacts (3 rows each), sparse rows = joint equalities, friction loss, limits
  const int ndeq = ndeq_<D>(m), nej = nej_<D>(m);
  const int nf = nfl_<D>(m);
  int mlo = 0, mhi = 0;   // bit d: lower / upper limit of dof d is active (dist < margin)
  WARP_FOR(d, nv) {
    if (m.dof_limited[d]) {
      Real q = s.st.qpos[m.dof_qadr[d]];
      if ((q - m.dof_range[d][0]) < m.dof_margin[d]) mlo |= 1 << d;
      if ((m.dof_range[d][1] - q) < m.dof_margin[d]) mhi |= 1 << d;
    }
  }
  mlo = warp_or(mlo); mhi = warp_or(mhi);
  int nl = popcount32(mlo) + popcount32(mhi);
  const int cape = s.cap_efc;   // <= D::MAXEFC
  int ncon = s.ncon;
  {
    int room = cape - ndeq - nej - nf - nl, roomd = D::MAXDENSE - ndeq;
    if (room < 0) { room = 0; }
    int cmax = (room < roomd ? room : roomd) / 3;
    if (cmax < 0) cmax = 0;
    if (ncon > cmax) { ncon = cmax; IF_LANE0 { s.overflow |= 2; s.ncon = ncon; } }
  }
  const int base_c = ndeq, nd = ndeq + 3 * ncon, rej0 = nd, rf0 = nd + nej, rl0 = rf0 + nf;
  int nefc = rl0 + nl;
  if (nefc > cape) { nefc = cape; IF_LANE0 s.overflow |= 2; }
  // row groups: dense rows that share one column set (used by the Hessian assembly)
  int ngrp = 0, coupled = 0;
  const int lowmask = (int)((1u << split_<D>(m)) - 1u);
  auto spans = [lowmask](int mask) { return (mask & lowmask) != 0 && (mask & ~lowmask) != 0; };
  for (int e = 0; e < neq_<D>(m); ++e) if (m.eq_kind[e] != EK_CONNECT && m.eq_o2[e] >= 0) coupled |= spans((1 << m.eq_o1[e]) | (1 << m.eq_o2[e]));
  {
    int row = 0;
    for (int e = 0; e < neq_<D>(m); ++e) if (m.eq_kind[e] == EK_CONNECT) {
      const int mask = (int)(m.body_dofmask[m.eq_o1[e]] | m.body_dofmask[m.eq_o2[e]]);
      IF_LANE0 { s.grp_row0[ngrp] = (uint8_t)row; s.grp_nrow[ngrp] = 3; s.grp_mask[ngrp] = mask; }
      coupled |= spans(mask);
      ++ngrp; row += 3;
    }
    if constexpr (D::HAS_CONTACT) {
      // consecutive contacts between the same two bodies share one column set (e.g. both boxes of a pad against the mug): one group
      int prev1 = -1, prev2 = -1;
      for (int c = 0; c < ncon; ++c) {
        const int p = s.con_pair[c], b1 = m.geom_body[m.pair_g1[p]], b2 = m.geom_body[m.pair_g2[p]];
        if (b1 != prev1 || b2 != prev2) {
          const int mask = (int)(m.body_dofmask[b1] ^ m.body_dofmask[b2]);
          IF_LANE0 { s.grp_row0[ngrp] = (uint8_t)(base_c + 3 * c); s.grp_nrow[ngrp] = 0; s.grp_mask[ngrp] = mask; }
          coupled |= spans(mask);
          ++ngrp; prev1 = b1; prev2 = b2;
        }
        IF_LANE0 s.grp_nrow[ngrp - 1] += 3;
      }
    }
  }
  IF_LANE0 { s.coupled = (short)coupled; s.ne = ndeq + nej; s.nf = nf; s.nl = nl; s.nefc = nefc; s.ngrp = ngrp; s.lim_lo = mlo; s.lim_hi = mhi; s.nd = nd; s.rf0 = rf0; s.rl0 = rl0; }
  WARP_FOR(d, nv) {
    const int k = m.dof_flrow[d], below = (1 << d) - 1;
    int r = rl0 + popcount32(mlo & below) + popcount32(mhi & below);
    s.sp_fl[d] = (uint8_t)((k >= 0 && rf0 + k < nefc) ? rf0 + k : 255);
    s.sp_lo[d] = (uint8_t)((((mlo >> d) & 1) && r < nefc) ? r : 255);
    if ((mlo >> d) & 1) ++r;
    s.sp_hi[d] = (uint8_t)((((mhi >> d) & 1) && r < nefc) ? r : 255);
    s.sp_ej[d] = 255;
  }
  WARP_SYNC();
  // rows: efc_aref temporarily holds pos, efc_jv holds margin
  {
    int row = 0, rj = rej0;
    for (int e = 0; e < neq_<D>(m); ++e) {
      if (m.eq_kind[e] == EK_CONNECT) {
        int b1 = m.eq_o1[e], b2 = m.eq_o2[e];
        Real a1[3], a2[3], v[3];
        mat_vec3(v, s.fr.k.xmat[b1], m.eq_data[e]); for (int k = 0; k < 3; ++k) a1[k] = s.xpos[b1][k] + v[k];
        mat_vec3(v, s.fr.k.xmat[b2], m.eq_data[e] + 3); for (int k = 0; k < 3; ++k) a2[k] = s.xpos[b2][k] + v[k];
        WARP_FOR(d, nv) {
          Real j1[3], j2[3]; jac_col(m, s, d, a1, b1, j1); jac_col(m, s, d, a2, b2, j2);
          for (int r = 0; r < 3; ++r) s.u.efc_J[row + r][d] = j1[r] - j2[r];
        }
        WARP_FOR(r, 3) { s.efc_aref[row + r] = r == 0 ? a1[0] - a2[0] : (r == 1 ? a1[1] - a2[1] : a1[2] - a2[2]); s.efc_jv[row + r] = 0; s.efc_type[row + r] = ROW_EQ; s.efc_id[row + r] = (uint8_t)e; }
        row += 3;
      } else {
        IF_LANE0 {
          int d1 = m.eq_o1[e], d2 = m.eq_o2[e];
          const Real* c = m.eq_data[e];
          Real p1 = s.st.qpos[m.dof_qadr[d1]] - m.qpos0[m.dof_qadr[d1]], pos, deriv = 0;
          if (d2 >= 0) {
            Real p2 = s.st.qpos[m.dof_qadr[d2]] - m.qpos0[m.dof_qadr[d2]];
            pos = p1 - (c[0] + p2 * (c[1] + p2 * (c[2] + p2 * (c[3] + p2 * c[4]))));
            deriv = c[1] + p2 * (2 * c[2] + p2 * (3 * c[3] + p2 * 4 * c[4]));
          } else pos = p1 - c[0];
          s.eqj_deriv[e] = deriv;
          if (rj < nefc) { s.sp_ej[d1] = (uint8_t)rj; if (d2 >= 0) s.sp_ej[d2] = (uint8_t)rj; }
          if (rj < D::MAXEFC) { s.efc_aref[rj] = pos; s.efc_jv[rj] = 0; s.efc_type[rj] = ROW_EQJ; s.efc_id[rj] = (uint8_t)e; }
        }
        rj += 1;
      }
    }
  }
  WARP_FOR(k, nf) {
    int d = m.fl_dof[k], r = rf0 + k;
    if (r < D::MAXEFC) { s.efc_aref[r] = 0; s.efc_jv[r] = 0; s.efc_type[r] = ROW_FRICTION; s.efc_id[r] = (uint8_t)d; }
  }
  WARP_FOR(i, 2 * nv) {
    int d = i >> 1, k = i & 1;
    int active = ((k == 0 ? mlo : mhi) >> d) & 1;
    if (active) {
      int below = (1 << d) - 1;
      int r = rl0 + popcount32(mlo & below) + popcount32(mhi & below) + (k == 1 ? ((mlo >> d) & 1) : 0);
      if (r < D::MAXEFC) {
        Real q = s.st.qpos[m.dof_qadr[d]];
        s.efc_aref[r] = k == 0 ? q - m.dof_range[d][0] : m.dof_range[d][1] - q;
        s.efc_jv[r] = m.dof_margin[d]; s.efc_type[r] = k == 0 ? ROW_LIMIT_LO : ROW_LIMIT_HI; s.efc_id[r] = (uint8_t)d;
      }
    }
  }
  if constexpr (D::HAS_CONTACT) {
    WARP_FOR(i, ncon * nv) {
      int c = i / nv, d = i - c * nv, p = s.con_pair[c];
      int b1 = m.geom_body[m.pair_g1[p]], b2 = m.geom_body[m.pair_g2[p]];
      Real j1[3], j2[3]; jac_col(m, s, d, s.con_pos[c], b1, j1); jac_col(m, s, d, s.con_pos[c], b2, j2);
      Real dj[3] = {j2[0] - j1[0], j2[1] - j1[1], j2[2] - j1[2]};
      int r0 = base_c + 3 * c;
      for (int r = 0; r < 3; ++r) s.u.efc_J[r0 + r][d] = dot3(s.cu.frame[c] + 3 * r, dj);
    }
    WARP_FOR(i, 3 * ncon) {
      int c = i / 3, r = i - 3 * c, row = base_c + i, p = s.con_pair[c];
      s.efc_aref[row] = r == 0 ? s.con_dist[c] : Real(0); s.efc_jv[row] = r == 0 ? m.pair_includemargin[p] : Real(0);
      s.efc_type[row] = (uint8_t)(ROW_CON_N + r); s.efc_id[row] = (uint8_t)c;
      if (r == 0) s.con_row[c] = (uint8_t)row;
    }
  }
  WARP_SYNC();
  // impedance, K/B, R, D, aref  (mj_makeImpedance + mj_referenceConstraint)
  WARP_FOR(r, nefc) {
    int t = s.efc_type[r], id = s.efc_id[r];
    Real pos = s.efc_aref[r], margin = s.efc_jv[r];
    const Real *solref, *solimp; Real diag; bool fric = false;
    if (t == ROW_EQ || t == ROW_EQJ) { solref = m.eq_solref[id]; solimp = m.eq_solimp[id]; diag = m.eq_invw[id]; }
    else if (t == ROW_FRICTION) { solref = m.dof_fl_solref[id]; solimp = m.dof_fl_solimp[id]; diag = m.dof_invw[id]; fric = true; }
    else if (t == ROW_LIMIT_LO || t == ROW_LIMIT_HI) { solref = m.dof_lim_solref[id]; solimp = m.dof_lim_solimp[id]; diag = m.dof_invw[id]; }
    else {
      int p = s.con_pair[id]; solref = m.pair_solref[p]; solimp = m.pair_solimp[p]; diag = m.pair_invw[p];
      if (t != ROW_CON_N) { fric = true; pos = 0; margin = 0; }
    }
    Real K, B; kb_params(solref, solimp, m.timestep, &K, &B);
    Real imp = impedance(solimp, pos, margin);
    Real R = rmax(Num<Real>::minval, (1 - imp) * diag / imp);
    if (t >= ROW_CON_N) {
      // elliptic cone: friction rows share the normal row's R scaled by 1/impratio (and by the friction ratio)
      int p = s.con_pair[id];
      Real impn = impedance(solimp, s.con_dist[id], m.pair_includemargin[p]);
      Real Rn = rmax(Num<Real>::minval, (1 - impn) * diag / impn);
      Real R1 = Rn / rmax(Num<Real>::minval, m.impratio);
      if (t == ROW_CON_N) { R = Rn; s.con_mu[id] = m.pair_friction[p][0] * Num<Real>::sqrt(R1 / Rn); }
      else if (t == ROW_CON_T1) R = R1;
      else R = R1 * m.pair_friction[p][0] * m.pair_friction[p][0] / (m.pair_friction[p][1] * m.pair_friction[p][1]);
    }
    if (fric) K = 0;
    const Real vel = row_dot(m, s, r, s.st.qvel);
    s.efc_D[r] = 1 / R;
    s.efc_aref[r] = -B * vel - K * imp * (pos - margin);
  }
  WARP_SYNC();
}

// ---------------------------------------------------------------- dense SPD solve on the augmented matrix
// Input: packed lower triangle s.fr.n.H (row i at i(i+1)/2; triangular offsets mod 32 are distinct, so one row per lane is
// bank-conflict free), rows 0..n-1 = SPD matrix, row n = right-hand side.  Output x[0..n) (shared memory).
// Right-looking Cholesky with one row per lane: at step k lane i (> k) scales its entry of column k and applies the
// rank-1 update to its own row, reading the raw column k as warp-wide broadcasts; one __syncwarp per step.  Loops are
// deliberately kept rolled: the step's code has to stay resident in the SM's 32 KB instruction cache (profiles/r1_summary.md).
// The right-hand side rides along as row n, so after the last step it holds y = L^-1 rhs; the back-substitution then
// runs column by column with the 1/diagonal saved during the factorisation.
template <typename Real, typename D>
UR3E_PHASE void chol_solve_aug(Arena<Real, D>& s, int n, Real* x) {
  // Factor (unscaled) with the forward substitution folded in: after step k, raw[i][k] = L[i][k] * L[k][k] and the
  // right-hand side (kept in y) has had column k eliminated.  Exact zeros (block / tree sparsity of M + J^T D J) are skipped.
  Real* y = s.colbuf[0];
  Real* const A = s.fr.n.H;
  WARP_FOR(k, n) y[k] = A[n * (n + 1) / 2 + k];
  WARP_SYNC();
  // the longest rows get a second lane: rows n-nh .. n-1 are updated by two lanes, each taking half of the column range
  const int nh = n > 8 ? ((n - 8) < (32 - n) ? (n - 8) : (32 - n)) : 0;
#pragma unroll 1
  for (int k = 0; k < n; ++k) {
    Real d = A[k * (k + 1) / 2 + k];
    d = d > Num<Real>::minval ? d : Num<Real>::minval;
    const Real inv = Real(1) / d, yk = y[k];
    WARP_FOR(it, n + nh) {
      const bool helper = it >= n;
      const int i = helper ? (n - nh) + (it - n) : it;
      if (i > k) {
        Real* row = A + i * (i + 1) / 2;
        const Real t = row[k] * inv;
        if (t != 0) {
          int lo = k + 1, hi = i;
          if (i >= n - nh) { const int mid = (lo + hi) >> 1; if (helper) lo = mid + 1; else hi = mid; }
          if (!helper) y[i] -= t * yk;
#pragma unroll 4
          for (int j = lo; j <= hi; ++j) row[j] -= t * A[j * (j + 1) / 2 + k];
        }
      }
    }
    WARP_SYNC();
  }
  // scale to the true factor once: L[i][k] = raw[i][k] / sqrt(d_k), z = L^-1 b, and keep 1 / L_kk
  WARP_FOR(k, n) {
    Real d = A[k * (k + 1) / 2 + k];
    d = d > Num<Real>::minval ? d : Num<Real>::minval;
    const Real rs = Real(1) / Num<Real>::sqrt(d);
    s.dinv[k] = rs;
    y[k] *= rs;
  }
  WARP_SYNC();
  WARP_FOR(i, n) { Real* row = A + i * (i + 1) / 2;
#pragma unroll 4
    for (int k = 0; k < i; ++k) row[k] *= s.dinv[k]; }
  WARP_SYNC();
  // back substitution L^T x = z; x is only ever written
#pragma unroll 1
  for (int k = n - 1; k >= 0; --k) {
    const Real xk = y[k] * s.dinv[k];
    const Real* Lk = A + k * (k + 1) / 2;
    WARP_FOR(i, k + 1) { if (i == k) x[i] = xk; else y[i] -= Lk[i] * xk; }
    WARP_SYNC();
  }
}

// ---------------------------------------------------------------- register-resident SPD solve (device only)
// Same right-looking elimination as chol_solve_aug, but lane i keeps row i of the matrix in registers (lane N the right-hand
// side) and the column entries travel by warp shuffle: step k costs one SHFL + one FFMA per remaining column for the whole
// warp, with no shared-memory traffic and no loop / address arithmetic (~25 instructions per column instead of ~200).
// Fully unrolled straight-line code (register indices must be static); it stays I-cache friendly because it is ONE
// out-of-line copy used by every Newton iteration and by the Euler step, and the warps of a block reach it at about the same time.
// Upper-triangle registers hold garbage that is never read by a valid lane.  Rows n..N-1 (model smaller than the size class)
// are identity rows, so the padded system has the same solution.  The unit factor L overwrites `tri`, w = D^-1 L^-1 rhs
// overwrites `rhs`; the back-substitution then runs with one unknown per lane (x_k broadcast by shuffle, L[k][lane] from
// shared memory).  `x` may alias `rhs`.
#ifndef UR3E_REG_CHOL
#define UR3E_REG_CHOL 1
#endif
#if defined(__CUDA_ARCH__) && UR3E_REG_CHOL
// `coupled` = false promises that the block [S, N) x [0, S) of the matrix is exactly zero: the updates of the columns >= S
// by the steps k < S are then exact no-ops for every row (and for the right-hand side) and are skipped -- 84 of the 190
// shuffle + FMA pairs for main.xml with the mug resting (S = 14).
template <typename Real, int N, int S = N>
__device__ __forceinline__ void chol_solve_reg_body(Real* tri, Real* rhs, int n, Real* x, bool coupled = true) {
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = UR3E_LANE;
  const bool isrow = lane < n, isrhs = lane == N;
  Real* const row = isrow ? tri + lane * (lane + 1) / 2 : rhs;
  const int jmax = isrow ? lane : (isrhs ? n - 1 : -1);   // this lane owns entries 0..jmax of `row`
  Real a[N];
  if (n == N) {
    // full-size matrix: plain loads.  Entries beyond a row's diagonal read the neighbouring rows (in bounds) and lanes > N read
    // the right-hand side: garbage that stays in registers no valid lane ever reads
#pragma unroll
    for (int j = 0; j < N; ++j) a[j] = row[j];
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j) {
      const Real ld = row[j <= jmax ? j : 0];
      a[j] = j <= jmax ? ld : ((!isrow && j == lane) ? Real(1) : Real(0));
    }
  }
  const int nstore = isrhs ? jmax + 1 : jmax;   // this lane stores a[k] for k < nstore: the strictly-lower L entries of its row; all of w
  // A = L D L^T with unit L: after step k register a[k] of lane i > k holds L[i][k]; lane N ends with w
#pragma unroll
  for (int k = 0; k < N; ++k) {
    Real d = __shfl_sync(FULL, a[k], k);
    d = d > Num<Real>::minval ? d : Num<Real>::minval;
    const Real t = a[k] * (Real(1) / d);
    if (k < S) {
#pragma unroll
      for (int j = k + 1; j < S; ++j) a[j] -= t * __shfl_sync(FULL, a[k], j);
      if (coupled) {
#pragma unroll
        for (int j = S; j < N; ++j) a[j] -= t * __shfl_sync(FULL, a[k], j);
      }
    } else {
#pragma unroll
      for (int j = k + 1; j < N; ++j) a[j] -= t * __shfl_sync(FULL, a[k], j);
    }
    if (k < nstore) row[k] = t;   // stored as soon as it is final, which frees the register
  }
  __syncwarp();
  Real xi = lane < n ? rhs[lane] : Real(0);
#pragma unroll
  for (int k = N - 1; k > 0; --k) {
    const Real xk = __shfl_sync(FULL, xi, k);
    if (lane < k && k < n) xi -= tri[k * (k + 1) / 2 + lane] * xk;
  }
  __syncwarp();
  if (lane < n) x[lane] = xi;
  __syncwarp();
}
template <typename Real, int N, int S>
__device__ __noinline__ void chol_solve_reg(Real* tri, Real* rhs, int n, Real* x, bool coupled) { chol_solve_reg_body<Real, N, S>(tri, rhs, n, x, coupled); }
#endif

// ---------------------------------------------------------------- Newton solver on the primal problem (SURVEY B.7)
// per-row cost derivative bookkeeping; cone contacts are processed by the lane that owns their normal row
template <typename Real, typename D>
UR3E_HD void constraint_update(const DevModel<Real>& m, Arena<Real, D>& s, bool want_hess) {
  WARP_FOR(r, s.nefc) {
    int t = s.efc_type[r];
    Real Dr = s.efc_D[r], x = s.efc_jar[r];
    if (t == ROW_EQ || t == ROW_EQJ) { s.efc_force[r] = -Dr * x; s.efc_Dact[r] = Dr; }
    else if (t == ROW_FRICTION) {
      Real f = m.dof_frictionloss[s.efc_id[r]], rf = f / Dr;
      if (x <= -rf) { s.efc_force[r] = f; s.efc_Dact[r] = 0; }
      else if (x >= rf) { s.efc_force[r] = -f; s.efc_Dact[r] = 0; }
      else { s.efc_force[r] = -Dr * x; s.efc_Dact[r] = Dr; }
    } else if (t == ROW_LIMIT_LO || t == ROW_LIMIT_HI) {
      if (x < 0) { s.efc_force[r] = -Dr * x; s.efc_Dact[r] = Dr; } else { s.efc_force[r] = 0; s.efc_Dact[r] = 0; }
    } else if (t == ROW_CON_N) {
      int c = s.efc_id[r], p = s.con_pair[c];
      Real mu = s.con_mu[c], f1 = m.pair_friction[p][0], f2 = m.pair_friction[p][1];
      Real U0 = x * mu, U1 = s.efc_jar[r + 1] * f1, U2 = s.efc_jar[r + 2] * f2;
      Real T = Num<Real>::sqrt(U1 * U1 + U2 * U2), N = U0;
      Real* Hc = s.cu.frame[c] + 3;
      if (N >= mu * T || (T <= 0 && N >= 0)) {
        for (int j = 0; j < 3; ++j) { s.efc_force[r + j] = 0; s.efc_Dact[r + j] = 0; }
        Hc[0] = -1;   // marker: no cone hessian
      } else if (mu * N + T <= 0 || (T <= 0 && N < 0)) {
        for (int j = 0; j < 3; ++j) { s.efc_force[r + j] = -s.efc_D[r + j] * s.efc_jar[r + j]; s.efc_Dact[r + j] = s.efc_D[r + j]; }
        Hc[0] = -1;
      } else {
        Real Dm = Dr / (mu * mu * (1 + mu * mu)), NmT = N - mu * T;
        Real f0 = -Dm * NmT * mu;
        s.efc_force[r] = f0; s.efc_force[r + 1] = -f0 / T * U1 * f1; s.efc_force[r + 2] = -f0 / T * U2 * f2;
        for (int j = 0; j < 3; ++j) s.efc_Dact[r + j] = 0;
        if (want_hess) {
          Real u1 = U1 / T, u2 = U2 / T, a = Dm * mu * mu, b = -Dm * mu * NmT / T;
          // symmetric 3x3 wrt jar: [00, 01, 02, 11, 12, 22]
          Hc[0] = Dm * mu * mu; Hc[1] = -Dm * mu * u1 * mu * f1; Hc[2] = -Dm * mu * u2 * mu * f2;
          Hc[3] = (a * u1 * u1 + b * (1 - u1 * u1)) * f1 * f1; Hc[4] = (a * u1 * u2 - b * u1 * u2) * f1 * f2; Hc[5] = (a * u2 * u2 + b * (1 - u2 * u2)) * f2 * f2;
        } else Hc[0] = 0;
      }
    }
  }
  WARP_SYNC();
}

// derivative / curvature of the cost along qacc + alpha * search (constraint part)
template <typename Real, typename D>
UR3E_HD void line_eval(const DevModel<Real>& m, const Arena<Real, D>& s, Real alpha, Real g1, Real g2, Real* dphi, Real* ddphi) {
  Real p1 = 0, p2 = 0;
  WARP_FOR(r, s.nefc) {
    int t = s.efc_type[r];
    Real Dr = s.efc_D[r], v = s.efc_jv[r], x = s.efc_jar[r] + alpha * v;
    if (t == ROW_EQ || t == ROW_EQJ) { p1 += Dr * x * v; p2 += Dr * v * v; }
    else if (t == ROW_FRICTION) {
      Real f = m.dof_frictionloss[s.efc_id[r]], rf = f / Dr;
      if (x <= -rf) p1 -= f * v; else if (x >= rf) p1 += f * v; else { p1 += Dr * x * v; p2 += Dr * v * v; }
    } else if (t == ROW_LIMIT_LO || t == ROW_LIMIT_HI) { if (x < 0) { p1 += Dr * x * v; p2 += Dr * v * v; } }
    else if (t == ROW_CON_N) {
      int c = s.efc_id[r], p = s.con_pair[c];
      Real mu = s.con_mu[c], f1 = m.pair_friction[p][0], f2 = m.pair_friction[p][1];
      Real x1 = s.efc_jar[r + 1] + alpha * s.efc_jv[r + 1], x2 = s.efc_jar[r + 2] + alpha * s.efc_jv[r + 2];
      Real U0 = x * mu, U1 = x1 * f1, U2 = x2 * f2, V0 = v * mu, V1 = s.efc_jv[r + 1] * f1, V2 = s.efc_jv[r + 2] * f2;
      Real T = Num<Real>::sqrt(U1 * U1 + U2 * U2), N = U0;
      if (N >= mu * T || (T <= 0 && N >= 0)) { }
      else if (mu * N + T <= 0 || (T <= 0 && N < 0)) {
        p1 += Dr * x * v + s.efc_D[r + 1] * x1 * s.efc_jv[r + 1] + s.efc_D[r + 2] * x2 * s.efc_jv[r + 2];
        p2 += Dr * v * v + s.efc_D[r + 1] * s.efc_jv[r + 1] * s.efc_jv[r + 1] + s.efc_D[r + 2] * s.efc_jv[r + 2] * s.efc_jv[r + 2];
      } else {
        Real Dm = Dr / (mu * mu * (1 + mu * mu)), NmT = N - mu * T;
        Real UV = U1 * V1 + U2 * V2, VV = V1 * V1 + V2 * V2;
        Real T1 = UV / T, T2 = VV / T - UV * UV / (T * T * T), dN = V0 - mu * T1;
        p1 += Dm * NmT * dN; p2 += Dm * (dN * dN - NmT * mu * T2);
      }
    }
  }
  *dphi = g1 + alpha * g2 + warp_sum(p1);
  *ddphi = g2 + warp_sum(p2);
}

template <typename Real> struct SolverOpts { int max_iter; int max_ls; Real tol; Real ls_tol; Real rtol; Real tol_improve; };

// one Newton iteration; returns 0 = took a step, 1 = converged before stepping, 2 = took a (negligible) last step
template <typename Real, typename D>
UR3E_HD int newton_iteration(const DevModel<Real>& m, Arena<Real, D>& s, const SolverOpts<Real>& opt, const Real scale) {
  const int nv = nv_<D>(m), nefc = s.nefc;
    constraint_update(m, s, true);
    Real gg = 0, gref = 0;
    WARP_FOR(d, nv) {
      Real g = s.Ma[d] - s.qfrc_smooth[d];
      const Real fc = col_dot(m, s, d, s.efc_force);
      g -= fc;
      s.qfrc_constraint[d] = fc;   // if this pass finds the point converged, these are the final constraint forces
      s.grad[d] = g; gg += g * g; gref += s.Ma[d] * s.Ma[d] + s.qfrc_smooth[d] * s.qfrc_smooth[d] + fc * fc;
    }
    gg = warp_sum(gg); gref = warp_sum(gref);
    // converged: MuJoCo's scaled-gradient test, or the gradient is at the rounding floor of its own terms
    if (scale * Num<Real>::sqrt(gg) < opt.tol || gg < opt.rtol * opt.rtol * gref) return 1;
    // H = M + J^T diag(Dact) J + cone blocks ; augmented row = -grad.
    // phase A: M and the rhs row (plain copies), then the rows with one or two entries: friction loss / limits / the joint
    // equality's squares on the diagonal (lane = dof) and the joint equality's single off-diagonal entry (lane = equality)
    {
      const int ntri = nv * (nv + 1) / 2;
#if defined(__CUDA_ARCH__)
      if constexpr (sizeof(Real) == 4 && D::EXACT && (D::NV * (D::NV + 1) / 2) % 2 == 0) {
        // exact-fit float classes: M -> H as 64-bit copies (both arrays are 8-byte aligned: see the static_asserts below Arena), then the rhs row
        const float2* src = reinterpret_cast<const float2*>(s.M); float2* dst = reinterpret_cast<float2*>(s.fr.n.H);
        WARP_FOR(e, ntri / 2 + nv) { if (e < ntri / 2) dst[e] = src[e]; else s.fr.n.H[ntri + e - ntri / 2] = -s.grad[e - ntri / 2]; }
      } else
#endif
      { WARP_FOR(e, ntri + nv) s.fr.n.H[e] = e < ntri ? s.M[e] : -s.grad[e - ntri]; }
      WARP_SYNC();
      WARP_FOR(i, nv + neq_<D>(m)) {
        if (i < nv) {
          Real h = 0;
          int r = s.sp_fl[i]; if (r != 255) h += s.efc_Dact[r];
          r = s.sp_lo[i]; if (r != 255) h += s.efc_Dact[r];
          r = s.sp_hi[i]; if (r != 255) h += s.efc_Dact[r];
          r = s.sp_ej[i]; if (r != 255) { const Real c = eqj_coef(m, s, i, r); h += s.efc_Dact[r] * c * c; }
          s.fr.n.H[i * (i + 1) / 2 + i] += h;
        } else {
          const int e = i - nv;
          if (m.eq_kind[e] != EK_CONNECT && m.eq_o2[e] >= 0) {
            const int d1 = m.eq_o1[e], d2 = m.eq_o2[e], r = s.sp_ej[d1], hi = d1 > d2 ? d1 : d2, lo = d1 > d2 ? d2 : d1;
            if (r != 255 && r == s.sp_ej[d2] && s.efc_id[r] == e) s.fr.n.H[hi * (hi + 1) / 2 + lo] -= s.efc_Dact[r] * s.eqj_deriv[e];
          }
        }
      }
      WARP_SYNC();
    }
    // phase B: one pass per row group over the lower triangle of its own column set
    for (int g = 0; g < s.ngrp; ++g) {
      const int r0 = s.grp_row0[g], r1 = r0 + s.grp_nrow[g], mask = s.grp_mask[g], kc = popcount32(mask);
      const bool contact = s.efc_type[r0] >= ROW_CON_N;
      // column list of the group: cols[k] = index of the k-th set bit of its dof mask (solver scratch; __fns is a slow software loop)
      uint8_t* cols = reinterpret_cast<uint8_t*>(s.colbuf[0]);
      WARP_FOR(d, 32) if ((mask >> d) & 1) cols[popcount32(mask & (int)((1u << d) - 1u))] = (uint8_t)d;
      WARP_SYNC();
      WARP_FOR(e, kc * (kc + 1) / 2) {
        int pq = m.tri_ab[e], a = cols[pq >> 8], b = cols[pq & 255];
        Real h = 0;
        if (!contact) {   // a connect equality: exactly three rows
          h = s.efc_Dact[r0] * s.u.efc_J[r0][a] * s.u.efc_J[r0][b] + s.efc_Dact[r0 + 1] * s.u.efc_J[r0 + 1][a] * s.u.efc_J[r0 + 1][b] +
              s.efc_Dact[r0 + 2] * s.u.efc_J[r0 + 2][a] * s.u.efc_J[r0 + 2][b];
        }
        else {
          for (int r = r0; r + 2 < r1 + 0 && r + 2 < D::MAXDENSE; r += 3) {
            Real a0 = s.u.efc_J[r][a], a1 = s.u.efc_J[r + 1][a], a2 = s.u.efc_J[r + 2][a];
            Real b0 = s.u.efc_J[r][b], b1 = s.u.efc_J[r + 1][b], b2 = s.u.efc_J[r + 2][b];
            const Real* Hc = s.cu.frame[s.efc_id[r]] + 3;
            if (Hc[0] > 0) h += Hc[0] * a0 * b0 + Hc[1] * (a0 * b1 + a1 * b0) + Hc[2] * (a0 * b2 + a2 * b0) + Hc[3] * a1 * b1 + Hc[4] * (a1 * b2 + a2 * b1) + Hc[5] * a2 * b2;
            else h += s.efc_Dact[r] * a0 * b0 + s.efc_Dact[r + 1] * a1 * b1 + s.efc_Dact[r + 2] * a2 * b2;
          }
        }
        s.fr.n.H[a * (a + 1) / 2 + b] += h;
      }
      WARP_SYNC();
    }
#if defined(__CUDA_ARCH__) && UR3E_REG_CHOL
    chol_solve_reg_body<Real, D::NV, D::SPLIT>(s.fr.n.H, s.fr.n.H + nv * (nv + 1) / 2, nv, s.search, s.coupled != 0 || split_<D>(m) != D::SPLIT);   // inlined in the Newton loop; the Euler step and the unconstrained case share the out-of-line copy
#else
    chol_solve_aug(s, nv, s.search);
#endif
    // Mv, jv, and the quadratic (Gauss) part of the line cost
    WARP_FOR(i, nv + nefc) {
      if (i < nv) s.Mv[i] = sym_matvec_row_n<Real, D::NV>(s.M, s.search, i, nv);
      else { int r = i - nv; s.efc_jv[r] = row_dot(m, s, r, s.search); }
    }
    WARP_SYNC();
    Real g1 = 0, g2 = 0, sn = 0, pred = 0;
    WARP_FOR(d, nv) { g1 += s.search[d] * (s.Ma[d] - s.qfrc_smooth[d]); g2 += s.search[d] * s.Mv[d]; sn += s.search[d] * s.search[d]; pred -= s.search[d] * s.grad[d]; }
    g1 = warp_sum(g1); g2 = warp_sum(g2); sn = warp_sum(sn); pred = Real(0.5) * warp_sum(pred);   // pred = Newton's model decrease of the cost
    // exact line search: safeguarded Newton on phi'(alpha)
    // At alpha = 0 nothing has to be evaluated: H is the exact Hessian of the (piecewise quadratic) cost at qacc and H search = -grad,
    // so phi'(0) = grad . search = -2 pred and phi''(0) = search . H search = 2 pred; the first trial point is the full Newton step.
    Real p1, p2, lo = 0, hi = -1, alpha = 1;
    if (!(pred > 0)) return 1;
    const Real p10 = 2 * pred;
    for (int ls = 0; ls < opt.max_ls; ++ls) {
      line_eval(m, s, alpha, g1, g2, &p1, &p2);
      if (Num<Real>::abs(p1) < opt.ls_tol * p10) break;
      if (p1 < 0) lo = alpha; else hi = alpha;
      Real na = alpha - p1 / p2;
      if (hi < 0) { if (!(na > lo)) na = 2 * alpha; }
      else if (!(na > lo && na < hi)) na = Real(0.5) * (lo + hi);
      if (na == alpha) break;
      alpha = na;
    }
    WARP_FOR(i, nv + nefc) {
      if (i < nv) { s.qacc[i] += alpha * s.search[i]; s.Ma[i] += alpha * s.Mv[i]; }
      else s.efc_jar[i - nv] += alpha * s.efc_jv[i - nv];
    }
    WARP_SYNC();
    if (scale * alpha * Num<Real>::sqrt(sn) * m.meaninertia < opt.tol * Real(1e-3)) return 2;
    // MuJoCo's `improvement < tolerance` test (scaled cost decrease of this iteration); disabled (0) in the validation build
    if (scale * pred < opt.tol_improve) return 2;
    return 0;
}

template <typename Real, typename D>
UR3E_HD void solve(const DevModel<Real>& m, Arena<Real, D>& s, const SolverOpts<Real>& opt) {
  const int nv = nv_<D>(m), nefc = s.nefc;
  if (nefc == 0) {
    // unconstrained: qacc = M^-1 qfrc_smooth
    WARP_FOR(e, nv * (nv + 1) / 2 + nv) { s.fr.n.H[e] = e < nv * (nv + 1) / 2 ? s.M[e] : s.qfrc_smooth[e - nv * (nv + 1) / 2]; }
    WARP_FOR(d, nv) s.qfrc_constraint[d] = 0;
    WARP_SYNC();
#if defined(__CUDA_ARCH__) && UR3E_REG_CHOL
    chol_solve_reg<Real, D::NV, D::SPLIT>(s.fr.n.H, s.fr.n.H + nv * (nv + 1) / 2, nv, s.qacc, split_<D>(m) != D::SPLIT);   // H = M here
#else
    chol_solve_aug(s, nv, s.qacc);
#endif
    IF_LANE0 s.solver_iter = 0;
    return;
  }
  const Real scale = Real(1) / (m.meaninertia * Real(nv > 1 ? nv : 1));
  WARP_FOR(d, nv) s.qacc[d] = s.st.qacc_ws[d];
  WARP_SYNC();
  WARP_FOR(i, nv + nefc) {
    if (i < nv) s.Ma[i] = sym_matvec_row_n<Real, D::NV>(s.M, s.qacc, i, nv);
    else { int r = i - nv; s.efc_jar[r] = row_dot(m, s, r, s.qacc) - s.efc_aref[r]; }
  }
  WARP_SYNC();
  // Newton iterations; each warp runs its own count (the block re-aligns at the barrier that follows the solve: lock-stepping
  // the iterations themselves measured 1.5 % slower once the iteration became cheap, profiles/r1_summary.md)
  int iter = 0, rc = 0;
  for (int it = 0; it < opt.max_iter; ++it) {
    rc = newton_iteration(m, s, opt, scale);
    if (rc != 1) ++iter;
    if (rc != 0) break;
  }
  if (rc != 1) {
    // the last pass moved qacc (negligible step, or the iteration cap): forces at the final point.  After a pass that found the point
    // converged (rc == 1, the normal exit) efc_force and qfrc_constraint are already those of the final point.
    constraint_update(m, s, false);
    WARP_FOR(d, nv) s.qfrc_constraint[d] = col_dot(m, s, d, s.efc_force);
  }
  IF_LANE0 s.solver_iter = iter;
  WARP_SYNC();
}

// ---------------------------------------------------------------- torque site sensors (reference assets/main.xml:384-391)
// mj_rnePostConstraint + mjSENS_TORQUE restated: body accelerations from the solver's qacc, inertial wrench of every body minus the
// external wrenches on it (contacts, connect equalities), summed over the subtree = the wrench the parent transmits to the link;
// its torque, moved to the site and expressed in the site frame, is the sensor value.  Cold path (only with a sensor buffer): the
// body frames and velocities are rebuilt here, in storage that is dead after the solve (the Jacobian's).
template <typename Real, typename D>
UR3E_PHASE void torque_sensors_cold(const DevModel<Real>& m, Arena<Real, D>& s, Real* out) {
  const int nb = nb_<D>(m), nv = nv_<D>(m);
  auto& y = s.u.dyn;
  // contact forces in world axes, taken before the frames' storage is rebuilt (tangents are recomputed from the normal: the solver keeps
  // the cone Hessians in their place); kept in the dead colbuf-free efc_jv / efc_Dact rows: [3c..3c+3) = world force of contact c
  if constexpr (D::HAS_CONTACT) {
    WARP_FOR(c, s.ncon) {
      Real f[9]; for (int k = 0; k < 3; ++k) f[k] = s.cu.frame[c][k];
      make_frame(f);
      const int r = s.con_row[c];
      const Real f0 = s.efc_force[r], f1 = s.efc_force[r + 1], f2 = s.efc_force[r + 2];
      for (int k = 0; k < 3; ++k) s.efc_jv[3 * c + k] = f[k] * f0 + f[3 + k] * f1 + f[6 + k] * f2;
    }
  }
  WARP_SYNC();
  kinematics(m, s);            // body frames, inertial frame positions, cdof (unchanged), site frames
  // body inertias + velocities about the tree reference point, cdof_dot (as in dynamics())
  WARP_FOR(b, nb) {
    Real* ci = y.cinert[b];
    if (b == 0 || m.body_lastdof[b] < 0) { for (int k = 0; k < 10; ++k) ci[k] = 0; for (int k = 0; k < 6; ++k) y.cvel[b][k] = 0; }
    else {
      const Real* ref = s.xpos[m.body_root[b]];
      Real dif[3] = {s.fr.k.xipos[b][0] - ref[0], s.fr.k.xipos[b][1] - ref[1], s.fr.k.xipos[b][2] - ref[2]};
      Real R[9]; mat_mul3(R, s.fr.k.xmat[b], m.body_imat[b]);
      const Real* in = m.body_inertia[b]; Real mass = m.body_mass[b];
      Real t00 = 0, t11 = 0, t22 = 0, t01 = 0, t02 = 0, t12 = 0;
      for (int k = 0; k < 3; ++k) {
        t00 += R[k] * in[k] * R[k]; t11 += R[3 + k] * in[k] * R[3 + k]; t22 += R[6 + k] * in[k] * R[6 + k];
        t01 += R[k] * in[k] * R[3 + k]; t02 += R[k] * in[k] * R[6 + k]; t12 += R[3 + k] * in[k] * R[6 + k];
      }
      ci[0] = t00 + mass * (dif[1] * dif[1] + dif[2] * dif[2]); ci[1] = t11 + mass * (dif[0] * dif[0] + dif[2] * dif[2]);
      ci[2] = t22 + mass * (dif[0] * dif[0] + dif[1] * dif[1]);
      ci[3] = t01 - mass * dif[0] * dif[1]; ci[4] = t02 - mass * dif[0] * dif[2]; ci[5] = t12 - mass * dif[1] * dif[2];
      ci[6] = mass * dif[0]; ci[7] = mass * dif[1]; ci[8] = mass * dif[2]; ci[9] = mass;
      Real cv[6] = {0, 0, 0, 0, 0, 0};
      for (int d = m.body_lastdof[b]; d >= 0; d = m.dof_parent[d]) { Real qd = s.st.qvel[d]; for (int k = 0; k < 6; ++k) cv[k] += s.cdof[d][k] * qd; }
      for (int k = 0; k < 6; ++k) y.cvel[b][k] = cv[k];
    }
  }
  WARP_SYNC();
  WARP_FOR(d, nv) {
    int b = m.dof_body[d], fk = m.dof_free_k[d];
    Real* cd = y.cdof_dot[d];
    if (fk >= 0 && fk < 3) { for (int k = 0; k < 6; ++k) cd[k] = 0; }
    else {
      Real vel[6];
      for (int k = 0; k < 6; ++k) vel[k] = y.cvel[m.body_parent[b]][k];
      if (fk >= 3) { int da = m.body_dadr[b]; for (int i = 0; i < 3; ++i) for (int k = 0; k < 6; ++k) vel[k] += s.cdof[da + i][k] * s.st.qvel[da + i]; }
      cross_motion(cd, vel, s.cdof[d]);
    }
  }
  WARP_SYNC();
  // inertial wrench of every body at the solver's acceleration: I a + v x* I v, a = -g + sum over the chain of cdof_dot qvel + cdof qacc
  WARP_FOR(b, nb) {
    Real* f = y.cfrc[b];
    if (b == 0 || m.body_lastdof[b] < 0) { for (int k = 0; k < 6; ++k) f[k] = 0; }
    else {
      Real a[6] = {0, 0, 0, -m.gravity[0], -m.gravity[1], -m.gravity[2]};
      for (int d = m.body_lastdof[b]; d >= 0; d = m.dof_parent[d]) { const Real qd = s.st.qvel[d], qa = s.qacc[d]; for (int k = 0; k < 6; ++k) a[k] += y.cdof_dot[d][k] * qd + s.cdof[d][k] * qa; }
      Real t1[6], t2[6];
      mul_inert(f, y.cinert[b], a);
      mul_inert(t1, y.cinert[b], y.cvel[b]); cross_force(t2, y.cvel[b], t1);
      for (int k = 0; k < 6; ++k) f[k] += t2[k];
    }
  }
  WARP_SYNC();
  // minus the external wrenches: contacts push geom2's body along the contact force and geom1's body against it; a connect equality
  // pulls its first body with +f at the first anchor and its second with -f at the second (world axes)
  auto apply = [&](int b, const Real* p, const Real* F, Real sign) {   // cfrc[b] -= sign * wrench of force F at point p
    if (b <= 0 || m.body_lastdof[b] < 0) return;
    const Real* ref = s.xpos[m.body_root[b]];
    const Real r[3] = {p[0] - ref[0], p[1] - ref[1], p[2] - ref[2]}; Real t[3]; cross3(t, r, F);
    IF_LANE0 { for (int k = 0; k < 3; ++k) { y.cfrc[b][k] -= sign * t[k]; y.cfrc[b][3 + k] -= sign * F[k]; } }
  };
  if constexpr (D::HAS_CONTACT) {
    for (int c = 0; c < s.ncon; ++c) {
      const int p = s.con_pair[c];
      const Real F[3] = {s.efc_jv[3 * c], s.efc_jv[3 * c + 1], s.efc_jv[3 * c + 2]};
      apply(m.geom_body[m.pair_g2[p]], s.con_pos[c], F, Real(1)); apply(m.geom_body[m.pair_g1[p]], s.con_pos[c], F, Real(-1));
      WARP_SYNC();
    }
  }
  {
    int row = 0;
    for (int e = 0; e < neq_<D>(m); ++e) if (m.eq_kind[e] == EK_CONNECT) {
      const int b1 = m.eq_o1[e], b2 = m.eq_o2[e];
      Real a1[3], a2[3], v[3];
      mat_vec3(v, s.fr.k.xmat[b1], m.eq_data[e]); for (int k = 0; k < 3; ++k) a1[k] = s.xpos[b1][k] + v[k];
      mat_vec3(v, s.fr.k.xmat[b2], m.eq_data[e] + 3); for (int k = 0; k < 3; ++k) a2[k] = s.xpos[b2][k] + v[k];
      const Real F[3] = {s.efc_force[row], s.efc_force[row + 1], s.efc_force[row + 2]};
      apply(b1, a1, F, Real(1)); apply(b2, a2, F, Real(-1));
      WARP_SYNC();
      row += 3;
    }
  }
  // subtree sums (lane = component, serial down the parent < child order)
  WARP_FOR(k, 6) { for (int b = nb - 1; b > 0; --b) { const int p = m.body_parent[b]; if (p > 0) y.cfrc[p][k] += y.cfrc[b][k]; } }
  WARP_SYNC();
  WARP_FOR(j, MAXTQ) {
    Real* o = out + 28 + 3 * j;
    if (j >= m.ntq) { o[0] = o[1] = o[2] = 0; }
    else {
      const int b = m.tq_body[j];
      const Real* ref = s.xpos[m.body_root[b]]; const Real* f = y.cfrc[b];
      Real sp[3], R[9], t[3];
      mat_vec3(sp, s.fr.k.xmat[b], m.tq_pos[j]); mat_mul3(R, s.fr.k.xmat[b], m.tq_mat[j]);
      const Real r[3] = {s.xpos[b][0] + sp[0] - ref[0], s.xpos[b][1] + sp[1] - ref[1], s.xpos[b][2] + sp[2] - ref[2]};
      cross3(t, r, f + 3);
      const Real tau[3] = {f[0] - t[0], f[1] - t[1], f[2] - t[2]};
      for (int i = 0; i < 3; ++i) o[i] = R[i] * tau[0] + R[3 + i] * tau[1] + R[6 + i] * tau[2];   // R^T tau
    }
  }
  WARP_SYNC();
}

// ---------------------------------------------------------------- logging sensors (reference assets/main.xml:392-408)
// out[0..7) = actuatorfrc of the (up to seven) actuators, out[9..21) = tcp site position and orientation matrix,
// out[7] / out[8] = touch sensors on the tracked sites 2 / 3
// (right_pad1_site, left_pad1_site; readers utils/utils.py:201-245, controller_func.py:191-211).  Runs right after the solve
// of a substep, i.e. on the same pre-integration state MuJoCo evaluates its sensors on.  Cold path: only when the caller gave
// the batch a sensor buffer.  Body frames are recomputed (their storage holds the Newton matrix by now; J is dead); the
// contact normals are still in place (the cone Hessians only reuse the tangents' storage).
template <typename Real, typename D>
UR3E_PHASE void sensors_cold(const DevModel<Real>& m, Arena<Real, D>& s, Real* out) {
  WARP_FOR(a, 7) { out[a] = a < nu_<D>(m) ? s.act_force[a] : Real(0); out[21 + a] = a < nu_<D>(m) ? s.ctrl[a] : Real(0); }   // [21..28): d.ctrl as the controller set it (unclamped)
  WARP_FOR(i, 12) out[9 + i] = nsite_<D>(m) > 0 ? (i < 3 ? s.site_xpos[0][i] : s.site_xmat[0][i - 3]) : Real(0);   // the tcp is the first tracked site
  Real touch[2] = {0, 0};
  if constexpr (D::HAS_CONTACT) {
    if (nsite_<D>(m) >= 4) {
      kin_frames(m, s);
      WARP_FOR(c, s.ncon) {
        const int p = s.con_pair[c], b1 = m.geom_body[m.pair_g1[p]], b2 = m.geom_body[m.pair_g2[p]];
        const Real fn = s.efc_force[s.con_row[c]];
        for (int k = 0; k < 2; ++k) {
          const int j = 2 + k, sb = m.site_body[j];
          if (fn > 0 && (b1 == sb || b2 == sb)) {
            Real R[9], dlt[3], loc[3];
            mat_mul3(R, s.fr.k.xmat[sb], m.site_mat[j]);
            for (int i = 0; i < 3; ++i) dlt[i] = s.con_pos[c][i] - s.site_xpos[j][i];
            for (int i = 0; i < 3; ++i) loc[i] = R[i] * dlt[0] + R[3 + i] * dlt[1] + R[6 + i] * dlt[2];   // R^T dlt
            const Real* nrm = s.cu.frame[c];   // contact normal (world)
            Real dir[3];
            for (int i = 0; i < 3; ++i) dir[i] = R[i] * nrm[0] + R[3 + i] * nrm[1] + R[6 + i] * nrm[2];
            const Real* sz = m.site_size[j];
            // MuJoCo's touch rule: the line through the contact point along the contact normal has to cross the site's box (slab test)
            Real lo = -Num<Real>::big, hi = Num<Real>::big;
            bool in = true;
            for (int i = 0; i < 3; ++i) {
              if (Num<Real>::abs(dir[i]) < Real(1e-12)) { if (Num<Real>::abs(loc[i]) > sz[i]) in = false; }
              else {
                const Real t1 = (-sz[i] - loc[i]) / dir[i], t2 = (sz[i] - loc[i]) / dir[i];
                lo = rmax(lo, rmin(t1, t2)); hi = rmin(hi, rmax(t1, t2));
              }
            }
            if (lo > hi) in = false;
            if (in) touch[k] += fn;
          }
        }
      }
    }
  }
  const Real t0 = warp_sum(touch[0]), t1 = warp_sum(touch[1]);
  IF_LANE0 { out[7] = t0; out[8] = t1; }
  WARP_SYNC();
  torque_sensors_cold(m, s, out);
}

// ---------------------------------------------------------------- one mj_step (SURVEY 3.4)
template <typename Real, typename D>
UR3E_HD void forward(const DevModel<Real>& m, Arena<Real, D>& s, const SolverOpts<Real>& opt, bool with_solver, bool aligned = false) {
  // `aligned`: every warp of the block is on this path (the regular substep), so block-wide barriers keep the warps in the
  // same phase and they share its code in the SM's instruction cache; all other callers (reset, set_state, redo after a
  // bad qacc) are warp-divergent and must not touch the barrier.
#ifndef UR3E_BARRIERS
#define UR3E_BARRIERS 16   // bit i: block barrier after phase i of the substep (kinematics, dynamics, collision, rows, solve).  One, after the only
                           // variable-length phase, is enough and measures 1 % faster than all five; a barrier before the solve instead: -20 %
#endif
  kinematics(m, s);
  if (aligned && (UR3E_BARRIERS & 1)) BLOCK_SYNC();
  dynamics(m, s);
  if (aligned && (UR3E_BARRIERS & 2)) BLOCK_SYNC();
  collision(m, s);
  if (with_solver) {
    if (aligned && (UR3E_BARRIERS & 4)) BLOCK_SYNC();
    make_constraint(m, s);
    if (aligned && (UR3E_BARRIERS & 8)) BLOCK_SYNC();
    solve(m, s, opt);
  }
}

// out-of-line copy of the full forward pass for the rare paths (redo after a bad qacc, reset): keeps them out of the step's hot code
template <typename Real, typename D>
UR3E_PHASE void forward_cold(const DevModel<Real>& m, Arena<Real, D>& s, const SolverOpts<Real>& opt, bool with_solver) { forward(m, s, opt, with_solver); }

template <typename Real, typename D>
UR3E_PHASE void reset_data(const DevModel<Real>& m, Arena<Real, D>& s) {
  WARP_FOR(i, nq_<D>(m)) s.st.qpos[i] = m.qpos0[i];
  WARP_FOR(i, nv_<D>(m)) { s.st.qvel[i] = 0; s.st.qacc_ws[i] = 0; s.qacc[i] = 0; }
  WARP_FOR(i, nu_<D>(m)) s.ctrl[i] = 0;
  WARP_SYNC();
}

template <typename Real> UR3E_HD int is_bad(Real x) { return !(Num<Real>::abs(x) <= Real(1e10)); }   // NaN or |x| > 1e10 (mj_checkPos/Vel/Acc)

// ---------------------------------------------------------------- tree-sparse solve for the Euler step
// (M + h diag(damping)) x = b.  M has the sparsity of the dof tree, so the reverse-order L^T D L factorisation has no
// fill-in (the scheme MuJoCo uses for mj_factorM): processing dof k only touches the entries between its ancestors.
// A = packed lower triangle (i(i+1)/2 + j) held in the Newton matrix storage; x in shared memory.
template <typename Real, typename D>
UR3E_PHASE void tree_ldl_solve(const DevModel<Real>& m, Arena<Real, D>& s, Real* x) {
  const int nv = nv_<D>(m);
  Real* A = s.fr.n.H;
#pragma unroll 1
  for (int k = nv - 1; k > 0; --k) {
    const int na = m.dof_nanc[k];
    if (na == 0) continue;
    const Real* rk = A + k * (k + 1) / 2;
    const Real inv = Real(1) / rk[k];
    WARP_FOR(e, na * (na + 1) / 2) {
      const int pq = m.tri_ab[e], i = m.dof_anc[k][pq & 255], j = m.dof_anc[k][pq >> 8];   // j <= i, both ancestors of k
      A[i * (i + 1) / 2 + j] -= rk[i] * rk[j] * inv;
    }
    WARP_SYNC();
  }
  WARP_FOR(k, nv) s.dinv[k] = Real(1) / A[k * (k + 1) / 2 + k];
  WARP_SYNC();
  // x <- L^-T x  (unit L, L[k][i] = A[k][i] / A[k][k])
#pragma unroll 1
  for (int k = nv - 1; k > 0; --k) {
    const int na = m.dof_nanc[k];
    if (na == 0) continue;
    const Real* rk = A + k * (k + 1) / 2;
    const Real xk = x[k] * s.dinv[k];
    WARP_FOR(t, na) { const int i = m.dof_anc[k][t]; x[i] -= rk[i] * xk; }
    WARP_SYNC();
  }
  WARP_FOR(k, nv) x[k] *= s.dinv[k];
  WARP_SYNC();
  // x <- L^-1 x, level by level down the dof tree
#pragma unroll 1
  for (int dep = 1; dep <= m.max_nanc; ++dep) {
    WARP_FOR(k, nv) {
      if (m.dof_nanc[k] == dep) {
        const Real* rk = A + k * (k + 1) / 2;
        Real v = 0;
        for (int t = 0; t < dep; ++t) { const int i = m.dof_anc[k][t]; v += rk[i] * x[i]; }
        x[k] -= v * s.dinv[k];
      }
    }
    WARP_SYNC();
  }
}

template <typename Real, typename D>
UR3E_HD void euler(const DevModel<Real>& m, Arena<Real, D>& s) {
  const int nv = nv_<D>(m); const Real h = m.timestep;
  Real* qa = s.qacc;
  if (has_damping_<D>(m)) {
    // (M + h diag(damping)) a = qfrc_smooth + qfrc_constraint   (SURVEY B.8)
#if defined(__CUDA_ARCH__) && UR3E_REG_CHOL
    // M is dead after this step (the next substep rebuilds it), so the damping goes onto its diagonal in place
    WARP_FOR(d, nv) { s.M[d * (d + 1) / 2 + d] += h * m.dof_damping[d]; s.search[d] = s.qfrc_smooth[d] + s.qfrc_constraint[d]; }
    WARP_SYNC();
    chol_solve_reg<Real, D::NV, D::SPLIT>(s.M, s.search, nv, s.search, split_<D>(m) != D::SPLIT);   // M + h B never couples two trees
#else
    Real* A = s.fr.n.H;
    WARP_FOR(e, nv * (nv + 1) / 2) { const int ab = m.tri_ab[e]; A[e] = s.M[e] + ((ab >> 8) == (ab & 255) ? h * m.dof_damping[ab >> 8] : Real(0)); }
    WARP_FOR(d, nv) s.search[d] = s.qfrc_smooth[d] + s.qfrc_constraint[d];
    WARP_SYNC();
    tree_ldl_solve(m, s, s.search);
#endif
    qa = s.search;
  }
  WARP_FOR(d, nv) s.st.qvel[d] += h * qa[d];
  WARP_SYNC();
  WARP_FOR(d, nv) {
    int fk = m.dof_free_k[d], q = m.dof_qadr[d];
    if (fk < 0 || fk < 3) s.st.qpos[q] += h * s.st.qvel[d];
    else if (fk == 3) {
      Real w[3] = {s.st.qvel[d], s.st.qvel[d + 1], s.st.qvel[d + 2]};
      Real n = Num<Real>::sqrt(dot3(w, w)), ang = h * n;
      Real qr[4] = {1, 0, 0, 0};
      if (n >= Num<Real>::minval && ang != 0) { Real sn, cs; Num<Real>::sincos(ang * Real(0.5), &sn, &cs); sn /= n; qr[0] = cs; qr[1] = w[0] * sn; qr[2] = w[1] * sn; qr[3] = w[2] * sn; }
      Real qq[4] = {s.st.qpos[q], s.st.qpos[q + 1], s.st.qpos[q + 2], s.st.qpos[q + 3]}, out[4];
      quat_normalize(qq); quat_mul(out, qq, qr);
      for (int k = 0; k < 4; ++k) s.st.qpos[q + k] = out[k];
    }
  }
  WARP_SYNC();
}

// returns a warning mask: 1 bad qpos, 2 bad qvel, 4 bad qacc (mj_checkPos/Vel/Acc + autoreset, SURVEY B.10)
// opt_cold: the same options in addressable (device) memory, for the out-of-line redo path
template <typename Real, typename D>
UR3E_HD int substep(const DevModel<Real>& m, Arena<Real, D>& s, const SolverOpts<Real>& opt, const SolverOpts<Real>& opt_cold, Real* sens_base = nullptr, long long env = 0) {
  int w = 0;
  WARP_FOR(i, nq_<D>(m) + nv_<D>(m)) w |= i < nq_<D>(m) ? is_bad(s.st.qpos[i]) : 2 * is_bad(s.st.qvel[i - nq_<D>(m)]);
  w = warp_or(w);
  if (w) reset_data(m, s);
  forward(m, s, opt, true, true);
  int wa = 0;
  WARP_FOR(i, nv_<D>(m)) wa |= 4 * is_bad(s.qacc[i]);
  wa = warp_or(wa);
  if (wa) { reset_data(m, s); forward_cold(m, s, opt_cold, true); w |= wa; }
  WARP_FOR(d, nv_<D>(m)) s.st.qacc_ws[d] = s.qacc[d];
  if (sens_base) sensors_cold(m, s, sens_base + env * NSENSOR);
  if (UR3E_BARRIERS & 16) BLOCK_SYNC(); else WARP_SYNC();
  euler(m, s);
  return w;
}

}  // namespace ur3e
