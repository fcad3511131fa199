// The sm_100a kernels that run the fused environment step + the typed batch object behind the C ABI.
// One warp per environment, WPB warps per block, one shared-memory Arena per warp (engine.cuh / env.cuh).
#pragma once
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <type_traits>
#include <vector>

#include "batch_base.h"
#include "compile_model.h"
#include "merge_bodies.h"
#include "distance.cuh"
#include "env.cuh"
#include "ik.cuh"
#include "query.cuh"
#include "query_fwd.cuh"
#include "query_inv.cuh"
#include "render.cuh"
#include "rollout.h"

#ifndef UR3E_BLOCKS_PER_SM
#define UR3E_BLOCKS_PER_SM 2
#endif
#ifndef UR3E_LS_TOL
#define UR3E_LS_TOL 1e-2   // float32 line-search tolerance on |phi'(alpha)| / |phi'(0)|: MuJoCo's default ls_tolerance (1e-5 measured 2-4 % slower, same iteration counts)
#endif
#ifndef UR3E_MAX_WPB
#define UR3E_MAX_WPB 16
#endif

namespace ur3e {
enum Op { OP_STEP = 0, OP_RESET = 1, OP_SET_STATE = 2 };

template <typename Real>
struct KArgs {
  const DevModel<Real>* m;
  EnvCfg<Real> c;
  SolverOpts<Real> opt;
  // device-memory copies of c / opt for the out-of-line cold paths (reset, redo): passing &a.c to a function would force the
  // whole parameter block into local memory and turn every c.* / opt.* read of the hot path into a local load
  const EnvCfg<Real>* c_dev; const SolverOpts<Real>* opt_dev;
  void* st;   // EnvState<Real, D>[n]; the lite and full size classes of a model share the record layout
  // two-tier stepping (see Batch::step): overflow hand-off from the lite kernel to the full kernel
  int* ovf_count; int* ovf_list;         // lite tier: environments it hands to the full tier (lite caps exceeded, or EnvState::tier > 0); not stored
  const int* list_count; const int* list;  // full tier: process exactly these environments
  int lite_maxcon, lite_maxefc;          // grasp / generic tier of a tiered batch: the lite caps, to maintain EnvState::tier
  int mid_maxcon, mid_maxefc;            // ... and the grasp tier's caps (0 = the batch has no grasp tier)
  int* ovf2_count; int* ovf2_list;       // lite tier: environments whose record says they need the generic class go straight to this list
  int* ovf_stat;                         // full tier: counts the environments whose step did not fit the lite caps (information only)
  int cap_con, cap_efc;                  // row / contact caps of this launch (0 = the size class's own)
  long long n;
  int op;
  const Real* act; Real* obs; Real* rew; uint8_t* term; uint8_t* trunc; Real* final_obs;
  Real* sens;   // optional [n, NSENSOR] logging-sensor output of every step (null = off, the normal case)
  const uint8_t* mask;
  unsigned long long seed, env_base;
  const Real* qpos_in; const Real* qvel_in; const Real* ws_in;
};

template <typename Real, typename D> __host__ __device__ constexpr size_t arena_stride() { return (sizeof(Arena<Real, D>) + 15) / 16 * 16; }
// warps (environments) per block: as many as fit one SM's shared memory (<= 16); the block's warps advance through the
// substep phases together (block barriers in forward()), so one block per SM shares each phase's code in the I-cache.
template <typename Real, typename D> __host__ __device__ constexpr int warps_per_block() {
  // UR3E_BLOCKS_PER_SM co-resident blocks: while one block waits at a barrier the other keeps the issue slots busy
#ifdef UR3E_FORCE_WPB
  return UR3E_FORCE_WPB;   // compile-only experiments (register budget at a given block size)
#endif
  int per_sm = (int)((233472 - 1024 * UR3E_BLOCKS_PER_SM) / arena_stride<Real, D>());
  int w = per_sm / UR3E_BLOCKS_PER_SM;
#ifdef UR3E_MID_MAX_WPB
  if (D::EXACT && D::MAXCON == 16 && w > UR3E_MID_MAX_WPB) w = UR3E_MID_MAX_WPB;   // A/B: register budget of the grasp tier
#endif
  return w > UR3E_MAX_WPB ? UR3E_MAX_WPB : (w < 1 ? 1 : w);
}

template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, D>() * 32) env_kernel(const KArgs<Real> a) {
  constexpr int WPB = warps_per_block<Real, D>();
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long e = (long long)blockIdx.x * WPB + warp;
  if (e >= a.n) return;
  Arena<Real, D>& s = *reinterpret_cast<Arena<Real, D>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, D>());
  const DevModel<Real>& m = *a.m;
  const EnvCfg<Real>& c = a.c;
  constexpr int NW = sizeof(EnvState<Real, D>) / 16;
  int4* gst = reinterpret_cast<int4*>(static_cast<EnvState<Real, D>*>(a.st) + e);
  int4* sst = reinterpret_cast<int4*>(&s.st);
  if (a.op == OP_RESET && a.mask && !a.mask[e]) return;
  WARP_FOR(i, NW) sst[i] = gst[i];
  IF_LANE0 { s.overflow = 0; s.ncon = 0; s.nefc = 0; s.solver_iter = 0; s.cap_con = D::MAXCON; s.cap_efc = D::MAXEFC; }
  WARP_SYNC();
  const int od = c.obs_dim;
  IF_LANE0 s.st.tier = 0;   // a reset / injected state starts on the lite tier again
  if (a.op == OP_RESET) {
    env_reset(m, c, s, a.opt, a.seed, a.env_base + (unsigned long long)e);
    ContactFlags cf = contact_flags(m, c, s);
    write_obs(m, c, s, cf);
    if (a.obs) { WARP_FOR(i, od) a.obs[e * od + i] = s.obs[i]; }
  } else if (a.op == OP_SET_STATE) {
    WARP_FOR(i, m.nq) s.st.qpos[i] = a.qpos_in[e * m.nq + i];
    WARP_FOR(i, m.nv) { s.st.qvel[i] = a.qvel_in[e * m.nv + i]; s.st.qacc_ws[i] = a.ws_in ? a.ws_in[e * m.nv + i] : Real(0); }
    WARP_SYNC();
    forward_cold(m, s, a.opt, false);
    update_cache(m, c, s);
  }
  WARP_SYNC();
  WARP_FOR(i, NW) gst[i] = sst[i];
}

// The step path.  One warp per environment; the block's warps pass the substep phases together (one block barrier per substep).
// A warp without work exits: a barrier only waits for the block's non-exited threads, and a warp that has no environment in one
// pass of the list loop has none in any later pass either (neither has the rest of its block).
// SENS: the variant that also writes the logging sensors (a.sens); the normal one carries no trace of that call.
constexpr int TIER_HOLD = 8;   // steps an environment keeps going straight to the full size class after it last needed it
template <typename Real, typename D, bool SENS = false>
__global__ void __launch_bounds__(warps_per_block<Real, D>() * 32, UR3E_BLOCKS_PER_SM) step_kernel(const KArgs<Real> a) {
  constexpr int WPB = warps_per_block<Real, D>();
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  Arena<Real, D>& s = *reinterpret_cast<Arena<Real, D>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, D>());
  const DevModel<Real>& m = *a.m;
  const EnvCfg<Real>& c = a.c;
  constexpr int NW = sizeof(EnvState<Real, D>) / 16;
  const int od = c.obs_dim;
  long long count = a.n; int iters = 1;
  if (a.list) { count = *a.list_count; const long long per = (long long)gridDim.x * WPB; iters = (int)((count + per - 1) / per); }
  for (int it = 0; it < iters; ++it) {
    const long long idx = ((long long)it * gridDim.x + blockIdx.x) * WPB + warp;
    if (idx >= count) return;
    const long long e = a.list ? (long long)a.list[idx] : idx;
    EnvState<Real, D>* const rec = static_cast<EnvState<Real, D>*>(a.st) + e;
    if (a.ovf_list && !a.list) {
      // lite tier: an environment that recently needed a larger size class goes straight to it (no wasted lite step): to the grasp
      // tier's list, or to the generic class's when it recently exceeded the grasp tier's caps too
      const int tier = rec->tier;
      if (tier & 0xff) {
        IF_LANE0 {
          if ((tier >> 8) && a.ovf2_list) { const int k = atomicAdd(a.ovf2_count, 1); a.ovf2_list[k] = (int)e; }
          else { const int k = atomicAdd(a.ovf_count, 1); a.ovf_list[k] = (int)e; }
        }
        return;
      }
    }
    int4* gst = reinterpret_cast<int4*>(rec);
    int4* sst = reinterpret_cast<int4*>(&s.st);
    WARP_FOR(i, NW) sst[i] = gst[i];
    IF_LANE0 {
      s.overflow = 0; s.ncon = 0; s.nefc = 0; s.solver_iter = 0;
      s.cap_con = (a.cap_con > 0 && a.cap_con < D::MAXCON) ? a.cap_con : D::MAXCON; s.cap_efc = (a.cap_efc > 0 && a.cap_efc < D::MAXEFC) ? a.cap_efc : D::MAXEFC;
    }
    WARP_SYNC();
    StepOut<Real> r = env_step(m, c, s, a.opt, a.act + e * c.act_dim, *a.opt_dev, SENS ? a.sens : nullptr, e);
    if (a.ovf_list && s.overflow) {
      // lite / grasp tier: this environment needed more rows / contacts than this size class's arena holds; leave its stored
      // state untouched and hand it to the next tier's list
      IF_LANE0 { const int k = atomicAdd(a.ovf_count, 1); a.ovf_list[k] = (int)e; }
      continue;   // (no block barrier follows in this pass)
    }
    if (a.lite_maxcon > 0) {
      // grasp / full tier of a tiered batch: keep the environment off the lite tier while its steps do not fit the lite caps (+ TIER_HOLD steps)
      IF_LANE0 {
        const bool big = s.max_ncon > a.lite_maxcon || s.max_nefc > a.lite_maxefc;
        const bool big2 = a.mid_maxcon > 0 && (s.max_ncon > a.mid_maxcon || s.max_nefc > a.mid_maxefc);
        const int h1 = s.st.tier & 0xff, h2 = s.st.tier >> 8;
        s.st.tier = (big ? TIER_HOLD : (h1 > 0 ? h1 - 1 : 0)) | ((big2 ? TIER_HOLD : (h2 > 0 ? h2 - 1 : 0)) << 8);
        if (big && a.ovf_stat) atomicAdd(a.ovf_stat, 1);
      }
    }
    const int done = r.terminated | r.truncated;
    if (done && a.final_obs) { WARP_FOR(i, od) a.final_obs[e * od + i] = s.obs[i]; }
    if (done && c.auto_reset) {
      env_reset(m, *a.c_dev, s, *a.opt_dev, a.seed, a.env_base + (unsigned long long)e);
      ContactFlags cf = contact_flags(m, c, s);
      write_obs(m, c, s, cf);
    }
    WARP_FOR(i, od) a.obs[e * od + i] = s.obs[i];
    IF_LANE0 { a.rew[e] = r.reward; a.term[e] = (uint8_t)r.terminated; a.trunc[e] = (uint8_t)r.truncated; }
    WARP_SYNC();
    WARP_FOR(i, NW) gst[i] = sst[i];
    WARP_SYNC();
  }
}

template <typename Real, typename D>
__global__ void state_io_kernel(EnvState<Real, D>* st, long long n, int nq, int nv, Real* qpos, Real* qvel, Real* ws) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long e = i / 64; int k = (int)(i % 64);
  if (e >= n) return;
  if (k < nq && qpos) qpos[e * nq + k] = st[e].qpos[k];
  if (k < nv && qvel) qvel[e * nv + k] = st[e].qvel[k];
  if (k < nv && ws) ws[e * nv + k] = st[e].qacc_ws[k];
}

template <typename Real, typename D>
__global__ void stats_kernel(EnvState<Real, D>* st, long long n, double* out, int reset) {
  long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (int k = 0; k < NSTAT; ++k) {
    double d = 0.0;
    if (e < n) { d = k == ST_RETURN ? (double)st[e].stat[k].f : (double)st[e].stat[k].i; if (reset) st[e].stat[k].i = 0; }
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
    if ((threadIdx.x & 31) == 0 && d != 0.0) atomicAdd(out + k, d);
  }
}

// Rollout sources: one warp per rollout j copies record ids[j] of the batch with 128-bit accesses, as step_kernel loads it, and zeroes
// the copy's stat[] counters (rollout_info_kernel reads them; the step never reads them, so no trajectory changes).  An id outside
// [0, n) gets a bad state instead: NaN qpos / qvel / warm start / cache, zero elsewhere, which the step's mj_checkPos/Vel guard resets
// to qpos0 at the first substep and counts in stat[ST_UNSTABLE].
template <typename Real, typename D>
__global__ void rollout_gather_kernel(const EnvState<Real, D>* src, long long n, const int* ids, EnvState<Real, D>* dst, long long m) {
  const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= m) return;
  constexpr int NW = sizeof(EnvState<Real, D>) / 16;
  const long long e = ids[j];
  int4* d = reinterpret_cast<int4*>(dst + j);
  const bool valid = e >= 0 && e < n;
  if (valid) {
    const int4* g = reinterpret_cast<const int4*>(src + e);
    for (int i = lane; i < NW; i += 32) d[i] = g[i];
  } else {
    for (int i = lane; i < NW; i += 32) d[i] = make_int4(0, 0, 0, 0);
  }
  __syncwarp();
  EnvState<Real, D>& r = dst[j];
  if (valid) {
    if (lane < NSTAT) r.stat[lane].i = 0;
  } else {
    const Real nan = std::numeric_limits<Real>::quiet_NaN();
    for (int i = lane; i < D::NQ; i += 32) r.qpos[i] = nan;
    for (int i = lane; i < D::NV; i += 32) { r.qvel[i] = nan; r.qacc_ws[i] = nan; }
    for (int i = lane; i < CACHE_SIZE; i += 32) r.cache[i] = nan;
  }
}

// Rollout info: env-steps with a bad-state reset and env-steps with an overflow, counted by the step in the scratch records since the gather.
template <typename Real, typename D>
__global__ void rollout_info_kernel(const EnvState<Real, D>* st, long long m, int32_t* info) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  info[2 * j] = st[j].stat[ST_UNSTABLE].i;
  info[2 * j + 1] = st[j].stat[ST_OVERFLOW].i;
}

template <typename Real, typename D>
struct QArgs {
  const DevModel<Real>* m;
  const EnvState<Real, D>* st;
  const QueryEntry<Real>* q; int k;
  long long n;
  Real *pos, *mat, *vel; int local;
};

// Kinematics queries (query.cuh): one warp per environment on the contact-free arena QueryDims<D>; reads qpos (and qvel when
// velocities are wanted) of the record, writes [n, k, 3 | 9 | 6] outputs, never the record.
template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, QueryDims<D>>() * 32) query_kernel(const QArgs<Real, D> a) {
  using DK = QueryDims<D>;
  constexpr int WPB = warps_per_block<Real, DK>();
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long e = (long long)blockIdx.x * WPB + warp;
  if (e >= a.n) return;
  Arena<Real, DK>& s = *reinterpret_cast<Arena<Real, DK>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, DK>());
  const DevModel<Real>& m = *a.m;
  const EnvState<Real, D>& rec = a.st[e];
  WARP_FOR(i, m.nq) s.st.qpos[i] = rec.qpos[i];
  if (a.vel) { WARP_FOR(i, m.nv) s.st.qvel[i] = rec.qvel[i]; }
  WARP_SYNC();
  const long long k = a.k;
  query_env(m, s, a.q, a.k, a.pos ? a.pos + e * k * 3 : nullptr, a.mat ? a.mat + e * k * 9 : nullptr, a.vel ? a.vel + e * k * 6 : nullptr, a.local);
}

template <typename Real, typename D>
struct QJArgs {
  const DevModel<Real>* m;
  const EnvState<Real, D>* st;
  const QueryEntry<Real>* q; int k;   // k = 0 (q null): no objects, M / qfrc_bias only
  long long n;
  Real *jacp, *jacr, *M, *bias;
};

// Jacobians, mass matrix and bias forces (query.cuh query_jac_env): one warp per environment on the same arena as query_kernel;
// reads qpos (and qvel when M or qfrc_bias is wanted) of the record, writes [n, k, 3, nv] / [n, nv, nv] / [n, nv], never the record.
template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, QueryDims<D>>() * 32) query_jac_kernel(const QJArgs<Real, D> a) {
  using DK = QueryDims<D>;
  constexpr int WPB = warps_per_block<Real, DK>();
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long e = (long long)blockIdx.x * WPB + warp;
  if (e >= a.n) return;
  Arena<Real, DK>& s = *reinterpret_cast<Arena<Real, DK>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, DK>());
  const DevModel<Real>& m = *a.m;
  const EnvState<Real, D>& rec = a.st[e];
  WARP_FOR(i, m.nq) s.st.qpos[i] = rec.qpos[i];
  if (a.M || a.bias) { WARP_FOR(i, m.nv) s.st.qvel[i] = rec.qvel[i]; }
  WARP_SYNC();
  const long long nv = m.nv, kj = (long long)a.k * 3 * nv;
  query_jac_env(m, s, a.q, a.k, a.jacp ? a.jacp + e * kj : nullptr, a.jacr ? a.jacr + e * kj : nullptr, a.M ? a.M + e * nv * nv : nullptr,
                a.bias ? a.bias + e * nv : nullptr);
}

template <typename Real, typename D>
struct QFArgs {
  const DevModel<Real>* m;
  const EnvState<Real, D>* st;
  SolverOpts<Real> opt;   // the step's own solver options
  long long n;
  const Real* ctrl;       // [n, nu] or null (zero)
  FwdOut<Real> o;         // batch-wide outputs: environment e's start at e times each output's per-environment size
};

// Forward-dynamics queries (query_fwd.cuh forward_query_env): one warp per environment on the generic size class's own arena, so the
// contact and row caps are the step's largest; reads the whole record (the solver warm-starts from qacc_ws), never writes it.
template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, D>() * 32, 1) query_fwd_kernel(const QFArgs<Real, D> a) {
  constexpr int WPB = warps_per_block<Real, D>();
  constexpr long long C = D::HAS_CONTACT ? D::MAXCON : 0;
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long e = (long long)blockIdx.x * WPB + warp;
  if (e >= a.n) return;
  Arena<Real, D>& s = *reinterpret_cast<Arena<Real, D>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, D>());
  const DevModel<Real>& m = *a.m;
  constexpr int NW = sizeof(EnvState<Real, D>) / 16;
  const int4* gst = reinterpret_cast<const int4*>(a.st + e);
  int4* sst = reinterpret_cast<int4*>(&s.st);
  WARP_FOR(i, NW) sst[i] = gst[i];
  const long long nv = m.nv;
  FwdOut<Real> o;
  o.qacc = a.o.qacc ? a.o.qacc + e * nv : nullptr;
  o.qfrc_constraint = a.o.qfrc_constraint ? a.o.qfrc_constraint + e * nv : nullptr;
  o.info = a.o.info ? a.o.info + e * 4 : nullptr;
  o.contact_geom = a.o.contact_geom ? a.o.contact_geom + e * C * 2 : nullptr;
  o.contact_dist = a.o.contact_dist ? a.o.contact_dist + e * C : nullptr;
  o.contact_pos = a.o.contact_pos ? a.o.contact_pos + e * C * 3 : nullptr;
  o.contact_frame = a.o.contact_frame ? a.o.contact_frame + e * C * 9 : nullptr;
  o.contact_force = a.o.contact_force ? a.o.contact_force + e * C * 6 : nullptr;
  o.flags = a.o.flags ? a.o.flags + e : nullptr;
  o.sensordata = a.o.sensordata ? a.o.sensordata + e * NSENSOR : nullptr;
  forward_query_env(m, s, a.opt, a.ctrl ? a.ctrl + e * m.nu : nullptr, o);
}

template <typename Real, typename D>
struct QIArgs {
  const DevModel<Real>* m;
  const EnvState<Real, D>* st;            // the stored state, read when qpos / qvel are null
  const Real* qpos; const Real* qvel;     // [count, nq], [count, nv] given states, or null
  long long count;
  const Real* qacc;                       // [count, nv]
  int discrete;
  InvOut<Real> o;                         // outputs: state i's start at i times each output's per-state size
};

// Inverse-dynamics queries (query_inv.cuh inverse_query_env): one warp per state on the generic size class's own arena, so the
// contact and row caps are those of the forward query; reads qpos and qvel of the record or of the given arrays, never writes a record.
template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, D>() * 32, 1) query_inv_kernel(const QIArgs<Real, D> a) {
  constexpr int WPB = warps_per_block<Real, D>();
  constexpr long long C = D::HAS_CONTACT ? D::MAXCON : 0;
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * WPB + warp;
  if (i >= a.count) return;
  Arena<Real, D>& s = *reinterpret_cast<Arena<Real, D>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, D>());
  const DevModel<Real>& m = *a.m;
  const long long nq = m.nq, nv = m.nv;
  const Real* qp = a.qpos ? a.qpos + i * nq : a.st[i].qpos;
  const Real* qv = a.qvel ? a.qvel + i * nv : a.st[i].qvel;
  WARP_FOR(j, m.nq) s.st.qpos[j] = qp[j];
  WARP_FOR(j, m.nv) s.st.qvel[j] = qv[j];
#ifdef UR3E_CANARY
  canary_set(s);
#endif
  InvOut<Real> o;
  o.qfrc_inverse = a.o.qfrc_inverse ? a.o.qfrc_inverse + i * nv : nullptr;
  o.qfrc_constraint = a.o.qfrc_constraint ? a.o.qfrc_constraint + i * nv : nullptr;
  o.info = a.o.info ? a.o.info + i * 3 : nullptr;
  o.contact_geom = a.o.contact_geom ? a.o.contact_geom + i * C * 2 : nullptr;
  o.contact_force = a.o.contact_force ? a.o.contact_force + i * C * 6 : nullptr;
  inverse_query_env(m, s, a.discrete != 0, a.qacc + i * nv, o);
#ifdef UR3E_CANARY
  WARP_SYNC();
  { const int bad = canary_bad(s); if (bad) { IF_LANE0 printf("ur3e_b200: arena guard word clobbered (mask 0x%x, inverse state %lld)\n", bad, i); } }
#endif
}

template <typename Real, typename D>
struct IKArgs {
  const DevModel<Real>* m;
  const EnvState<Real, D>* st;
  const IkTable<Real>* tab;
  long long n, count;                 // batch size, problems
  const int* env_ids;                 // [count] or null
  const Real* qpos0;                  // [count, nq] or null (neither: environment i)
  const Real* target_pos; const Real* target_quat;   // [count, 3], [count, 4]; either may be null
  IkOpts<Real> opt;
  Real* qpos; Real* err_norm; int32_t* info;         // [count, nq], [count], [count, 2]; any may be null
};

// Inverse kinematics (ik.cuh ik_env): one warp per problem on the kinematics queries' arena; reads qpos of the record or of the
// caller's array, never writes a record.  An environment id outside [0, n) gets NaN qpos and err_norm and status IK_BAD_ENV.
template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, QueryDims<D>>() * 32) ik_kernel(const IKArgs<Real, D> a) {
  using DK = QueryDims<D>;
  constexpr int WPB = warps_per_block<Real, DK>();
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * WPB + warp;
  if (i >= a.count) return;
  const DevModel<Real>& m = *a.m;
  const long long nq = m.nq;
  Real* const qo = a.qpos ? a.qpos + i * nq : nullptr;
  Real* const eo = a.err_norm ? a.err_norm + i : nullptr;
  int32_t* const io = a.info ? a.info + 2 * i : nullptr;
  const Real* src;
  if (a.qpos0) src = a.qpos0 + i * nq;
  else {
    const long long e = a.env_ids ? (long long)a.env_ids[i] : i;
    if (e < 0 || e >= a.n) {
      const Real nan = std::numeric_limits<Real>::quiet_NaN();
      if (qo) { WARP_FOR(j, m.nq) qo[j] = nan; }
      IF_LANE0 { if (eo) *eo = nan; if (io) { io[0] = 0; io[1] = IK_BAD_ENV; } }
      return;
    }
    src = a.st[e].qpos;
  }
  Arena<Real, DK>& s = *reinterpret_cast<Arena<Real, DK>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, DK>());
  WARP_FOR(j, m.nq) s.st.qpos[j] = src[j];
  WARP_SYNC();
  const IkResult<Real> r = ik_env(m, s, *a.tab, a.target_pos ? a.target_pos + 3 * i : nullptr, a.target_quat ? a.target_quat + 4 * i : nullptr, a.opt);
  if (qo) { WARP_FOR(j, m.nq) qo[j] = s.st.qpos[j]; }
  IF_LANE0 { if (eo) *eo = r.err_norm; if (io) { io[0] = r.steps; io[1] = r.status; } }
}

template <typename Real, typename D>
struct DistArgs {
  const DevModel<Real>* m;
  const EnvState<Real, D>* st;
  const DistPair<Real>* tab; int k;
  long long n, count;                 // batch size, states
  const int* env_ids;                 // [count] or null
  const Real* qpos;                   // [count, nq] or null (neither: environment i)
  Real distmax;
  Real* dist; Real* fromto;           // [count, k], [count, k, 6]; either may be null
};

// Geom distances (distance.cuh distance_env): one warp per state on the kinematics queries' arena, whose union u holds the overlapping
// pairs' staging rows; reads qpos of the record or of the caller's array, never writes a record.  An environment id outside [0, n)
// gets NaN dist and fromto.
template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, QueryDims<D>>() * 32) distance_kernel(const DistArgs<Real, D> a) {
  using DK = QueryDims<D>;
  constexpr int WPB = warps_per_block<Real, DK>();
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * WPB + warp;
  if (i >= a.count) return;
  const DevModel<Real>& m = *a.m;
  const long long k = a.k;
  Real* const dst = a.dist ? a.dist + i * k : nullptr;
  Real* const ft = a.fromto ? a.fromto + i * k * 6 : nullptr;
  const Real* src;
  if (a.qpos) src = a.qpos + i * (long long)m.nq;
  else {
    const long long e = a.env_ids ? (long long)a.env_ids[i] : i;
    if (e < 0 || e >= a.n) {
      const Real nan = std::numeric_limits<Real>::quiet_NaN();
      if (dst) { WARP_FOR(j, a.k) dst[j] = nan; }
      if (ft) { WARP_FOR(j, 6 * a.k) ft[j] = nan; }
      return;
    }
    src = a.st[e].qpos;
  }
  Arena<Real, DK>& s = *reinterpret_cast<Arena<Real, DK>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, DK>());
#ifdef UR3E_CANARY
  canary_set(s);
#endif
  WARP_FOR(j, m.nq) s.st.qpos[j] = src[j];
  WARP_SYNC();
  distance_env(m, s, a.tab, a.k, a.distmax, dst, ft);
#ifdef UR3E_CANARY
  WARP_SYNC();
  { const int bad = canary_bad(s); if (bad) { IF_LANE0 printf("ur3e_b200: arena guard word clobbered (mask 0x%x, distance state %lld)\n", bad, i); } }
#endif
}

template <typename Real, typename D>
struct RPArgs {
  const DevModel<Real>* m;
  const EnvState<Real, D>* st;
  const QueryEntry<Real>* q; int k;   // k geoms, then the camera
  long long n, count;                 // batch size, selected environments
  const int* env_ids;                 // [count] or null (environment i)
  Real* pose;                         // [count, k + 1, 12]
};

// Render pose pass (render.cuh render_pose_env): one warp per selected environment on the kinematics queries' arena; reads qpos of
// the record, writes the world poses of the renderer's geoms and camera.  An environment id outside [0, n) gets no pose (the pixel
// pass draws background for it).
template <typename Real, typename D>
__global__ void __launch_bounds__(warps_per_block<Real, QueryDims<D>>() * 32) render_pose_kernel(const RPArgs<Real, D> a) {
  using DK = QueryDims<D>;
  constexpr int WPB = warps_per_block<Real, DK>();
  extern __shared__ int4 smem_raw[];
  const int warp = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * WPB + warp;
  if (i >= a.count) return;
  const long long e = a.env_ids ? (long long)a.env_ids[i] : i;
  if (e < 0 || e >= a.n) return;
  Arena<Real, DK>& s = *reinterpret_cast<Arena<Real, DK>*>(reinterpret_cast<unsigned char*>(smem_raw) + warp * arena_stride<Real, DK>());
  const DevModel<Real>& m = *a.m;
  const EnvState<Real, D>& rec = a.st[e];
  WARP_FOR(j, m.nq) s.st.qpos[j] = rec.qpos[j];
  WARP_SYNC();
  render_pose_env(m, s, a.q, a.k, a.pose + i * 12 * (a.k + 1));
}

template <typename Real>
struct RArgs {
  const RenderGeom<Real>* geoms; int k;
  RenderCam<Real> cam;
  const Real* pose;                   // [m, k + 1, 12] from render_pose_kernel
  const int* env_ids; long long n;
  unsigned char* rgb; Real* depth; int* seg;   // [m, H, W, 3], [m, H, W], [m, H, W]; any may be null
};

constexpr int RENDER_THREADS = 256, RENDER_TILE = 1024;   // pixels per block: the staged scene is shared by RENDER_TILE rays
// Render pixel pass (render.cuh render_pixel): block (i, tile) stages environment i's camera and geoms in shared memory, then each
// thread casts the rays of its pixels; outputs are written along image rows.
template <typename Real>
__global__ void __launch_bounds__(RENDER_THREADS) render_kernel(const RArgs<Real> a) {
  extern __shared__ int4 smem_raw[];
  const int k = a.k;
  Real* sp = reinterpret_cast<Real*>(smem_raw);
  RenderGeom<Real>* sg = reinterpret_cast<RenderGeom<Real>*>(sp + 12 * (k + 1));
  const long long i = blockIdx.x;
  const long long e = a.env_ids ? (long long)a.env_ids[i] : i;
  const bool valid = e >= 0 && e < a.n;   // uniform over the block
  if (valid) {
    const Real* src = a.pose + i * 12 * (k + 1);
    for (int t = threadIdx.x; t < 12 * (k + 1); t += blockDim.x) sp[t] = src[t];
    for (int t = threadIdx.x; t < k; t += blockDim.x) sg[t] = a.geoms[t];
  }
  __syncthreads();
  const int W = a.cam.width, npx = W * a.cam.height;
  const int p0 = blockIdx.y * RENDER_TILE, p1 = p0 + RENDER_TILE < npx ? p0 + RENDER_TILE : npx;
  for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
    RenderPixel<Real> r;
    if (valid) r = render_pixel(a.cam, sp, sg, k, p % W, p / W);
    else { r.depth = a.cam.zfar; r.seg = -1; r.rgb[0] = r.rgb[1] = r.rgb[2] = 0; }
    const long long o = i * npx + p;
    if (a.rgb) { a.rgb[3 * o] = r.rgb[0]; a.rgb[3 * o + 1] = r.rgb[1]; a.rgb[3 * o + 2] = r.rgb[2]; }
    if (a.depth) a.depth[o] = r.depth;
    if (a.seg) a.seg[o] = r.seg;
  }
}

// D: generic size class of the model family; DL: lite twin (small caps, exact-fit) or D; DM: grasp-tier twin (caps between DL's and D's,
// exact-fit) or D.  Tiers hand environments up through device-side lists: DL -> DM -> D.
template <typename Real, typename D, typename DL = D, typename DM = D>
struct Batch : BatchBase {
  static constexpr bool HAS_LITE = !std::is_same<D, DL>::value;
  static constexpr bool HAS_MID = !std::is_same<D, DM>::value;
  static_assert(sizeof(EnvState<Real, D>) == sizeof(EnvState<Real, DM>), "all size classes of a model must share the record layout");
  int *d_ovf_list2 = nullptr, *d_ovf_list3 = nullptr;
  // overflow-counter slots, each with its own side stream and events: one per range of step_host (slot 0 is also step's), then the rollouts'
  static constexpr int HOST_CHUNKS = 4, ROLLOUT_SLOT = HOST_CHUNKS, NSLOT = HOST_CHUNKS + 1;
  cudaStream_t aux_stream[NSLOT] = {}; cudaEvent_t fork_ev[NSLOT] = {}, join_ev[NSLOT] = {};
  static_assert(sizeof(EnvState<Real, D>) == sizeof(EnvState<Real, DL>), "lite and full size classes must share the record layout");
  int *d_ovf_count = nullptr, *d_ovf_list = nullptr, *h_ovf = nullptr; cudaEvent_t ovf_ev = nullptr, order_ev = nullptr; bool ovf_pending = false; int h_ovf_seen = 0;
  cudaStream_t last_stream = nullptr;   // stream of the latest asynchronous call on this handle (step_host orders itself after it)
  long long lite_steps = 0, full_steps = 0; bool single_tier = false; int lite_cap_con = DL::MAXCON, lite_cap_efc = DL::MAXEFC;
  void tier_steps(int64_t* lite, int64_t* full) const override { *lite = lite_steps; *full = full_steps; }
  int64_t last_overflow() const override { return (ovf_pending && cudaEventQuery(ovf_ev) != cudaSuccess) ? h_ovf_seen : (h_ovf ? *h_ovf : 0); }
  void* sens_dev = nullptr;
  DevModel<Real>* d_model = nullptr;
  struct DevConsts { EnvCfg<Real> c; SolverOpts<Real> opt; };
  DevConsts* d_consts = nullptr;
  EnvState<Real, D>* d_state = nullptr;
  KArgs<Real> base;
  HostModel hm;
  int act_dim = 0, obs_dim = 0;
  // staging for the host-buffer entry point
  Real *d_act = nullptr, *d_obs = nullptr, *d_rew = nullptr; uint8_t *d_term = nullptr, *d_trunc = nullptr;
  cudaStream_t own_stream = nullptr, own_stream2 = nullptr;
  uint64_t seed = 0;
  int sm_count = 148;

  ~Batch() override {
    cudaSetDevice(device);
    cudaFree(d_ovf_count); cudaFree(d_ovf_list); cudaFree(d_ovf_list2); cudaFree(d_ovf_list3);
    for (int k = 0; k < NSLOT; ++k) { if (aux_stream[k]) cudaStreamDestroy(aux_stream[k]); if (fork_ev[k]) cudaEventDestroy(fork_ev[k]); if (join_ev[k]) cudaEventDestroy(join_ev[k]); } if (h_ovf) cudaFreeHost(h_ovf); if (ovf_ev) cudaEventDestroy(ovf_ev); if (order_ev) cudaEventDestroy(order_ev);
    cudaFree(d_model); cudaFree(d_consts); cudaFree(d_state); cudaFree(d_act); cudaFree(d_obs); cudaFree(d_rew); cudaFree(d_term); cudaFree(d_trunc);
    for (auto& t : timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (auto e : ev_pool) cudaEventDestroy(e);
    for (auto& q : queries) cudaFree(q.table);
    for (auto& r : renders) { cudaFree(r.table); cudaFree(r.geoms); }
    for (auto t : iks) cudaFree(t);
    for (auto& d : dists) cudaFree(d.table);
    cudaFree(d_pose); cudaFree(d_roll);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (own_stream2) cudaStreamDestroy(own_stream2);
  }
  static constexpr int WPB = warps_per_block<Real, D>();
  // env_kernel and the queries: one warp per environment of the batch, one arena of class DA per warp
  // (count: how many environments the kernel runs, the batch's n when 0)
  template <typename DA, typename A> int launch_warps(void (*kernel)(A), const A& a, cudaStream_t s, long long count = 0) {
    constexpr int W = warps_per_block<Real, DA>();
    const long long c = count > 0 ? count : n;
    kernel<<<(unsigned)((c + W - 1) / W), W * 32, arena_stride<Real, DA>() * W, s>>>(a);
    ++launches;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
  int init(const HostModel& h, const ur3e_env_config& cfg, long long n_envs, int dev) {
    device = dev; n = n_envs; hm = h;
    CUDA_OK(cudaSetDevice(dev));
    std::vector<int> bmap;
    const HostModel hmerged = merge_fixed_bodies(h, bmap);
    if (hmerged.nbody > D::NB) return set_err("merged model has more bodies than the kernel size class");
    DevModel<Real> m = compile_model<Real>(hmerged);
    if (m.ngeom > D::NG || m.npair > D::NPAIR || m.nv > D::NV || m.nq > D::NQ || m.nu > D::NU) return set_err("model exceeds the kernel size class (geoms / pairs / dofs)");
    if (m.ndeq > 3 * D::MAXCONNECT) return set_err("model has more connect equalities than the kernel size class stores rows for");
    auto body = [&](const char* nm) { int b = h.name2id(OBJ_BODY, nm); return b >= 0 ? bmap[b] : -1; };
    set_geom_flags(h, m);
    CUDA_OK(cudaMalloc(&d_model, sizeof m)); CUDA_OK(cudaMemcpy(d_model, &m, sizeof m, cudaMemcpyHostToDevice));
    CUDA_OK(cudaMalloc(&d_state, sizeof(EnvState<Real, D>) * n_envs)); CUDA_OK(cudaMemset(d_state, 0, sizeof(EnvState<Real, D>) * n_envs));
    std::memset(&base, 0, sizeof base);
    EnvCfg<Real>& c = base.c;
    c.ctrl_mode = cfg.ctrl_mode; c.obs_kind = cfg.obs_kind; c.reward_kind = cfg.reward_kind; c.term_kind = cfg.term_kind;
    c.frame_skip = cfg.frame_skip; c.act_dim = cfg.act_dim; c.obs_dim = cfg.obs_dim; c.max_steps = cfg.max_steps;
    c.reset_key = cfg.reset_key; c.reset_noise = cfg.reset_noise; c.auto_reset = cfg.auto_reset;
    for (int k = 0; k < 24; ++k) c.gains[k] = (Real)cfg.gains[k];
    for (int k = 0; k < 3; ++k) c.tool_rotvec[k] = (Real)cfg.tool_rotvec[k];
    auto tracked = [&](const char* nm) { for (int k = 0; k < m.nsite; ++k) if (std::string(tracked_site_names()[k]) == nm) return k; return -1; };
    c.site_tcp = tracked("tcp"); c.site_mug = tracked("handle_site"); c.site_pad = tracked("right_pad1_site");
    c.body_mug = body("fish"); c.body_ghost = body("ghost");
    c.body_lpad = body("left_pad"); c.body_rpad = body("right_pad"); c.body_table = body("table");
    c.finger_q = 6;  // utils/utils.py:319-326 reads d.qpos[6] / d.qvel[6]
    c.topple_z = 0;
    if (c.body_mug >= 0) {
      for (int g = 0; g < h.ngeom; ++g) if (h.I("geom_bodyid")[g] == h.name2id(OBJ_BODY, "fish")) {  // utils/utils.py:193-196 get_body_size = first geom
        const double* sz = &h.D("geom_size")[3 * g];
        for (int k = 0; k < 3; ++k) c.mug_size[k] = (Real)sz[k];
        c.topple_z = (Real)(sz[0] > sz[1] ? sz[0] : sz[1]);
        break;
      }
    }
    bool needs_task = c.ctrl_mode == CTRL_PID_TASK || c.ctrl_mode == CTRL_PID_TASK_ENV || c.ctrl_mode == CTRL_PINV;
    if (needs_task && c.site_tcp < 0) return set_err("controller needs a 'tcp' site");
    if (c.obs_kind != OBS_STATE && (c.site_tcp < 0 || c.site_mug < 0 || c.body_ghost < 0 || c.body_mug < 0)) return set_err("observation kind needs the tcp/handle_site sites and the fish/ghost bodies (main.xml)");
    if (c.obs_kind == OBS_V0 && c.site_pad < 0) return set_err("OBS_V0 needs right_pad1_site");
    int want_obs = c.obs_kind == OBS_STATE ? h.nq + h.nv : c.obs_kind == OBS_V2 ? 24 : 13;
    if (c.obs_dim != want_obs || c.obs_dim > 32) return set_err("obs_dim does not match obs_kind (expected " + std::to_string(want_obs) + ")");
    int want_act = c.ctrl_mode == CTRL_RAW ? h.nu : c.ctrl_mode == CTRL_PD_JOINT ? (h.nu > 6 ? 7 : 6) : (c.ctrl_mode == CTRL_PID_TASK || c.ctrl_mode == CTRL_PINV) ? 7 : 4;
    if (c.act_dim != want_act) return set_err("act_dim does not match ctrl_mode (expected " + std::to_string(want_act) + ")");
    if (c.frame_skip < 1 || c.frame_skip > MAX_FRAME_SKIP) return set_err("frame_skip must be in [1, " + std::to_string(MAX_FRAME_SKIP) + "]");
    if (c.reset_key >= h.nkey) return set_err("reset_key out of range");
    const bool f64 = sizeof(Real) == 8;
    base.opt.max_iter = cfg.solver_iterations > 0 ? cfg.solver_iterations : (f64 ? 50 : 8);
    base.opt.tol = cfg.solver_tolerance > 0 ? (Real)cfg.solver_tolerance : (f64 ? Real(1e-15) : Real(1e-7));
    base.opt.max_ls = f64 ? 50 : 12; base.opt.ls_tol = f64 ? Real(1e-14) : Real(UR3E_LS_TOL);
    base.opt.rtol = f64 ? Real(1e-15) : Real(2e-6);
    base.opt.tol_improve = f64 ? Real(0) : Real(1e-8);   // MuJoCo's default solver tolerance (assets/*.xml do not override it)
    base.m = d_model; base.st = d_state; base.n = n_envs; base.env_base = (unsigned long long)cfg.env_id_base;
    { DevConsts hc; hc.c = base.c; hc.opt = base.opt;
      CUDA_OK(cudaMalloc(&d_consts, sizeof hc)); CUDA_OK(cudaMemcpy(d_consts, &hc, sizeof hc, cudaMemcpyHostToDevice));
      base.c_dev = &d_consts->c; base.opt_dev = &d_consts->opt; }
    act_dim = c.act_dim; obs_dim = c.obs_dim; single_tier = cfg.single_tier != 0;
    if constexpr (HAS_LITE && DL::EXACT) {
      // the lite kernel is compiled for exactly these sizes (Dims::EXACT); any other model of this class runs on the full tier alone
      if (m.nv != DL::NV || m.nbody != DL::NB || m.nq != DL::NQ || m.nu != DL::NU || m.ngeom != DL::NG || m.npair != DL::NPAIR) single_tier = true;
      using SM = StaticModel<DL>;
      if (m.nlevel != SM::NLEVEL || m.nM != SM::NM || m.nfl != SM::NFL || m.neq != SM::NEQ || m.nsite != SM::NSITE || m.ndeq != SM::NDEQ || m.nej != SM::NEJ ||
          (m.has_damping != 0) != SM::DAMPING || m.split != DL::SPLIT) single_tier = true;
    }
    if constexpr (HAS_MID) {
      static_assert(HAS_LITE && DM::EXACT, "the grasp tier sits between an exact-fit lite tier and the generic class");
      constexpr int WM = warps_per_block<Real, DM>();
      CUDA_OK(cudaFuncSetAttribute(step_kernel<Real, DM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(arena_stride<Real, DM>() * WM)));
      CUDA_OK(cudaFuncSetAttribute(step_kernel<Real, DM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(arena_stride<Real, DM>() * WM)));
      CUDA_OK(cudaMalloc(&d_ovf_list2, sizeof(int) * n_envs)); CUDA_OK(cudaMalloc(&d_ovf_list3, sizeof(int) * n_envs));
      cudaFuncAttributes fm; CUDA_OK(cudaFuncGetAttributes(&fm, step_kernel<Real, DM>));
      mid_wpb = WM; mid_arena_bytes = (int)arena_stride<Real, DM>(); mid_regs = fm.numRegs;
    }
    if (cfg.lite_max_contacts > 0 && cfg.lite_max_contacts < DL::MAXCON) lite_cap_con = cfg.lite_max_contacts;
    if (cfg.lite_max_rows > 0 && cfg.lite_max_rows < DL::MAXEFC) lite_cap_efc = cfg.lite_max_rows;
    size_t smem = arena_stride<Real, D>() * WPB;
    CUDA_OK(cudaFuncSetAttribute(env_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaFuncAttributes fa; CUDA_OK(cudaFuncGetAttributes(&fa, env_kernel<Real, D>));
    wpb = WPB; regs = fa.numRegs; arena_bytes = (int)arena_stride<Real, D>(); state_bytes = (int)sizeof(EnvState<Real, D>);
    CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, env_kernel<Real, D>, WPB * 32, smem));
    CUDA_OK(cudaFuncSetAttribute(step_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_OK(cudaFuncSetAttribute(step_kernel<Real, D, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_OK(cudaFuncSetAttribute(query_fwd_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_OK(cudaFuncSetAttribute(query_inv_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    { using DK = QueryDims<D>;
      const int qsmem = (int)(arena_stride<Real, DK>() * warps_per_block<Real, DK>());
      CUDA_OK(cudaFuncSetAttribute(query_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, qsmem));
      CUDA_OK(cudaFuncSetAttribute(query_jac_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, qsmem));
      CUDA_OK(cudaFuncSetAttribute(render_pose_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, qsmem));
      CUDA_OK(cudaFuncSetAttribute(ik_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, qsmem));
      CUDA_OK(cudaFuncSetAttribute(distance_kernel<Real, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, qsmem)); }
    static_assert(sizeof(Real) * 12 * (RENDER_MAX_GEOMS + 1) + sizeof(RenderGeom<Real>) * RENDER_MAX_GEOMS <= 48 * 1024, "render_kernel's staged scene fits the default shared-memory limit");
    cudaDeviceProp prop; CUDA_OK(cudaGetDeviceProperties(&prop, dev)); sm_count = prop.multiProcessorCount;
    if constexpr (HAS_LITE) {
      constexpr int WL = warps_per_block<Real, DL>();
      CUDA_OK(cudaFuncSetAttribute(step_kernel<Real, DL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(arena_stride<Real, DL>() * WL)));
      CUDA_OK(cudaFuncSetAttribute(step_kernel<Real, DL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(arena_stride<Real, DL>() * WL)));
      CUDA_OK(cudaMalloc(&d_ovf_count, sizeof(int) * 4 * NSLOT)); CUDA_OK(cudaMalloc(&d_ovf_list, sizeof(int) * n_envs));
      CUDA_OK(cudaMallocHost(&h_ovf, sizeof(int))); *h_ovf = 0;
      CUDA_OK(cudaEventCreateWithFlags(&ovf_ev, cudaEventDisableTiming));
      cudaFuncAttributes fl; CUDA_OK(cudaFuncGetAttributes(&fl, step_kernel<Real, DL>));
      lite_wpb = WL; lite_arena_bytes = (int)arena_stride<Real, DL>(); lite_regs = fl.numRegs;
      CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&lite_blocks_per_sm, step_kernel<Real, DL>, WL * 32, arena_stride<Real, DL>() * WL));
    }
    { cudaFuncAttributes fs; CUDA_OK(cudaFuncGetAttributes(&fs, step_kernel<Real, D>)); regs = fs.numRegs;
      CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, step_kernel<Real, D>, WPB * 32, smem)); }
    CUDA_OK(cudaStreamCreateWithFlags(&own_stream, cudaStreamNonBlocking));
    return 0;
  }
  int reset(const uint8_t* mask, uint64_t sd, void* obs, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    seed = sd; last_stream = s;
    KArgs<Real> a = base; a.op = OP_RESET; a.mask = mask; a.seed = sd; a.obs = (Real*)obs;
    return launch_warps<D>(env_kernel<Real, D>, a, s);
  }
  // ---- optional per-launch timing (cudaEvent pairs on the launching stream)
  struct Timed { cudaEvent_t a, b; int tier; };
  bool timing = false; std::vector<Timed> timed; std::vector<cudaEvent_t> ev_pool; double t_ms[3] = {0, 0, 0}; long long t_n[3] = {0, 0, 0};
  int kernel_timing(int enable) override {
    double tmp[6]; if (int rc = kernel_times(tmp)) return rc;   // drain
    for (int k = 0; k < 3; ++k) { t_ms[k] = 0; t_n[k] = 0; }
    timing = enable != 0;
    return 0;
  }
  int kernel_times(double* out4) override {
    CUDA_OK(cudaSetDevice(device));
    for (auto& t : timed) {
      CUDA_OK(cudaEventSynchronize(t.b));
      float ms = 0; CUDA_OK(cudaEventElapsedTime(&ms, t.a, t.b));
      t_ms[t.tier] += ms; t_n[t.tier] += 1; ev_pool.push_back(t.a); ev_pool.push_back(t.b);
    }
    timed.clear();
    for (int k = 0; k < 3; ++k) { out4[2 * k] = t_ms[k]; out4[2 * k + 1] = (double)t_n[k]; }
    return 0;
  }
  int get_event(cudaEvent_t* e) { if (!ev_pool.empty()) { *e = ev_pool.back(); ev_pool.pop_back(); return 0; } CUDA_OK(cudaEventCreate(e)); return 0; }
  // tclass (timing only): 0 = lite tier, 1 = grasp / generic tier on the caller's stream (the step's critical path), 2 = generic tier on the side stream
  template <typename DD> int launch_step(KArgs<Real>& a, cudaStream_t s, unsigned blocks, int tclass = -1) {
    constexpr int W = warps_per_block<Real, DD>();
    Timed t{nullptr, nullptr, tclass >= 0 ? tclass : ((HAS_LITE && std::is_same<DD, DL>::value) ? 0 : 1)};
    if (timing) { if (int rc = get_event(&t.a)) return rc; if (int rc = get_event(&t.b)) return rc; CUDA_OK(cudaEventRecord(t.a, s)); }
    if (a.sens) step_kernel<Real, DD, true><<<blocks, W * 32, arena_stride<Real, DD>() * W, s>>>(a);
    else step_kernel<Real, DD><<<blocks, W * 32, arena_stride<Real, DD>() * W, s>>>(a);
    if (timing) { CUDA_OK(cudaEventRecord(t.b, s)); timed.push_back(t); }
    ++launches;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
  int step(const void* act, void* obs, void* rew, uint8_t* term, uint8_t* trunc, void* fobs, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    if (!act || !obs || !rew || !term || !trunc) return set_err("step: null buffer");
    last_stream = s;
    return step_range(live_range(0, n, 0), act, obs, rew, term, trunc, fobs, s);
  }
  // What one tiered step runs on: `cnt` records at `st`; the overflow counters, side stream and events of `slot` (so that targets
  // stepped concurrently on different streams share none) and its tier lists ([cnt] each); the sensor output (null = none); the
  // global id of the first record (auto-reset noise).  `live`: the batch's own records, auto-reset as configured and counted in
  // tier_info; otherwise a rollout's scratch records, never auto-reset.
  struct StepTarget { EnvState<Real, D>* st; long long cnt; int slot; int *list1, *list2, *list3; Real* sens; unsigned long long env_base; bool live; };
  // the batch's environments [lo, lo + cnt)
  StepTarget live_range(long long lo, long long cnt, int slot) const {
    auto at = [lo](int* l) { return l ? l + lo : nullptr; };
    return {d_state + lo, cnt, slot, at(d_ovf_list), at(d_ovf_list2), at(d_ovf_list3), sens_dev ? (Real*)sens_dev + lo * NSENSOR : nullptr,
            base.env_base + (unsigned long long)lo, true};
  }
  // One step of target g; the buffers are g's own ([g.cnt, ...]).
  int step_range(const StepTarget& g, const void* act, void* obs, void* rew, uint8_t* term, uint8_t* trunc, void* fobs, cudaStream_t s) {
    KArgs<Real> a = base; a.op = OP_STEP; a.seed = seed;
    if (!g.live) a.c.auto_reset = 0;
    const long long cnt = g.cnt; const int slot = g.slot;
    a.n = cnt; a.st = g.st; a.env_base = g.env_base;
    a.act = (const Real*)act; a.obs = (Real*)obs; a.rew = (Real*)rew; a.term = term; a.trunc = trunc;
    a.final_obs = (Real*)fobs;
    a.sens = g.sens;
    constexpr int WF = warps_per_block<Real, D>();
    const unsigned full_blocks = (unsigned)((cnt + WF - 1) / WF);
    if constexpr (!HAS_LITE) return launch_step<D>(a, s, full_blocks);
    else {
      // Tiered stepping.  The lite size class (small row / contact caps -> small arena -> more resident warps) steps every environment
      // except those whose record says they recently needed a larger size class (EnvState::tier); these, and the few that turn
      // out to exceed the lite caps during the step (left untouched by the lite kernel), are appended to device-side lists that
      // the larger size classes then step from resident grids.  The choice is a function of each environment's own history, made on
      // the device: no host read-back, no dependence on the batch size, the chunking of step_host, the world size or timing.
      // the four counters of a slot are adjacent (one memset): list 1, statistics, list 2, list 3
      int* const counter = d_ovf_count + 4 * slot;
      a.lite_maxcon = lite_cap_con; a.lite_maxefc = lite_cap_efc; a.ovf_stat = counter + 1;
      if (single_tier) {   // testing aid: the full size class alone, every environment
        a.lite_maxcon = 0;
        if (int rc = launch_step<D>(a, s, full_blocks)) return rc;
        if (g.live) ++full_steps;
        return 0;
      }
      constexpr int WL = warps_per_block<Real, DL>();
      constexpr bool CAN_OVERFLOW = DL::MAXCON < D::MAXCON || DL::MAXEFC < D::MAXEFC;   // an exact-fit twin with the same caps never overflows: no list, no tail
      const unsigned lite_blocks = (unsigned)((cnt + WL - 1) / WL);
      if constexpr (!CAN_OVERFLOW) {
        KArgs<Real> l = a; l.lite_maxcon = 0; l.ovf_stat = nullptr;
        if (int rc = launch_step<DL>(l, s, lite_blocks)) return rc;
        if (g.live) ++lite_steps;
        return 0;
      }
      int* const counter2 = counter + 2;   // list 2: straight to the generic class (from the lite tier's routing)
      int* const counter3 = counter + 3;   // list 3: exceeded the grasp tier's caps during this step
      CUDA_OK(cudaMemsetAsync(counter, 0, 4 * sizeof(int), s));
      const unsigned tail_blocks = (unsigned)(UR3E_BLOCKS_PER_SM * sm_count);
      KArgs<Real> l = a;
      l.ovf_count = counter; l.ovf_list = g.list1; l.cap_con = lite_cap_con; l.cap_efc = lite_cap_efc; l.lite_maxcon = 0; l.ovf_stat = nullptr;
      if constexpr (HAS_MID) {
        // Three tiers: lite -> grasp tier (list 1) -> generic class (lists 2 and 3).  The generic class's kernel takes the latency of one
        // environment step however short its list is, so the environments known to need it (list 2, routed by the lite tier from their
        // records) are stepped on a side stream WHILE the grasp tier steps list 1; only what the grasp tier itself could not hold
        // (list 3, normally empty) is stepped afterwards.
        constexpr int WM = warps_per_block<Real, DM>();
        const unsigned mid_blocks = (unsigned)((cnt + WM - 1) / WM);
        if (!aux_stream[slot]) {
          CUDA_OK(cudaStreamCreateWithFlags(&aux_stream[slot], cudaStreamNonBlocking));
          CUDA_OK(cudaEventCreateWithFlags(&fork_ev[slot], cudaEventDisableTiming)); CUDA_OK(cudaEventCreateWithFlags(&join_ev[slot], cudaEventDisableTiming));
        }
        l.ovf2_count = counter2; l.ovf2_list = g.list2;
        if (int rc = launch_step<DL>(l, s, lite_blocks)) return rc;
        a.mid_maxcon = DM::MAXCON; a.mid_maxefc = DM::MAXEFC;
        CUDA_OK(cudaEventRecord(fork_ev[slot], s)); CUDA_OK(cudaStreamWaitEvent(aux_stream[slot], fork_ev[slot], 0));
        KArgs<Real> f2 = a; f2.list_count = counter2; f2.list = g.list2;
        if (int rc = launch_step<D>(f2, aux_stream[slot], tail_blocks < full_blocks ? tail_blocks : full_blocks, 2)) return rc;
        KArgs<Real> mk = a;
        mk.list_count = counter; mk.list = g.list1; mk.ovf_count = counter3; mk.ovf_list = g.list3;
        if (int rc = launch_step<DM>(mk, s, tail_blocks < mid_blocks ? tail_blocks : mid_blocks)) return rc;
        CUDA_OK(cudaEventRecord(join_ev[slot], aux_stream[slot])); CUDA_OK(cudaStreamWaitEvent(s, join_ev[slot], 0));
        a.list_count = counter3; a.list = g.list3;
      } else {
        if (int rc = launch_step<DL>(l, s, lite_blocks)) return rc;
        a.list_count = counter; a.list = g.list1;
      }
      if (int rc = launch_step<D>(a, s, tail_blocks < full_blocks ? tail_blocks : full_blocks)) return rc;
      if (!g.live) return 0;
      ++lite_steps;
      if (!ovf_pending && slot == 0) {   // information only (ur3e_batch_tier_info): size of the full tier's list, read back without synchronising
        CUDA_OK(cudaMemcpyAsync(h_ovf, counter, sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaEventRecord(ovf_ev, s));
        ovf_pending = true;
      } else if (ovf_pending && cudaEventQuery(ovf_ev) == cudaSuccess) { ovf_pending = false; h_ovf_seen = *h_ovf; }
      return 0;
    }
  }
  int ensure_staging() {
    if (d_act) return 0;
    CUDA_OK(cudaMalloc(&d_act, sizeof(Real) * n * act_dim)); CUDA_OK(cudaMalloc(&d_obs, sizeof(Real) * n * obs_dim));
    CUDA_OK(cudaMalloc(&d_rew, sizeof(Real) * n)); CUDA_OK(cudaMalloc(&d_term, n)); CUDA_OK(cudaMalloc(&d_trunc, n));
    return 0;
  }
  // Host-buffer entry point.  The batch is cut into HOST_CHUNKS ranges that alternate between two streams, so that the
  // action upload and the result download of one range overlap the stepping of the next (pinned host buffers assumed;
  // pageable ones still work, the copies then serialise).
  int step_host(const void* act, void* obs, void* rew, uint8_t* term, uint8_t* trunc) override {
    CUDA_OK(cudaSetDevice(device));
    if (int rc = ensure_staging()) return rc;
    if (!own_stream2) CUDA_OK(cudaStreamCreateWithFlags(&own_stream2, cudaStreamNonBlocking));
    // this call runs on the batch's own streams: order it after the latest asynchronous call on this handle (a reset, step or
    // set_state on the caller's stream) with an event, so that no other stream of the device is stalled (a trainer's forward pass)
    if (!order_ev) CUDA_OK(cudaEventCreateWithFlags(&order_ev, cudaEventDisableTiming));
    CUDA_OK(cudaEventRecord(order_ev, last_stream));
    CUDA_OK(cudaStreamWaitEvent(own_stream, order_ev, 0));
    CUDA_OK(cudaStreamWaitEvent(own_stream2, order_ev, 0));
    const int chunks = n >= 4096 * HOST_CHUNKS ? HOST_CHUNKS : 1;
    const long long per = (n + chunks - 1) / chunks;
    for (int c = 0; c < chunks; ++c) {
      const long long lo = c * per, cnt = (lo + per <= n ? per : n - lo);
      if (cnt <= 0) break;
      cudaStream_t s = (c & 1) ? own_stream2 : own_stream;
      CUDA_OK(cudaMemcpyAsync(d_act + lo * act_dim, (const Real*)act + lo * act_dim, sizeof(Real) * cnt * act_dim, cudaMemcpyHostToDevice, s));
      if (int rc = step_range(live_range(lo, cnt, c), d_act + lo * act_dim, d_obs + lo * obs_dim, d_rew + lo, d_term + lo, d_trunc + lo, nullptr, s)) return rc;
      CUDA_OK(cudaMemcpyAsync((Real*)obs + lo * obs_dim, d_obs + lo * obs_dim, sizeof(Real) * cnt * obs_dim, cudaMemcpyDeviceToHost, s));
      CUDA_OK(cudaMemcpyAsync((Real*)rew + lo, d_rew + lo, sizeof(Real) * cnt, cudaMemcpyDeviceToHost, s));
      CUDA_OK(cudaMemcpyAsync(term + lo, d_term + lo, cnt, cudaMemcpyDeviceToHost, s));
      CUDA_OK(cudaMemcpyAsync(trunc + lo, d_trunc + lo, cnt, cudaMemcpyDeviceToHost, s));
    }
    CUDA_OK(cudaStreamSynchronize(own_stream));
    CUDA_OK(cudaStreamSynchronize(own_stream2));
    return 0;
  }
  // ---- kinematics queries (query.cuh); the tables live until the batch is destroyed
  struct Query { QueryEntry<Real>* table; int k; };
  std::vector<Query> queries;
  int query_create(const int32_t* objtype, const int32_t* objid, int k) override {
    CUDA_OK(cudaSetDevice(device));
    std::vector<QueryEntry<Real>> tab;
    const std::string err = compile_query<Real>(hm, objtype, objid, k, tab);
    if (!err.empty()) return set_err("query_create: " + err);
    Query q{nullptr, k};
    CUDA_OK(cudaMalloc(&q.table, sizeof(QueryEntry<Real>) * k));
    queries.push_back(q);
    CUDA_OK(cudaMemcpy(q.table, tab.data(), sizeof(QueryEntry<Real>) * k, cudaMemcpyHostToDevice));
    return (int)queries.size() - 1;
  }
  int query(int id, void* pos, void* mat, void* vel, int local, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    if (id < 0 || id >= (int)queries.size()) return set_err("query: unknown query id " + std::to_string(id));
    if (!pos && !mat && !vel) return set_err("query: all outputs are null");
    // a read-only call: last_stream (what step_host orders itself after) stays that of the latest state-changing call
    QArgs<Real, D> a{d_model, d_state, queries[id].table, queries[id].k, n, (Real*)pos, (Real*)mat, (Real*)vel, local != 0};
    return launch_warps<QueryDims<D>>(query_kernel<Real, D>, a, s);
  }
  int query_jac(int id, void* jacp, void* jacr, void* M, void* bias, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    const std::string err = query_jac_check(id, (int)queries.size(), jacp || jacr, jacp || jacr || M || bias);
    if (!err.empty()) return set_err("query_jac: " + err);
    // read-only, like query(): last_stream stays that of the latest state-changing call
    QJArgs<Real, D> a{d_model, d_state, id >= 0 ? queries[id].table : nullptr, id >= 0 ? queries[id].k : 0, n, (Real*)jacp, (Real*)jacr, (Real*)M, (Real*)bias};
    return launch_warps<QueryDims<D>>(query_jac_kernel<Real, D>, a, s);
  }
  static constexpr int NCMAX = D::HAS_CONTACT ? D::MAXCON : 0;
  int max_contacts() const override { return NCMAX; }
  int forward(const void* ctrl, const ur3e_forward_out* out, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    const bool con = out && (out->contact_geom || out->contact_dist || out->contact_pos || out->contact_frame || out->contact_force);
    const bool any = out && (con || out->qacc || out->qfrc_constraint || out->info || out->flags || out->sensordata);
    const std::string err = forward_query_check(out != nullptr, con, any, NCMAX);
    if (!err.empty()) return set_err("forward: " + err);
    // read-only, like query(): last_stream stays that of the latest state-changing call
    QFArgs<Real, D> a{d_model, d_state, base.opt, n, (const Real*)ctrl,
                      FwdOut<Real>{(Real*)out->qacc, (Real*)out->qfrc_constraint, out->info, out->contact_geom, (Real*)out->contact_dist,
                                   (Real*)out->contact_pos, (Real*)out->contact_frame, (Real*)out->contact_force, out->flags, (Real*)out->sensordata}};
    return launch_warps<D>(query_fwd_kernel<Real, D>, a, s);
  }
  int inverse(const void* qpos, const void* qvel, long long m, const void* qacc, int discrete, const ur3e_inverse_out* out, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    const bool con = out && (out->contact_geom || out->contact_force);
    const bool any = out && (con || out->qfrc_inverse || out->qfrc_constraint || out->info);
    const std::string err = inverse_query_check(qpos != nullptr, qvel != nullptr, m, n, qacc != nullptr, out != nullptr, con, any, NCMAX);
    if (!err.empty()) return set_err("inverse: " + err);
    // read-only, like query(): last_stream stays that of the latest state-changing call
    QIArgs<Real, D> a{d_model, d_state, (const Real*)qpos, (const Real*)qvel, m, (const Real*)qacc, discrete != 0,
                      InvOut<Real>{(Real*)out->qfrc_inverse, (Real*)out->qfrc_constraint, out->info, out->contact_geom, (Real*)out->contact_force}};
    return launch_warps<D>(query_inv_kernel<Real, D>, a, s, m);
  }
  // ---- offscreen rendering (render.cuh); renderers and the pose scratch live until the batch is destroyed
  struct Render { QueryEntry<Real>* table; RenderGeom<Real>* geoms; int k; RenderCam<Real> cam; };
  std::vector<Render> renders;
  Real* d_pose = nullptr; long long pose_cap = 0;   // [m, k + 1, 12] of the latest call, grown to the largest seen
  static size_t render_smem(int k) { return sizeof(Real) * 12 * (k + 1) + sizeof(RenderGeom<Real>) * k; }
  int render_create(const ur3e_camera* cam, const int32_t* geom_ids, int k, const float* rgba, int width, int height) override {
    CUDA_OK(cudaSetDevice(device));
    std::vector<QueryEntry<Real>> tab; std::vector<RenderGeom<Real>> geoms; RenderCam<Real> rc{};
    const std::string err = compile_render<Real>(hm, cam, geom_ids, k, rgba, width, height, tab, geoms, rc);
    if (!err.empty()) return set_err("render_create: " + err);
    Render r{nullptr, nullptr, k, rc};
    CUDA_OK(cudaMalloc(&r.table, sizeof(QueryEntry<Real>) * (k + 1)));
    if (cudaMalloc(&r.geoms, sizeof(RenderGeom<Real>) * k) != cudaSuccess) { cudaFree(r.table); return set_err("render_create: out of device memory", -2); }
    renders.push_back(r);
    CUDA_OK(cudaMemcpy(r.table, tab.data(), sizeof(QueryEntry<Real>) * (k + 1), cudaMemcpyHostToDevice));
    CUDA_OK(cudaMemcpy(r.geoms, geoms.data(), sizeof(RenderGeom<Real>) * k, cudaMemcpyHostToDevice));
    return (int)renders.size() - 1;
  }
  int render(int id, const int32_t* env_ids, long long m, uint8_t* rgb, void* depth, int32_t* seg, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    const std::string err = render_check(id, (int)renders.size(), rgb || depth || seg, m, n, env_ids != nullptr);
    if (!err.empty()) return set_err("render: " + err);
    const Render& r = renders[id];
    const long long need = m * 12 * (r.k + 1);
    if (need > pose_cap) {
      // cudaFree waits for the device, so a call still reading the old scratch finishes first
      CUDA_OK(cudaFree(d_pose)); d_pose = nullptr; pose_cap = 0;
      CUDA_OK(cudaMalloc(&d_pose, sizeof(Real) * need)); pose_cap = need;
    }
    // read-only, like query(): last_stream stays that of the latest state-changing call
    RPArgs<Real, D> pa{d_model, d_state, r.table, r.k, n, m, env_ids, d_pose};
    if (int rc = launch_warps<QueryDims<D>>(render_pose_kernel<Real, D>, pa, s, m)) return rc;
    RArgs<Real> ra{r.geoms, r.k, r.cam, d_pose, env_ids, n, rgb, (Real*)depth, seg};
    const unsigned tiles = (unsigned)((r.cam.width * r.cam.height + RENDER_TILE - 1) / RENDER_TILE);
    render_kernel<Real><<<dim3((unsigned)m, tiles), RENDER_THREADS, render_smem(r.k), s>>>(ra);
    ++launches;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
  // ---- inverse kinematics (ik.cuh); the tables live until the batch is destroyed
  std::vector<IkTable<Real>*> iks;
  int ik_create(int32_t objtype, int32_t objid, const int32_t* joint_ids, int nj) override {
    CUDA_OK(cudaSetDevice(device));
    IkTable<Real> tab;
    const std::string err = compile_ik<Real>(hm, objtype, objid, joint_ids, nj, tab);
    if (!err.empty()) return set_err("ik_create: " + err);
    IkTable<Real>* d = nullptr;
    CUDA_OK(cudaMalloc(&d, sizeof tab));
    iks.push_back(d);
    CUDA_OK(cudaMemcpy(d, &tab, sizeof tab, cudaMemcpyHostToDevice));
    return (int)iks.size() - 1;
  }
  int ik(int id, const int32_t* env_ids, const void* qpos0, long long m, const void* target_pos, const void* target_quat, const ur3e_ik_options* opt,
         const ur3e_ik_out* out, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    const bool any = out && (out->qpos || out->err_norm || out->info);
    const std::string err = ik_check(id, (int)iks.size(), m, n, env_ids != nullptr, qpos0 != nullptr, target_pos != nullptr, target_quat != nullptr,
                                     out != nullptr, any, opt);
    if (!err.empty()) return set_err("ik: " + err);
    const ur3e_ik_options o = opt ? *opt : ur3e_ik_options{ik_default_tol<Real>(), 1.0, 0.1, 3e-2, 2.0, 20.0, 100, 0};
    const IkOpts<Real> ko{(Real)o.tol, (Real)o.rot_weight, (Real)o.regularization_threshold, (Real)o.regularization_strength, (Real)o.max_update_norm,
                          (Real)o.progress_thresh, o.max_steps};
    // read-only, like query(): last_stream stays that of the latest state-changing call
    IKArgs<Real, D> a{d_model, d_state, iks[id], n, m, env_ids, (const Real*)qpos0, (const Real*)target_pos, (const Real*)target_quat, ko,
                      (Real*)out->qpos, (Real*)out->err_norm, out->info};
    return launch_warps<QueryDims<D>>(ik_kernel<Real, D>, a, s, m);
  }
  // ---- geom distances (distance.cuh); the pair tables live until the batch is destroyed
  struct DistSet { DistPair<Real>* table; int k; };
  std::vector<DistSet> dists;
  int distance_create(const int32_t* geom1, const int32_t* geom2, int k) override {
    CUDA_OK(cudaSetDevice(device));
    std::vector<DistPair<Real>> tab;
    const std::string err = compile_distance<Real>(hm, geom1, geom2, k, tab);
    if (!err.empty()) return set_err("distance_create: " + err);
    DistPair<Real>* d = nullptr;
    CUDA_OK(cudaMalloc(&d, sizeof(DistPair<Real>) * k));
    dists.push_back(DistSet{d, k});
    CUDA_OK(cudaMemcpy(d, tab.data(), sizeof(DistPair<Real>) * k, cudaMemcpyHostToDevice));
    return (int)dists.size() - 1;
  }
  int distance(int id, const int32_t* env_ids, const void* qpos, long long m, double distmax, void* dist, void* fromto, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    const std::string err = distance_check(id, (int)dists.size(), m, n, env_ids != nullptr, qpos != nullptr, dist || fromto, distmax);
    if (!err.empty()) return set_err("distance: " + err);
    // read-only, like query(): last_stream stays that of the latest state-changing call
    DistArgs<Real, D> a{d_model, d_state, dists[id].table, dists[id].k, n, m, env_ids, (const Real*)qpos, (Real)distmax, (Real*)dist, (Real*)fromto};
    return launch_warps<QueryDims<D>>(distance_kernel<Real, D>, a, s, m);
  }
  // ---- rollouts: T tiered steps (step_range) of a scratch batch of m records on the counter slot ROLLOUT_SLOT.  The workspace is
  // grown to the largest m seen: records [m], the three tier lists [m], and obs [m, obs_dim], reward [m], terminated [m] and
  // truncated [m] for the outputs the caller did not ask for (the step kernels always write them).
  unsigned char* d_roll = nullptr; long long roll_cap = 0;
  static size_t align256(size_t b) { return (b + 255) / 256 * 256; }
  int rollout(const int32_t* src, const void* qpos0, const void* qvel0, const void* ws0, long long m, int T, const void* act,
              const ur3e_rollout_out* out, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    const bool any = out && (out->qpos || out->qvel || out->obs || out->reward || out->terminated || out->truncated || out->sensordata || out->info);
    const std::string err = rollout_check(m, T, act != nullptr, src != nullptr, qpos0 != nullptr, qvel0 != nullptr, ws0 != nullptr, out != nullptr, any);
    if (!err.empty()) return set_err("rollout: " + err);
    const size_t b_st = align256(sizeof(EnvState<Real, D>) * m), b_list = align256(sizeof(int) * m), b_obs = align256(sizeof(Real) * m * obs_dim),
                 b_rew = align256(sizeof(Real) * m);
    if (m > roll_cap) {
      // cudaFree waits for the device, so a call still using the old workspace finishes first
      CUDA_OK(cudaFree(d_roll)); d_roll = nullptr; roll_cap = 0;
      CUDA_OK(cudaMalloc(&d_roll, b_st + 3 * b_list + b_obs + b_rew + 2 * align256(m))); roll_cap = m;
    }
    EnvState<Real, D>* const st = reinterpret_cast<EnvState<Real, D>*>(d_roll);
    unsigned char* p = d_roll + b_st;
    int* const lists = reinterpret_cast<int*>(p); p += 3 * b_list;
    Real* const s_obs = reinterpret_cast<Real*>(p); p += b_obs;
    Real* const s_rew = reinterpret_cast<Real*>(p); p += b_rew;
    uint8_t* const s_term = p; uint8_t* const s_trunc = p + align256(m);
    // read-only for the batch, like query(): last_stream stays that of the latest state-changing call
    if (src) {
      rollout_gather_kernel<Real, D><<<(unsigned)((m * 32 + 255) / 256), 256, 0, s>>>(d_state, n, src, st, m);
      ++launches;
      CUDA_OK(cudaGetLastError());
    } else {
      CUDA_OK(cudaMemsetAsync(st, 0, sizeof(EnvState<Real, D>) * m, s));
      KArgs<Real> a = base; a.op = OP_SET_STATE; a.st = st; a.n = m;
      a.qpos_in = (const Real*)qpos0; a.qvel_in = (const Real*)qvel0; a.ws_in = (const Real*)ws0;
      if (int rc = launch_warps<D>(env_kernel<Real, D>, a, s, m)) return rc;
    }
    StepTarget g{st, m, ROLLOUT_SLOT, lists, lists + b_list / sizeof(int), lists + 2 * (b_list / sizeof(int)), nullptr, 0, false};
    const int nq = hm.nq, nv = hm.nv;
    for (int t = 0; t < T; ++t) {
      const long long o = (long long)t * m;
      g.sens = out->sensordata ? (Real*)out->sensordata + o * NSENSOR : nullptr;
      if (int rc = step_range(g, (const Real*)act + o * act_dim, out->obs ? (Real*)out->obs + o * obs_dim : s_obs, out->reward ? (Real*)out->reward + o : s_rew,
                              out->terminated ? out->terminated + o : s_term, out->truncated ? out->truncated + o : s_trunc, nullptr, s)) return rc;
      if (out->qpos || out->qvel) {
        state_io_kernel<Real, D><<<(unsigned)((m * 64 + 255) / 256), 256, 0, s>>>(st, m, nq, nv, out->qpos ? (Real*)out->qpos + o * nq : nullptr,
                                                                                 out->qvel ? (Real*)out->qvel + o * nv : nullptr, nullptr);
        ++launches;
        CUDA_OK(cudaGetLastError());
      }
    }
    if (out->info) {
      rollout_info_kernel<Real, D><<<(unsigned)((m + 255) / 256), 256, 0, s>>>(st, m, out->info);
      ++launches;
      CUDA_OK(cudaGetLastError());
    }
    return 0;
  }
  int set_sensor_buffer(void* buf) override { sens_dev = buf; return 0; }
  int get_state(void* qpos, void* qvel, void* ws, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    last_stream = s;
    long long tot = n * 64;
    state_io_kernel<Real, D><<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(d_state, n, hm.nq, hm.nv, (Real*)qpos, (Real*)qvel, (Real*)ws);
    ++launches;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
  int set_state(const void* qpos, const void* qvel, const void* ws, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    if (!qpos || !qvel) return set_err("set_state: null buffer");
    last_stream = s;
    KArgs<Real> a = base; a.op = OP_SET_STATE; a.qpos_in = (const Real*)qpos; a.qvel_in = (const Real*)qvel; a.ws_in = (const Real*)ws;
    return launch_warps<D>(env_kernel<Real, D>, a, s);
  }
  int stats(double* out, int rst, cudaStream_t s) override {
    CUDA_OK(cudaSetDevice(device));
    last_stream = s;
    CUDA_OK(cudaMemsetAsync(out, 0, 16 * sizeof(double), s));
    stats_kernel<Real, D><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_state, n, out, rst);
    ++launches;
    CUDA_OK(cudaGetLastError());
    return 0;
  }
};


template <typename Real, typename D, typename DL = D, typename DM = D>
std::unique_ptr<BatchBase> make_batch(const HostModel& h, const ur3e_env_config& cfg, long long n, int device) {
  auto p = std::make_unique<Batch<Real, D, DL, DM>>();
  if (p->init(h, cfg, n, device)) return nullptr;
  return p;
}

}  // namespace ur3e
