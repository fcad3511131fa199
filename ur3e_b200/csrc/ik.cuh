// Inverse kinematics: the joint positions that put one object (a kinematics query's entry: site, body frame, inertial frame or geom)
// at a target position and / or orientation, by dm_control's qpos_from_site_pose loop (damped least squares on the object's
// Jacobian), one problem per warp off the step path.  Read-only: the caller loads qpos into the arena; nothing is written back to a
// record.  Like engine.cuh this file uses only warp_model.cuh constructs, so tests/hostcheck compiles it for the CPU.
//
// Semantics (dm_control.utils.inverse_kinematics.qpos_from_site_pose, batched), for step = 0, 1, ...:
//   kinematics at q;  e_pos = p* - p,  e_rot = rotvec(R(q*) R(q)^T) (world frame);  err_norm = |e_pos| + rot_weight |e_rot|
//   err_norm < tol: converged (IK_CONVERGED);  max_steps updates applied: IK_MAX_STEPS_HIT
//   J = the r x nj block of [jacp; jacr] at the object's point for the selected joints' dofs, rows only for the targets given
//   lambda = regularization_strength if err_norm > regularization_threshold, else 0;  dq = (J^T J + lambda I)^-1 J^T e
//   err_norm / |dq| > progress_thresh: IK_NO_PROGRESS, dq not applied
//   dq scaled down to max_update_norm;  q[joint] += dq (hinges: mj_integratePos is an add);  limited joints clamped to jnt_range
// Deliberate differences from dm_control:
//   - the limit clamp (a result outside the limits is pushed back by the step's limit rows); runs whose iterates stay inside the
//     limits are dm_control's;
//   - err_norm and steps describe the returned qpos: its error, and the number of updates applied (dm_control reports the error
//     before its last update and max_steps - 1 on exhaustion); converged means the returned qpos is within tol;
//   - any kinematics-query object, not only sites;
//   - with lambda = 0 the result is the minimum-norm least-squares step (J's pseudo-inverse, numpy's default lstsq cut-off);
//     dm_control's lstsq(J^T J, J^T e, rcond=-1) keeps rounding-noise singular values of the rank-deficient J^T J when r < nj.
// Only the selected joints' qpos entries change; equality constraints (the 2F85's four-bar) are not enforced.
#pragma once
#include <cmath>
#include <string>
#include <vector>

#include "env.cuh"
#include "query.cuh"

namespace ur3e {

constexpr int IK_MAX_JOINTS = 32;        // body_dofmask is 32 bits wide; a model has at most that many dofs
constexpr int IK_MAX_STEPS_CAP = 10000;  // the largest max_steps a call accepts (one warp per problem runs them back to back)
enum IkStatus { IK_CONVERGED = 0, IK_MAX_STEPS_HIT = 1, IK_NO_PROGRESS = 2, IK_BAD_ENV = 3 };

template <typename Real>
struct IkJoint {
  Real lo, hi;             // jnt_range, used when limited
  int dof, qadr, limited, pad_;
};

// One compiled IK problem family (ur3e_batch_ik_create): the object and the joints it may move.
template <typename Real>
struct IkTable {
  QueryEntry<Real> obj;
  int nj, pad_[3];
  IkJoint<Real> j[IK_MAX_JOINTS];
};

template <typename Real>
struct IkOpts {
  Real tol, rot_weight, reg_threshold, reg_strength, max_update_norm, progress_thresh;
  int max_steps;
};

// With lambda = 0 a pivot of the <= 6 x 6 LDL^T below this fraction of the system's largest diagonal entry contributes zero: J is
// singular there up to rounding (about a hundred times the unit roundoff of the normal equations).  lstsq's result differs from
// this only at exact singularities, as for CTRL_PINV's pseudo-inverse.
template <typename Real> constexpr Real ik_pivot_frac() { return sizeof(Real) == 8 ? Real(1e-13) : Real(1e-5); }

// tol when the caller gives none: dm_control's 1e-14 in float64; in float32 a value above the float32 noise floor of err_norm on
// main.xml (DESIGN §3)
template <typename Real> constexpr double ik_default_tol() { return sizeof(Real) == 8 ? 1e-14 : 1e-5; }

// Compiles the object (objtype, objid) of the loaded model h and the nj joints it may move.  Returns "" on success, else the reason.
template <typename Real>
std::string compile_ik(const HostModel& h, int32_t objtype, int32_t objid, const int32_t* joint_ids, int nj, IkTable<Real>& out) {
  std::vector<QueryEntry<Real>> q;
  const std::string err = compile_query<Real>(h, &objtype, &objid, 1, q);
  if (!err.empty()) return err;
  if (!joint_ids) return "null joint list";
  if (nj < 1 || nj > h.nv) return "nj=" + std::to_string(nj) + " joints is outside [1, nv=" + std::to_string(h.nv) + "]";
  out = IkTable<Real>{};
  out.obj = q[0]; out.nj = nj;
  const auto &jt = h.I("jnt_type"), &jd = h.I("jnt_dofadr"), &jq = h.I("jnt_qposadr"), &jl = h.I("jnt_limited");
  const auto& jr = h.D("jnt_range");
  for (int i = 0; i < nj; ++i) {
    const int j = joint_ids[i];
    if (j < 0 || j >= h.njnt) return "joint " + std::to_string(i) + ": id " + std::to_string(j) + " is out of range [0, " + std::to_string(h.njnt) + ")";
    for (int k = 0; k < i; ++k)
      if (joint_ids[k] == j) return "joint " + std::to_string(i) + ": id " + std::to_string(j) + " is listed twice";
    if (jt[j] != JNT_HINGE && jt[j] != JNT_SLIDE) return "joint " + std::to_string(i) + ": id " + std::to_string(j) + " is not a hinge or slide joint";
    IkJoint<Real>& o = out.j[i];
    o.dof = jd[j]; o.qadr = jq[j]; o.limited = jl[j] != 0;
    o.lo = o.limited ? (Real)jr[2 * j] : Real(0); o.hi = o.limited ? (Real)jr[2 * j + 1] : Real(0);
  }
  return "";
}

// Arguments of an IK call (ur3e_batch_ik): problem family `id` of `nik`, m problems, the batch's n, which sources and targets are
// given, `out` given, `any` = some output requested, the options (null = the defaults).  Returns "" when valid, else the reason.
inline std::string ik_check(int id, int nik, long long m, long long n, bool env_ids, bool qpos0, bool pos, bool quat, bool out, bool any,
                            const ur3e_ik_options* opt) {
  if (id < 0 || id >= nik) return "unknown ik id " + std::to_string(id);
  if (m < 1 || m > 2147483647LL) return "m=" + std::to_string(m) + " problems (1 .. 2^31 - 1)";
  if (env_ids && qpos0) return "give env_ids or qpos0, not both";
  if (!env_ids && !qpos0 && m != n) return "m=" + std::to_string(m) + " for the stored state of n=" + std::to_string(n) + " environments (m must equal n)";
  if (!pos && !quat) return "no target: target_pos and target_quat are both null";
  if (!out) return "out is null";
  if (!any) return "all outputs are null";
  if (opt) {
    // written as !(x >= 0) so that NaN is rejected too
    if (!(opt->tol >= 0)) return "tol must be >= 0";
    if (!(opt->rot_weight >= 0)) return "rot_weight must be >= 0";
    if (!(opt->regularization_threshold >= 0)) return "regularization_threshold must be >= 0";
    if (!(opt->regularization_strength >= 0)) return "regularization_strength must be >= 0";
    if (!(opt->max_update_norm > 0)) return "max_update_norm must be > 0";
    if (!(opt->progress_thresh > 0)) return "progress_thresh must be > 0";
    if (opt->max_steps < 1 || opt->max_steps > IK_MAX_STEPS_CAP) return "max_steps=" + std::to_string(opt->max_steps) + " is outside [1, " + std::to_string(IK_MAX_STEPS_CAP) + "]";
  }
  return "";
}

// Rotation vector (axis times angle in [0, pi]) of a quaternion (w, x, y, z), normalised first; |q| < 1e-15 is the identity (mju_normalize4)
template <typename Real> UR3E_HD void ik_quat_rotvec(const Real* q, Real* rv) {
  Real w = q[0], x = q[1], y = q[2], z = q[3];
  const Real nq = Num<Real>::sqrt(w * w + x * x + y * y + z * z);
  if (nq < Real(1e-15)) { rv[0] = rv[1] = rv[2] = 0; return; }
  w /= nq; x /= nq; y /= nq; z /= nq;
  if (w < 0) { w = -w; x = -x; y = -y; z = -z; }
  const Real sn = Num<Real>::sqrt(x * x + y * y + z * z);
  const Real k = sn > 0 ? 2 * Num<Real>::atan2(sn, w) / sn : Real(2);
  rv[0] = k * x; rv[1] = k * y; rv[2] = k * z;
}

template <typename Real> struct IkResult { Real err_norm; int steps, status; };

// Solves the one IK problem of this warp.  The caller has loaded qpos into s.st; target_pos [3] and / or target_quat [4] (either may
// be null, not both).  On return s.st.qpos holds the result; the error of that configuration, the updates applied and the status are
// returned (the same on every lane).
//
// Storage (DESIGN §3): the object's frame, J, the small system and the step live in the union u, whose kinematics view (the bodies'
// local frames) is dead once kinematics() returns and is rewritten only by the next iteration's kinematics(); M's packed storage is
// smaller than J for the raw and 2F85 size classes.  The targets, which must outlive kinematics(), live in qacc, which no phase here
// uses.  Shared-memory copies keep the frame and the targets out of registers (the float64 kernels would spill).  Every lane
// evaluates the error redundantly (a handful of 3-vectors); lanes share J's and the system's entries; lane 0 factors the <= 6 x 6
// system.
template <typename Real, typename D>
UR3E_HD IkResult<Real> ik_env(const DevModel<Real>& m, Arena<Real, D>& s, const IkTable<Real>& t, const Real* target_pos, const Real* target_quat,
                              const IkOpts<Real>& opt) {
  constexpr int NV = D::NV;
  static_assert(sizeof(s.u) >= sizeof(Real) * (7 * NV + 69) && NV >= 6, "IK scratch fits the arena's union u, the target qacc");
  Real* const J = reinterpret_cast<Real*>(&s.u);   // [r][nj]
  Real* const A = J + 6 * NV;                       // [ns][ns]: L below the diagonal after the factorisation
  Real* const B = A + 36;                           // right-hand side [ns]
  Real* const X = B + 6;                            // solution [ns]
  Real* const E = X + 6;                            // stacked error [r]
  Real* const Dg = E + 6;                           // pivots [ns]
  Real* const DQ = Dg + 6;                          // the step [nj]
  Real* const RO = DQ + NV;                         // the object's frame R(q) [9]
  Real* const TG = s.qacc;                          // target position [3], rotation vector [3]: kinematics() leaves qacc alone
  const QueryEntry<Real>& o = t.obj;
  const int nj = t.nj;
  const bool has_pos = target_pos != nullptr, has_rot = target_quat != nullptr;
  const int pr = has_pos ? 3 : 0, r = pr + (has_rot ? 3 : 0);
  const bool push = r <= nj;                        // solve the smaller SPD system: J J^T (r x r) or J^T J (nj x nj)
  const int ns = push ? r : nj;
  IF_LANE0 {
    if (has_pos) { TG[0] = target_pos[0]; TG[1] = target_pos[1]; TG[2] = target_pos[2]; }
    if (has_rot) ik_quat_rotvec(target_quat, TG + 3);
  }
  WARP_SYNC();
  int steps = 0, status = IK_MAX_STEPS_HIT;
  Real err_norm;
  for (;;) {
    kinematics(m, s);
    WARP_FOR(c, 9) RO[c] = entry_rot(s, o, c / 3, c - 3 * (c / 3));
    WARP_SYNC();
    Real p[3], ep[3] = {0, 0, 0}, er[3] = {0, 0, 0};
    entry_point(s, o, p);
    Real en = 0;
    if (has_pos) {
      for (int c = 0; c < 3; ++c) ep[c] = TG[c] - p[c];
      en = Num<Real>::sqrt(ep[0] * ep[0] + ep[1] * ep[1] + ep[2] * ep[2]);
    }
    if (has_rot) {
      rot_err(RO, TG + 3, er);
      en += opt.rot_weight * Num<Real>::sqrt(er[0] * er[0] + er[1] * er[1] + er[2] * er[2]);
    }
    err_norm = en;
    if (err_norm < opt.tol) { status = IK_CONVERGED; break; }
    if (steps == opt.max_steps) break;
    // J: the rows of the targets given, the selected joints' dofs as query_jac_env forms them
    WARP_FOR(i, r * nj) {
      const int row = i / nj, col = i - nj * row, d = t.j[col].dof;
      Real v;
      if (row < pr) { Real c3[3]; jac_col(m, s, d, p, o.body, c3); v = row == 0 ? c3[0] : (row == 1 ? c3[1] : c3[2]); }
      else v = ((m.body_dofmask[o.body] >> d) & 1u) ? s.cdof[d][row - pr] : Real(0);
      J[i] = v;
    }
    IF_LANE0 {
      if (has_pos) { E[0] = ep[0]; E[1] = ep[1]; E[2] = ep[2]; }
      if (has_rot) { E[pr] = er[0]; E[pr + 1] = er[1]; E[pr + 2] = er[2]; }
    }
    WARP_SYNC();
    const Real lam = err_norm > opt.reg_threshold ? opt.reg_strength : Real(0);
    WARP_FOR(i, ns * ns) {
      const int a = i / ns, b = i - ns * a;
      Real v = a == b ? lam : Real(0);
      if (push) { for (int k = 0; k < nj; ++k) v += J[a * nj + k] * J[b * nj + k]; }
      else { for (int k = 0; k < r; ++k) v += J[k * nj + a] * J[k * nj + b]; }
      A[i] = v;
    }
    WARP_FOR(i, ns) {
      Real v;
      if (push) v = E[i];
      else { v = 0; for (int k = 0; k < r; ++k) v += J[k * nj + i] * E[k]; }
      B[i] = v;
    }
    WARP_SYNC();
    IF_LANE0 {
      // LDL^T of the SPD system (serial: at most 6 x 6); with lambda = 0 a pivot at rounding level contributes zero
      Real dmax = 0;
      for (int k = 0; k < ns; ++k) dmax = rmax(dmax, A[k * ns + k]);
      const Real cut = lam > 0 ? Real(0) : ik_pivot_frac<Real>() * dmax;
      for (int c = 0; c < ns; ++c) {
        Real d = A[c * ns + c];
        for (int k = 0; k < c; ++k) d -= A[c * ns + k] * A[c * ns + k] * Dg[k];
        const bool keep = d > cut;
        Dg[c] = keep ? d : Real(0);
        const Real di = keep ? Real(1) / d : Real(0);
        for (int i = c + 1; i < ns; ++i) {
          Real v = A[i * ns + c];
          for (int k = 0; k < c; ++k) v -= A[i * ns + k] * A[c * ns + k] * Dg[k];
          A[i * ns + c] = v * di;
        }
      }
      for (int i = 0; i < ns; ++i) {
        Real v = B[i];
        for (int k = 0; k < i; ++k) v -= A[i * ns + k] * X[k];
        X[i] = v;
      }
      for (int i = 0; i < ns; ++i) X[i] = Dg[i] > 0 ? X[i] / Dg[i] : Real(0);
      for (int i = ns - 1; i >= 0; --i) {
        Real v = X[i];
        for (int k = i + 1; k < ns; ++k) v -= A[k * ns + i] * X[k];
        X[i] = v;
      }
    }
    WARP_SYNC();
    WARP_FOR(c, nj) {
      Real v;
      if (push) { v = 0; for (int k = 0; k < r; ++k) v += J[k * nj + c] * X[k]; }
      else v = X[c];
      DQ[c] = v;
    }
    WARP_SYNC();
    Real dn2 = 0;
    for (int c = 0; c < nj; ++c) dn2 += DQ[c] * DQ[c];
    const Real dn = Num<Real>::sqrt(dn2);
    if (err_norm / dn > opt.progress_thresh) { status = IK_NO_PROGRESS; break; }
    const Real scale = dn > opt.max_update_norm ? opt.max_update_norm / dn : Real(1);
    WARP_FOR(c, nj) {
      const IkJoint<Real>& jn = t.j[c];
      Real q = s.st.qpos[jn.qadr] + DQ[c] * scale;
      if (jn.limited) q = rmin(rmax(q, jn.lo), jn.hi);
      s.st.qpos[jn.qadr] = q;
    }
    WARP_SYNC();
    ++steps;
  }
  return IkResult<Real>{err_norm, steps, status};
}

}  // namespace ur3e
