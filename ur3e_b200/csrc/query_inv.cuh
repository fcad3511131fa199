// Inverse-dynamics queries: MuJoCo's mj_inverse of one state, off the step path.  Given (qpos, qvel) and an acceleration, the
// generalised force that produces it (qfrc_inverse, actuation excluded), and the constraint and contact forces the soft-constraint
// model implies at that acceleration (mj_invConstraint).  Read-only: the caller loads qpos and qvel into the arena; nothing is written
// back.  Like engine.cuh this file uses only warp_model.cuh constructs, so tests/hostcheck compiles it for the CPU.
//
// Semantics (mujoco 3.3.3 mj_inverse, soft constraints, Euler integrator, no sensors):
//   a = M^-1 (M + h diag(damping)) qacc     with `discrete` (mjENBL_INVDISCRETE, mj_discreteAcc): qacc is the acceleration the step's
//                                           implicit-damping Euler update applied, (qvel_next - qvel) / timestep of one mj_step
//   a = qacc                                without (MuJoCo's default), or when the model has no damping
//   efc_force = the constraint law at jar = J a - aref       (constraint_update, the per-row law the Newton solver minimises)
//   qfrc_constraint = J^T efc_force
//   qfrc_inverse = M a + qfrc_bias - qfrc_passive - qfrc_constraint,   qfrc_passive = -damping qvel - stiffness (q - springref)
#pragma once
#include <string>

#include "query_fwd.cuh"

namespace ur3e {

// Outputs of one state; any may be null.  C = contacts per state (D::MAXCON, 0 without contacts).
template <typename Real>
struct InvOut {
  Real* qfrc_inverse;      // [nv]
  Real* qfrc_constraint;   // [nv]
  int32_t* info;           // [3]: ncon, nefc, overflow bits (1 contacts / narrow-phase slots, 2 rows)
  int32_t* contact_geom;   // [C][2]: geom1, geom2 of the loaded model; -1 past ncon
  Real* contact_force;     // [C][6]: mj_contactForce at the given acceleration, [fn, ft1, ft2, 0, 0, 0] in the contact frame
};

// Arguments of an inverse query (ur3e_batch_inverse): which of the given states' qpos / qvel are given (neither = the stored state of
// the batch's n environments), m states, qacc given, `out` given, `con` = some contact output requested, `any` = some output requested,
// `ncmax` = contacts per state.  Returns "" when valid, else the reason the call is rejected.
inline std::string inverse_query_check(bool qpos, bool qvel, long long m, long long n, bool qacc, bool out, bool con, bool any, int ncmax) {
  if (qpos != qvel) return qpos ? "qpos is given without qvel" : "qvel is given without qpos";
  if (m < 1 || m > 2147483647LL) return "m=" + std::to_string(m) + " states (1 .. 2^31 - 1)";
  if (!qpos && m != n) return "m=" + std::to_string(m) + " for the stored state of n=" + std::to_string(n) + " environments (m must equal n)";
  if (!qacc) return "qacc is null";
  if (!out) return "out is null";
  if (!any) return "all outputs are null";
  if (con && ncmax == 0) return "contact outputs need a model with contact pairs (max_contacts = 0)";
  return "";
}

// mj_inverse of one state.  The caller has loaded qpos and qvel into s.st; qacc [nv].
//
// The phases of forward() up to the rows, then the non-iterative inverse in place of the solver.  Aliasing (DESIGN §3): collision()
// overwrites the dynamics buffers with its staging rows and make_constraint() those with the Jacobian, but M and qfrc_bias have their
// own storage; the contact geometry is written right after collision(); the body frames are read last by make_constraint() (connect
// equalities), so only then does the M solve of the discrete convention take their storage (H); constraint_update() without cone
// Hessians leaves a marker in each contact's tangent storage, which nothing here reads afterwards.
template <typename Real, typename D>
UR3E_HD void inverse_query_env(const DevModel<Real>& m, Arena<Real, D>& s, bool discrete, const Real* qacc, const InvOut<Real>& o) {
  constexpr int C = D::HAS_CONTACT ? D::MAXCON : 0;
  const int nv = nv_<D>(m);
  IF_LANE0 { s.overflow = 0; s.ncon = 0; s.nefc = 0; s.solver_iter = 0; s.cap_con = D::MAXCON; s.cap_efc = D::MAXEFC; }
  WARP_FOR(a, nu_<D>(m)) s.ctrl[a] = Real(0);   // dynamics() also forms the actuator forces, which qfrc_inverse excludes
  WARP_FOR(d, nv) s.qacc[d] = qacc[d];
  WARP_SYNC();
  kinematics(m, s);
  dynamics(m, s);
  collision(m, s);
  const int ncon = s.ncon;
  if constexpr (C > 0) {
    if (o.contact_geom) contact_list_out(m, s, ncon, o.contact_geom, (Real*)nullptr, (Real*)nullptr, (Real*)nullptr);
  }
  WARP_SYNC();
  make_constraint(m, s);
  // the passive forces as dynamics() forms them (its qfrc_smooth also holds the actuator forces, which a general actuator's bias terms
  // make nonzero even at ctrl = 0): qfrc_smooth is dead past this point and holds them
  WARP_FOR(d, nv) {
    Real f = -m.dof_damping[d] * s.st.qvel[d];
    if (m.dof_free_k[d] < 0) f -= m.dof_stiffness[d] * (s.st.qpos[m.dof_qadr[d]] - m.dof_springref[d]);
    s.qfrc_smooth[d] = f;
  }
  if (discrete && has_damping_<D>(m)) {
    // mj_discreteAcc: a = M^-1 (M + h diag(damping)) qacc, the exact inverse of euler()'s implicit-damping solve
    const Real h = m.timestep;
    Real* A = s.fr.n.H;
    WARP_FOR(e, nv * (nv + 1) / 2) A[e] = s.M[e];
    WARP_FOR(d, nv) s.search[d] = sym_matvec_row_n<Real, D::NV>(s.M, s.qacc, d, nv) + h * m.dof_damping[d] * s.qacc[d];
    WARP_SYNC();
    tree_ldl_solve(m, s, s.search);
    WARP_FOR(d, nv) s.qacc[d] = s.search[d];
    WARP_SYNC();
  }
  // mj_invConstraint: the row law at jar = J a - aref
  WARP_FOR(r, s.nefc) s.efc_jar[r] = row_dot(m, s, r, s.qacc) - s.efc_aref[r];
  WARP_SYNC();
  constraint_update(m, s, false);
  WARP_FOR(d, nv) {
    const Real fc = col_dot(m, s, d, s.efc_force);
    s.qfrc_constraint[d] = fc;
    s.Ma[d] = sym_matvec_row_n<Real, D::NV>(s.M, s.qacc, d, nv) + s.qfrc_bias[d] - s.qfrc_smooth[d] - fc;
  }
  WARP_SYNC();
  if constexpr (C > 0) {
    if (o.contact_force) contact_force_out(s, o.contact_force);
  }
  if (o.qfrc_inverse) { WARP_FOR(d, nv) o.qfrc_inverse[d] = s.Ma[d]; }
  if (o.qfrc_constraint) { WARP_FOR(d, nv) o.qfrc_constraint[d] = s.qfrc_constraint[d]; }
  if (o.info) {
    IF_LANE0 { o.info[0] = ncon; o.info[1] = s.nefc; o.info[2] = s.overflow; }
  }
}

}  // namespace ur3e
