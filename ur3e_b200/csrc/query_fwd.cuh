// Forward-dynamics queries: one mj_forward of one environment at its stored state, off the step path, exposing what the step
// computes and discards -- the contact list (MuJoCo's d.contact), the contact forces (mj_contactForce), d.qacc,
// d.qfrc_constraint and d.sensordata.  Read-only: the caller loads the environment's record into the arena; nothing is written
// back.  Like engine.cuh this file uses only warp_model.cuh constructs, so tests/hostcheck compiles it for the CPU.
//
// Semantics: MuJoCo's values after mj_forward at (qpos, qvel, qacc_warmstart) with the given ctrl, i.e. after reset / set_state.
// After mj_step MuJoCo's d.contact, d.efc_force and d.sensordata still hold the last substep's pre-integration values (SURVEY F9);
// a query after a step is one substep newer than those and describes the same state the kinematics queries see.
#pragma once
#include <string>

#include "env.cuh"

namespace ur3e {

// Outputs of one environment; any may be null.  C = contacts per environment (D::MAXCON, 0 without contacts).
template <typename Real>
struct FwdOut {
  Real* qacc;              // [nv]
  Real* qfrc_constraint;   // [nv]
  int32_t* info;           // [4]: ncon, nefc, solver iterations, overflow bits (1 contacts / narrow-phase slots, 2 rows)
  int32_t* contact_geom;   // [C][2]: geom1, geom2 of the loaded model; -1 past ncon
  Real* contact_dist;      // [C]
  Real* contact_pos;       // [C][3]
  Real* contact_frame;     // [C][9]: row 0 the normal (geom1 -> geom2), rows 1-2 the tangents
  Real* contact_force;     // [C][6]: mj_contactForce in the contact frame, [fn, ft1, ft2, 0, 0, 0] (elliptic cone, condim 3)
  int32_t* flags;          // [1]: contact_bits() over all ncon contacts (see forward_query_env)
  Real* sensordata;        // [NSENSOR]: the step's logging record
};

// Arguments of a forward query (ur3e_batch_forward): `out` given, `con` = some contact_* output requested, `any` = some output
// requested, `ncmax` = contacts per environment.  Returns "" when valid, else the reason the call is rejected.
inline std::string forward_query_check(bool out, bool con, bool any, int ncmax) {
  if (!out) return "out is null";
  if (!any) return "all outputs are null";
  if (con && ncmax == 0) return "contact outputs need a model with contact pairs (max_contacts = 0)";
  return "";
}

// The contact list (d.contact[k].geom1 / geom2, dist, pos, frame) of the `ncon` contacts collision() found, padded to C = D::MAXCON
// entries with geom -1 and zeros; any output may be null.  Call it right after collision(), while every contact frame is intact (the
// solver keeps its cone Hessians in the tangents' storage).  Shared by the forward and the inverse query.
template <typename Real, typename D>
UR3E_HD void contact_list_out(const DevModel<Real>& m, const Arena<Real, D>& s, int ncon, int32_t* geom, Real* dist, Real* pos, Real* frame) {
  constexpr int C = D::MAXCON;
  if (geom) {
    WARP_FOR(i, 2 * C) {
      const int c = i >> 1;
      geom[i] = c < ncon ? ((i & 1) ? m.pair_src_g2[s.con_pair[c]] : m.pair_src_g1[s.con_pair[c]]) : -1;
    }
  }
  if (dist) { WARP_FOR(c, C) dist[c] = c < ncon ? s.con_dist[c] : Real(0); }
  if (pos) { WARP_FOR(i, 3 * C) { const int c = i / 3; pos[i] = c < ncon ? s.con_pos[c][i - 3 * c] : Real(0); } }
  if (frame) { WARP_FOR(i, 9 * C) { const int c = i / 9; frame[i] = c < ncon ? s.cu.frame[c][i - 9 * c] : Real(0); } }
}

// mj_contactForce of every contact from the rows' efc_force, [C][6]: [fn, ft1, ft2, 0, 0, 0] in the contact frame.  s.ncon is the
// count make_constraint() left, the contacts it found rows for (con_row[c] is the normal row, the two tangent rows follow); a contact
// past it, cut on a row overflow, and the padding report zero.
template <typename Real, typename D>
UR3E_HD void contact_force_out(const Arena<Real, D>& s, Real* out) {
  WARP_FOR(i, 6 * D::MAXCON) {
    const int c = i / 6, k = i - 6 * c;
    out[i] = (c < s.ncon && k < 3) ? s.efc_force[s.con_row[c] + k] : Real(0);
  }
}

// The full pass runs when an output needs dynamics (qacc, qfrc_constraint, contact_force, sensordata); otherwise the
// contacts-only pass runs (contact geometry, info, flags): kinematics and collision alone, since collision reads nothing else.
template <typename Real>
UR3E_HD bool forward_query_full(const FwdOut<Real>& o) { return o.qacc || o.qfrc_constraint || o.contact_force || o.sensordata; }

// mj_forward of one environment.  The caller has loaded the whole record (qpos, qvel and the warm start qacc_ws, which the solver
// starts from as MuJoCo's does from d.qacc_warmstart).  ctrl [nu] or null (zero).
//
// Full pass: the phases of forward(m, s, opt, true) in its order, with no block barriers (aligned = false), so that the contact
// count the collision kept is known before make_constraint() shortens the list on a row overflow; contacts without rows then
// report zero force.  Contacts-only pass: kinematics() and collision(); info's nefc and iterations are 0 and the row bit is never set.
// The contact geometry and flags are written right after collision() in both passes, while every contact frame is intact (the
// solver keeps its cone Hessians in the tangents' storage): the two passes give identical geometry.  The flags therefore cover every
// contact of the list, as the reference's predicates do over d.contact; on a row overflow the step's contact_flags() runs after
// make_constraint() has cut the list to the contacts with rows, so there the step's bits can miss a contact these include.
template <typename Real, typename D>
UR3E_HD void forward_query_env(const DevModel<Real>& m, Arena<Real, D>& s, const SolverOpts<Real>& opt, const Real* ctrl, const FwdOut<Real>& o) {
  constexpr int C = D::HAS_CONTACT ? D::MAXCON : 0;
  const bool full = forward_query_full(o);
  IF_LANE0 { s.overflow = 0; s.ncon = 0; s.nefc = 0; s.solver_iter = 0; s.cap_con = D::MAXCON; s.cap_efc = D::MAXEFC; }
  WARP_FOR(a, nu_<D>(m)) s.ctrl[a] = ctrl ? ctrl[a] : Real(0);
  WARP_SYNC();
  kinematics(m, s);
  if (full) dynamics(m, s);
  collision(m, s);
  const int ncon = s.ncon;
  if constexpr (C > 0) contact_list_out(m, s, ncon, o.contact_geom, o.contact_dist, o.contact_pos, o.contact_frame);
  if (o.flags) {
    const int f = contact_bits(m, s);
    IF_LANE0 o.flags[0] = f;
  }
  WARP_SYNC();
  if (full) {
    make_constraint(m, s);
    solve(m, s, opt);
  }
  if constexpr (C > 0) {
    if (o.contact_force) contact_force_out(s, o.contact_force);
  }
  if (o.qacc) { WARP_FOR(d, nv_<D>(m)) o.qacc[d] = s.qacc[d]; }
  if (o.qfrc_constraint) { WARP_FOR(d, nv_<D>(m)) o.qfrc_constraint[d] = s.qfrc_constraint[d]; }
  if (o.info) {
    IF_LANE0 { o.info[0] = ncon; o.info[1] = s.nefc; o.info[2] = s.solver_iter; o.info[3] = s.overflow; }
  }
  WARP_SYNC();
  if (o.sensordata) sensors_cold(m, s, o.sensordata);   // rebuilds the body frames the Newton matrix overwrote
}

}  // namespace ur3e
