// Kinematics queries: poses and velocities of a fixed list of objects (query_model.h) for one environment, evaluated at its
// stored state, and their Jacobians with the mass matrix and the bias forces.  Read-only: the caller loads qpos (and qvel when
// velocities or dynamics are wanted) into the arena's record copy; nothing is written back.  Like engine.cuh this file uses only
// warp_model.cuh constructs, so tests/hostcheck compiles it for the CPU.
//
// Semantics: MuJoCo's d.xpos / d.xipos / d.geom_xpos / d.site_xpos (and xmat), mj_objectVelocity, mj_jac*, mj_fullM and
// d.qfrc_bias after mj_forward at (qpos, qvel), i.e. after reset / set_state.  After mj_step MuJoCo's arrays still hold the last
// substep's pre-integration values (SURVEY F9); a query after a step is one substep newer than those.
#pragma once
#include "engine.cuh"
#include "query_model.h"

namespace ur3e {

// Arena size class of the query: the generic class's bodies, dofs and geoms with no contact or constraint-row storage (the
// query runs kinematics only, so it fits more environments per SM than the step)
template <typename D> using QueryDims = Dims<D::NB, D::NV, D::NQ, D::NU, D::NG, D::NPAIR, 0, 0, D::SPLIT>;

// World frame of a compiled entry after kinematics(): position xpos[a] + R_a lpos, and element (r, c) of R_a lmat
template <typename Real, typename D>
UR3E_HD void entry_point(const Arena<Real, D>& s, const QueryEntry<Real>& o, Real* p) {
  Real v[3]; mat_vec3(v, s.fr.k.xmat[o.body], o.lpos);
  for (int c = 0; c < 3; ++c) p[c] = s.xpos[o.body][c] + v[c];
}
template <typename Real, typename D>
UR3E_HD Real entry_rot(const Arena<Real, D>& s, const QueryEntry<Real>& o, int r, int c) {
  const Real* Ra = s.fr.k.xmat[o.body] + 3 * r; const Real* L = o.lmat + c;
  return Ra[0] * L[0] + Ra[1] * L[3] + Ra[2] * L[6];
}

// pos [k][3], mat [k][9] (row-major), vel [k][6] = [rot(3), lin(3)] of this environment; any may be null.  local != 0: velocities
// in the object's frame (mj_objectVelocity's flg_local).
template <typename Real, typename D>
UR3E_HD void query_env(const DevModel<Real>& m, Arena<Real, D>& s, const QueryEntry<Real>* q, int k, Real* pos, Real* mat, Real* vel, int local) {
  kinematics(m, s);
  auto& cvel = s.u.dyn.cvel;
  if (vel) {
    // body velocities about the tree reference point: the dof-chain sum of dynamics()
    WARP_FOR(b, nb_<D>(m)) {
      Real cv[6] = {0, 0, 0, 0, 0, 0};
      if (b > 0) for (int d = m.body_lastdof[b]; d >= 0; d = m.dof_parent[d]) { Real qd = s.st.qvel[d]; for (int c = 0; c < 6; ++c) cv[c] += s.cdof[d][c] * qd; }
      for (int c = 0; c < 6; ++c) cvel[b][c] = cv[c];
    }
    WARP_SYNC();
  }
  const auto& xmat = s.fr.k.xmat;
  // world position of object j: xpos[a] + R_a lpos
  auto point = [&](const QueryEntry<Real>& o, Real* p) { entry_point(s, o, p); };
  if (pos) {
    WARP_FOR(i, 3 * k) {
      const int j = i / 3, r = i - 3 * j;
      Real p[3]; point(q[j], p);
      pos[i] = r == 0 ? p[0] : (r == 1 ? p[1] : p[2]);   // selects, not a dynamically indexed (local-memory) array
    }
  }
  if (mat) {
    WARP_FOR(i, 9 * k) {
      const int j = i / 9, e = i - 9 * j, r = e / 3, c = e - 3 * r;
      const Real* Ra = xmat[q[j].body] + 3 * r; const Real* L = q[j].lmat + c;
      mat[i] = Ra[0] * L[0] + Ra[1] * L[3] + Ra[2] * L[6];
    }
  }
  if (vel) {
    // mj_objectVelocity: [w, v_ref + w x (p - ref)], ref = xpos of the tree root; flg_local rotates both by (R_a lmat)^T
    WARP_FOR(i, 6 * k) {
      const int j = i / 6, e = i - 6 * j, half = e / 3, r = e - 3 * half;
      const QueryEntry<Real>& o = q[j];
      const Real* cv = cvel[o.body];
      Real w[3];
      if (half == 0) { w[0] = cv[0]; w[1] = cv[1]; w[2] = cv[2]; }
      else {
        Real p[3], t[3]; point(o, p);
        const Real* ref = s.xpos[o.root];
        const Real off[3] = {p[0] - ref[0], p[1] - ref[1], p[2] - ref[2]};
        cross3(t, cv, off);
        for (int c = 0; c < 3; ++c) w[c] = cv[3 + c] + t[c];
      }
      if (local) {
        const Real* Ra = xmat[o.body];
        Real a[3];   // R_a^T w
        for (int c = 0; c < 3; ++c) a[c] = Ra[c] * w[0] + Ra[3 + c] * w[1] + Ra[6 + c] * w[2];
        vel[i] = o.lmat[r] * a[0] + o.lmat[3 + r] * a[1] + o.lmat[6 + r] * a[2];
      } else {
        vel[i] = r == 0 ? w[0] : (r == 1 ? w[1] : w[2]);
      }
    }
  }
}

// Arguments of a Jacobian / mass-matrix call (ur3e_batch_query_jac): query `id` of `nquery` compiled ones, or -1 for none, with
// `jac` = jacp or jacr requested and `any` = some output requested.  Returns "" when valid, else the reason the call is rejected.
inline std::string query_jac_check(int id, int nquery, bool jac, bool any) {
  if (id < -1 || id >= nquery) return "unknown query id " + std::to_string(id);
  if (!any) return "all outputs are null";
  if (id == -1 && jac) return "jacp / jacr need a query's objects (query_id = -1 has none)";
  return "";
}

// mj_jacSite / mj_jacBody / mj_jacBodyCom / mj_jacGeom of the k objects, at each object's world point xpos[a] + R_a lpos (the
// site, body frame, inertial frame or geom of query_model.h's entry): jacp, jacr [k][3][nv] (MuJoCo's row-major (3, nv) per
// object); mj_fullM: M [nv][nv], dense and symmetric; d.qfrc_bias [nv].  Any output may be null; q may be null when k = 0.  The
// caller loads qpos, and qvel when M or qfrc_bias is wanted.  M and qfrc_bias are the step's own dynamics() (CRBA with armature,
// RNE); that pass also forms the actuator forces, so ctrl is zeroed first rather than left as uninitialised shared memory.
template <typename Real, typename D>
UR3E_HD void query_jac_env(const DevModel<Real>& m, Arena<Real, D>& s, const QueryEntry<Real>* q, int k, Real* jacp, Real* jacr, Real* M, Real* bias) {
  kinematics(m, s);
  if (M || bias) {
    WARP_FOR(a, nu_<D>(m)) s.ctrl[a] = 0;
    WARP_SYNC();
    dynamics(m, s);
  }
  const int nv = nv_<D>(m);
  if (jacp || jacr) {
    const auto& xmat = s.fr.k.xmat;
    const int per = 3 * nv;
    WARP_FOR(i, k * per) {
      const int j = i / per, e = i - per * j, r = e / nv, d = e - nv * r;
      const QueryEntry<Real>& o = q[j];
      if (jacp) {
        Real v[3], p[3], col[3];
        mat_vec3(v, xmat[o.body], o.lpos);
        for (int c = 0; c < 3; ++c) p[c] = s.xpos[o.body][c] + v[c];
        jac_col(m, s, d, p, o.body, col);
        jacp[i] = r == 0 ? col[0] : (r == 1 ? col[1] : col[2]);   // selects, not a dynamically indexed (local-memory) array
      }
      if (jacr) jacr[i] = ((m.body_dofmask[o.body] >> d) & 1u) ? s.cdof[d][r] : Real(0);
    }
  }
  if (M) {
    WARP_FOR(i, nv * nv) {
      const int r = i / nv, c = i - nv * r, hi = r > c ? r : c, lo = r > c ? c : r;
      M[i] = s.M[hi * (hi + 1) / 2 + lo];
    }
  }
  if (bias) { WARP_FOR(i, nv) bias[i] = s.qfrc_bias[i]; }
}

}  // namespace ur3e
