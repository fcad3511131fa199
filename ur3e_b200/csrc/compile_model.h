// HostModel (MuJoCo-named arrays from mjcf.cpp) -> DevModel<Real> (kernel tables).
#pragma once
#include <cmath>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "dev_model.h"
#include "host_model.h"

namespace ur3e {

inline const char* const* tracked_site_names() {
  static const char* const n[MAXSITE] = {"tcp", "handle_site", "right_pad1_site", "left_pad1_site"};
  return n;
}

template <typename Real>
DevModel<Real> compile_model(const HostModel& h) {
  auto req = [](bool ok, const std::string& msg) { if (!ok) throw std::runtime_error("compile_model: " + msg); };
  DevModel<Real> m;
  std::memset(&m, 0, sizeof m);
  req(h.nbody <= MAXB && h.nv <= MAXV && h.nq <= MAXQ && h.nu <= MAXU && h.neq <= MAXEQ && h.nkey <= MAXKEY, "model exceeds the kernel's static limits");
  m.nq = h.nq; m.nv = h.nv; m.nu = h.nu; m.nbody = h.nbody; m.neq = h.neq; m.nkey = h.nkey;
  m.timestep = (Real)h.timestep; for (int k = 0; k < 3; ++k) m.gravity[k] = (Real)h.gravity[k];
  m.impratio = (Real)h.impratio; m.meaninertia = (Real)h.meaninertia;
  req(h.npair == 0 || h.cone_elliptic, "contacts require <option cone=\"elliptic\"> (the reference scenes' setting)");
  const auto &par = h.I("body_parentid"), &bja = h.I("body_jntadr"), &bjn = h.I("body_jntnum"), &jt = h.I("jnt_type"), &jq = h.I("jnt_qposadr"), &jd = h.I("jnt_dofadr"),
             &root = h.I("body_rootid"), &dpar = h.I("dof_parentid"), &dbody = h.I("dof_bodyid"), &djnt = h.I("dof_jntid"), &jlim = h.I("jnt_limited");
  auto cp = [](Real* dst, const std::vector<double>& src, int off, int n) { for (int k = 0; k < n; ++k) dst[k] = (Real)src[off + k]; };
  // unit quaternion (w, x, y, z) at src[off..off+4) -> row-major rotation matrix, evaluated in double
  auto cpmat = [](Real* dst, const std::vector<double>& src, int off) {
    double w = src[off], x = src[off + 1], y = src[off + 2], z = src[off + 3], n = std::sqrt(w * w + x * x + y * y + z * z);
    if (n < 1e-15) { w = 1; x = y = z = 0; } else { w /= n; x /= n; y /= n; z /= n; }
    const double R[9] = {w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y), 2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                         2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z};
    for (int k = 0; k < 9; ++k) dst[k] = (Real)R[k];
  };
  std::vector<int> lastdof(h.nbody, -1);
  int nlevel = 1;
  for (int b = 0; b < h.nbody; ++b) {
    m.body_parent[b] = par[b];
    m.body_level[b] = b == 0 ? 0 : m.body_level[par[b]] + 1;
    if (m.body_level[b] + 1 > nlevel) nlevel = m.body_level[b] + 1;
    m.body_root[b] = root[b];
    cp(m.body_pos[b], h.D("body_pos"), 3 * b, 3); cpmat(m.body_mat[b], h.D("body_quat"), 4 * b);
    cp(m.body_ipos[b], h.D("body_ipos"), 3 * b, 3); cpmat(m.body_imat[b], h.D("body_iquat"), 4 * b);
    m.body_mass[b] = (Real)h.D("body_mass")[b]; cp(m.body_inertia[b], h.D("body_inertia"), 3 * b, 3);
    cp(m.body_invw[b], h.D("body_invweight0"), 2 * b, 2);
    m.body_jkind[b] = JK_NONE; m.body_qadr[b] = -1; m.body_dadr[b] = -1;
    lastdof[b] = b == 0 ? -1 : lastdof[par[b]];
    m.body_dofmask[b] = b == 0 ? 0u : m.body_dofmask[par[b]];
    if (bjn[b] == 1) {
      int j = bja[b];
      m.body_jkind[b] = jt[j] == JNT_FREE ? JK_FREE : JK_HINGE;
      req(jt[j] == JNT_FREE || jt[j] == JNT_HINGE, "only hinge and free joints");
      req(jt[j] != JNT_FREE || par[b] == 0, "free joints must be children of the world");
      req(jt[j] != JNT_HINGE || root[b] != b, "a hinge body directly under the world needs a static base body above it");
      m.body_qadr[b] = jq[j]; m.body_dadr[b] = jd[j];
      cp(m.jnt_pos[b], h.D("jnt_pos"), 3 * j, 3);
      { const double* ax = &h.D("jnt_axis")[3 * j]; double n = std::sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]); if (n < 1e-15) n = 1;
        for (int k = 0; k < 3; ++k) m.jnt_axis[b][k] = (Real)(ax[k] / n); }   // unit axis (the kernel builds the joint rotation by Rodrigues' formula)
      m.jnt_q0[b] = (Real)h.D("qpos0")[jq[j]];
      int nd = jt[j] == JNT_FREE ? 6 : 1;
      for (int k = 0; k < nd; ++k) m.body_dofmask[b] |= 1u << (jd[j] + k);
      lastdof[b] = jd[j] + nd - 1;
    } else req(bjn[b] == 0, "at most one joint per body");
    m.body_lastdof[b] = lastdof[b];
  }
  m.nlevel = nlevel;
  { int k = 0; for (int l = 1; l < nlevel; ++l) { m.lev_start[l] = k; for (int b = 1; b < h.nbody; ++b) if (m.body_level[b] == l) m.lev_body[k++] = b; } m.lev_start[nlevel] = k; m.lev_start[0] = 0; }
  int nfl = 0, damp = 0;
  for (int d = 0; d < h.nv; ++d) {
    int j = djnt[d];
    m.dof_body[d] = dbody[d]; m.dof_parent[d] = dpar[d];
    int k = d - jd[j];
    if (jt[j] == JNT_FREE) { m.dof_free_k[d] = k; m.dof_qadr[d] = k < 3 ? jq[j] + k : jq[j] + 3; }
    else { m.dof_free_k[d] = -1; m.dof_qadr[d] = jq[j]; }
    m.dof_limited[d] = jt[j] == JNT_HINGE ? jlim[j] : 0;
    m.dof_armature[d] = (Real)h.D("dof_armature")[d]; m.dof_damping[d] = (Real)h.D("dof_damping")[d];
    m.dof_frictionloss[d] = (Real)h.D("dof_frictionloss")[d]; m.dof_invw[d] = (Real)h.D("dof_invweight0")[d];
    m.dof_stiffness[d] = jt[j] == JNT_HINGE ? (Real)h.D("jnt_stiffness")[j] : Real(0);
    m.dof_springref[d] = (Real)h.D("qpos_spring")[m.dof_qadr[d]];
    cp(m.dof_range[d], h.D("jnt_range"), 2 * j, 2); m.dof_margin[d] = (Real)h.D("jnt_margin")[j];
    cp(m.dof_lim_solref[d], h.D("jnt_solref"), 2 * j, 2); cp(m.dof_lim_solimp[d], h.D("jnt_solimp"), 5 * j, 5);
    cp(m.dof_fl_solref[d], h.D("dof_solref"), 2 * d, 2); cp(m.dof_fl_solimp[d], h.D("dof_solimp"), 5 * d, 5);
    m.dof_flrow[d] = -1;
    if (h.D("dof_frictionloss")[d] > 0) { m.dof_flrow[d] = nfl; m.fl_dof[nfl++] = d; }
    if (h.D("dof_damping")[d] > 0) damp = 1;
  }
  m.nfl = nfl; m.has_damping = damp;
  m.max_nanc = 0;
  for (int d = 0; d < h.nv; ++d) {
    int na = 0;
    for (int a = dpar[d]; a >= 0; a = dpar[a]) { req(na < MAXANC, "dof tree too deep"); m.dof_anc[d][na++] = a; }
    m.dof_nanc[d] = na; if (na > m.max_nanc) m.max_nanc = na;
  }
  int nM = 0;
  for (int i = 0; i < h.nv; ++i) for (int j = i; j >= 0; j = dpar[j]) { req(nM < MAXNM, "mass-matrix pattern too large"); m.M_i[nM] = i; m.M_j[nM] = j; ++nM; }
  m.nM = nM;
  { int e = 0; for (int a = 0; a <= h.nv; ++a) for (int b = 0; b <= a; ++b) m.tri_ab[e++] = (a << 8) | b; }

  // candidate pairs -> collidable geom list; planes shadowed by a higher parallel plane for the same box are dropped
  const auto &pg1 = h.I("pair_geom1"), &pg2 = h.I("pair_geom2"), &gt = h.I("geom_type"), &gb = h.I("geom_bodyid");
  const auto &gpos = h.D("geom_pos"), &gquat = h.D("geom_quat"), &gsize = h.D("geom_size");
  auto static_plane_height = [&](int g, double* nz) {
    // only handles planes on static, unrotated bodies (the reference scenes); returns z offset
    int b = gb[g]; double z = gpos[3 * g + 2];
    for (int a = b; a > 0; a = par[a]) z += h.D("body_pos")[3 * a + 2];
    *nz = (gquat[4 * g] > 0.999999 && h.I("body_weldid")[b] == 0) ? 1.0 : 0.0;
    return z;
  };
  std::vector<int> keep;
  for (int p = 0; p < h.npair; ++p) {
    bool drop = false;
    if (gt[pg1[p]] == GEOM_PLANE) {
      double nz, z = static_plane_height(pg1[p], &nz);
      if (nz == 1.0) for (int q = 0; q < h.npair && !drop; ++q) if (q != p && pg2[q] == pg2[p] && gt[pg1[q]] == GEOM_PLANE) {
        double nz2, z2 = static_plane_height(pg1[q], &nz2);
        const double* sz = &gsize[3 * pg2[p]]; double diag = 2 * std::sqrt(sz[0] * sz[0] + sz[1] * sz[1] + sz[2] * sz[2]);
        if (nz2 == 1.0 && z2 - z > diag) drop = true;
      }
    }
    if (!drop) keep.push_back(p);
  }
  std::vector<int> gmap(h.ngeom, -1); int ng = 0;
  auto use_geom = [&](int g) {
    if (gmap[g] >= 0) return gmap[g];
    req(ng < MAXG, "too many collidable geoms");
    int i = ng++; gmap[g] = i;
    m.geom_body[i] = gb[g]; m.geom_kind[i] = gt[g] == GEOM_PLANE ? GK_PLANE : GK_BOX; m.geom_src[i] = g;
    cp(m.geom_pos[i], gpos, 3 * g, 3); cpmat(m.geom_mat[i], gquat, 4 * g); cp(m.geom_size[i], gsize, 3 * g, 3);
    m.geom_rbound[i] = gt[g] == GEOM_PLANE ? Real(0) : (Real)std::sqrt(gsize[3 * g] * gsize[3 * g] + gsize[3 * g + 1] * gsize[3 * g + 1] + gsize[3 * g + 2] * gsize[3 * g + 2]);
    if (gt[g] == GEOM_PLANE) {
      // world normal of a plane: its body chain is static, so the frame is a model constant
      req(h.I("body_weldid")[gb[g]] == 0, "plane geoms must belong to static bodies");
      double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
      auto lmul = [&](const double* q4) {   // R <- Q R
        double w = q4[0], x = q4[1], y = q4[2], z = q4[3], n = std::sqrt(w * w + x * x + y * y + z * z); if (n < 1e-15) { w = 1; x = y = z = 0; n = 1; } w /= n; x /= n; y /= n; z /= n;
        const double Q[9] = {w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y), 2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                             2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z};
        double T[9]; for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) T[3 * r + c] = Q[3 * r] * R[c] + Q[3 * r + 1] * R[3 + c] + Q[3 * r + 2] * R[6 + c];
        for (int k = 0; k < 9; ++k) R[k] = T[k];
      };
      lmul(&gquat[4 * g]);
      for (int a = gb[g]; a > 0; a = par[a]) lmul(&h.D("body_quat")[4 * a]);
      for (int k = 0; k < 3; ++k) m.geom_nrm[i][k] = (Real)R[3 * k + 2];
    }
    return i;
  };
  req((int)keep.size() <= MAXPAIR, "too many candidate contact pairs");
  int np = 0;
  for (int p : keep) {
    m.pair_src_g1[np] = pg1[p]; m.pair_src_g2[np] = pg2[p];
    m.pair_g1[np] = use_geom(pg1[p]); m.pair_g2[np] = use_geom(pg2[p]);
    m.pair_friction[np][0] = (Real)h.D("pair_friction")[5 * p]; m.pair_friction[np][1] = (Real)h.D("pair_friction")[5 * p + 1];
    cp(m.pair_solref[np], h.D("pair_solref"), 2 * p, 2); cp(m.pair_solimp[np], h.D("pair_solimp"), 5 * p, 5);
    m.pair_margin[np] = (Real)h.D("pair_margin")[p]; m.pair_includemargin[np] = (Real)(h.D("pair_margin")[p] - h.D("pair_gap")[p]);
    m.pair_invw[np] = (Real)(h.D("geom_invweight0")[pg1[p]] + h.D("geom_invweight0")[pg2[p]]);
    m.pair_code[np] = m.pair_g1[np] | (m.pair_g2[np] << 8) | ((gt[pg1[p]] == GEOM_PLANE ? 1 : 0) << 16);
    m.pair_rsum[np] = m.geom_rbound[m.pair_g1[np]] + m.geom_rbound[m.pair_g2[np]] + m.pair_margin[np];
    ++np;
  }
  m.npair = np; m.ngeom = ng;

  for (int e = 0; e < h.neq; ++e) {
    int t = h.I("eq_type")[e], o1 = h.I("eq_obj1id")[e], o2 = h.I("eq_obj2id")[e];
    cp(m.eq_solref[e], h.D("eq_solref"), 2 * e, 2); cp(m.eq_solimp[e], h.D("eq_solimp"), 5 * e, 5);
    if (t == EQ_CONNECT) {
      m.eq_kind[e] = EK_CONNECT; m.eq_o1[e] = o1; m.eq_o2[e] = o2; cp(m.eq_data[e], h.D("eq_data"), 11 * e, 6);
      m.eq_invw[e] = (Real)h.D("eq_invweight0")[e];
    } else {
      req(t == EQ_JOINT, "equality type");
      req(jt[o1] == JNT_HINGE && (o2 < 0 || jt[o2] == JNT_HINGE), "joint equality needs hinge joints");
      m.eq_kind[e] = EK_JOINT; m.eq_o1[e] = jd[o1]; m.eq_o2[e] = o2 >= 0 ? jd[o2] : -1; cp(m.eq_data[e], h.D("eq_data"), 11 * e, 5);
      m.eq_invw[e] = (Real)h.D("eq_invweight0")[e];
    }
  }
  int ns = 0;
  for (int k = 0; k < MAXSITE; ++k) {
    int sid = h.name2id(OBJ_SITE, tracked_site_names()[k]);
    if (sid < 0) break;   // tracked sites are a prefix: tcp, handle_site, right_pad1_site, left_pad1_site
    m.site_body[ns] = h.I("site_bodyid")[sid]; cp(m.site_pos[ns], h.D("site_pos"), 3 * sid, 3); cpmat(m.site_mat[ns], h.D("site_quat"), 4 * sid); cp(m.site_size[ns], h.D("site_size"), 3 * sid, 3); ++ns;
  }
  // main.xml has all four; ur3e_2f85.xml lacks handle_site: track tcp only there unless the prefix continues
  m.nsite = ns;
  m.ntq = 0;
  if (h.arr.count("sensor_torque_site")) for (int sid : h.I("sensor_torque_site")) {
    if (m.ntq >= MAXTQ) break;
    m.tq_body[m.ntq] = h.I("site_bodyid")[sid]; cp(m.tq_pos[m.ntq], h.D("site_pos"), 3 * sid, 3); cpmat(m.tq_mat[m.ntq], h.D("site_quat"), 4 * sid); ++m.ntq;
  }
  for (int a = 0; a < h.nu; ++a) {
    double gear = h.D("actuator_gear")[a];
    m.act_dof[a][0] = m.act_dof[a][1] = -1;
    if (h.I("actuator_trntype")[a] == TRN_JOINT) {
      int j = h.I("actuator_trnid")[a]; req(jt[j] == JNT_HINGE, "actuated joint must be a hinge");
      m.act_dof[a][0] = jd[j]; m.act_coef[a][0] = (Real)gear;
    } else {
      int t = h.I("actuator_trnid")[a], adr = h.I("tendon_adr")[t], n = h.I("tendon_num")[t];
      req(n <= 2, "fixed tendon with more than two joints");
      for (int k = 0; k < n; ++k) { m.act_dof[a][k] = jd[h.I("wrap_jnt")[adr + k]]; m.act_coef[a][k] = (Real)(h.D("wrap_coef")[adr + k] * gear); }
    }
    m.act_gain[a] = (Real)h.D("actuator_gainprm")[a]; cp(m.act_bias[a], h.D("actuator_biasprm"), 3 * a, 3);
    cp(m.act_ctrlrange[a], h.D("actuator_ctrlrange"), 2 * a, 2); cp(m.act_forcerange[a], h.D("actuator_forcerange"), 2 * a, 2);
    m.act_ctrllimited[a] = h.I("actuator_ctrllimited")[a]; m.act_forcelimited[a] = h.I("actuator_forcelimited")[a];
  }
  for (int d = 0; d < h.nv; ++d) m.dof_nact[d] = 0;
  for (int a = 0; a < h.nu; ++a) for (int k = 0; k < 2; ++k) {
    const int d = m.act_dof[a][k];
    if (d < 0) continue;
    req(m.dof_nact[d] < 2, "more than two actuators on one dof");
    m.dof_act[d][m.dof_nact[d]] = a; m.dof_actcoef[d][m.dof_nact[d]] = m.act_coef[a][k]; ++m.dof_nact[d];
  }
  m.split = h.nv;
  if (h.nv > 0) {
    const int last_root = root[dbody[h.nv - 1]];
    int s0 = h.nv - 1;
    while (s0 > 0 && root[dbody[s0 - 1]] == last_root) --s0;
    if (s0 > 0) m.split = s0;   // dofs [s0, nv) form the last tree; dofs are numbered tree by tree, so nothing before s0 shares it
  }
  m.ndeq = 0; m.nej = 0;
  for (int e = 0; e < h.neq; ++e) { if (m.eq_kind[e] == EK_CONNECT) m.ndeq += 3; else m.nej += 1; }
  cp(m.qpos0, h.D("qpos0"), 0, h.nq);
  for (int k = 0; k < h.nkey; ++k) { cp(m.key_qpos[k], h.D("key_qpos"), k * h.nq, h.nq); cp(m.key_qvel[k], h.D("key_qvel"), k * h.nv, h.nv); }
  return m;
}

// The contact predicates of utils/gym_utils.py name bodies of the loaded model `h`: classify every collidable geom of `m` (compiled
// from h, or from h with its fixed bodies merged: geom ids are the same) by them (GeomFlag)
template <typename Real>
void set_geom_flags(const HostModel& h, DevModel<Real>& m) {
  const auto& par = h.I("body_parentid"); const auto& gbid = h.I("geom_bodyid");
  auto under = [&](int b, int root) { if (root < 0) return false; for (int a = b; a > 0; a = par[a]) if (a == root) return true; return false; };
  const int arm = h.name2id(OBJ_BODY, "robot_base"), grip = h.name2id(OBJ_BODY, "robotiq_base_mount"), table = h.name2id(OBJ_BODY, "table"),
            mug = h.name2id(OBJ_BODY, "fish"), lpad = h.name2id(OBJ_BODY, "left_pad"), rpad = h.name2id(OBJ_BODY, "right_pad");
  for (int i = 0; i < m.ngeom; ++i) {
    const int b = gbid[m.geom_src[i]];
    int f = 0;
    if (under(b, arm)) f |= GF_ARM;
    if (under(b, grip)) f |= GF_GRIPPER;
    if (b == table && table >= 0) f |= GF_TABLE;
    if (b == mug && mug >= 0) f |= GF_MUG;
    if (b == lpad && lpad >= 0) f |= GF_LPAD;
    if (b == rpad && rpad >= 0) f |= GF_RPAD;
    m.geom_flags[i] = f;
  }
}

}  // namespace ur3e
