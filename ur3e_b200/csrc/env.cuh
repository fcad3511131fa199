// Environment layer fused around the physics substeps: controller, observation, reward, termination,
// truncation and in-kernel auto-reset (reference gymnasium_env/envs/ur3e_env2.py, ur3e_env.py,
// imitation_env_*.py; controller/controller_func.py; utils/gym_utils.py).  Same warp model as engine.cuh.
#pragma once
#include "engine.cuh"

namespace ur3e {

// ---------------------------------------------------------------- counter-based RNG (Philox4x32-10)
UR3E_HD void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
template <typename Real> UR3E_HD Real u01(uint32_t x) { return (Real)((double)x * (1.0 / 4294967296.0)); }

// ---------------------------------------------------------------- controllers
// rotvec of R_target * R_site^T  (controller_func.py:30-48, scipy conventions: SURVEY App. C)
template <typename Real> UR3E_HD void rot_err(const Real* xmat, const Real* rv, Real* err) {
  Real ang = Num<Real>::sqrt(dot3(rv, rv)), q[4] = {1, 0, 0, 0};
  if (ang > Real(1e-30)) { Real sn, cs; Num<Real>::sincos(ang * Real(0.5), &sn, &cs); sn /= ang; q[0] = cs; q[1] = rv[0] * sn; q[2] = rv[1] * sn; q[3] = rv[2] * sn; }
  Real Rt[9], E[9]; quat2mat(Rt, q);
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) E[3 * i + j] = Rt[3 * i] * xmat[3 * j] + Rt[3 * i + 1] * xmat[3 * j + 1] + Rt[3 * i + 2] * xmat[3 * j + 2];
  Real tr = E[0] + E[4] + E[8], w, x, y, z;
  if (tr > 0) { Real s = Num<Real>::sqrt(tr + 1) * 2; w = Real(0.25) * s; x = (E[7] - E[5]) / s; y = (E[2] - E[6]) / s; z = (E[3] - E[1]) / s; }
  else if (E[0] > E[4] && E[0] > E[8]) { Real s = Num<Real>::sqrt(1 + E[0] - E[4] - E[8]) * 2; w = (E[7] - E[5]) / s; x = Real(0.25) * s; y = (E[1] + E[3]) / s; z = (E[2] + E[6]) / s; }
  else if (E[4] > E[8]) { Real s = Num<Real>::sqrt(1 + E[4] - E[0] - E[8]) * 2; w = (E[2] - E[6]) / s; x = (E[1] + E[3]) / s; y = Real(0.25) * s; z = (E[5] + E[7]) / s; }
  else { Real s = Num<Real>::sqrt(1 + E[8] - E[0] - E[4]) * 2; w = (E[3] - E[1]) / s; x = (E[2] + E[6]) / s; y = (E[5] + E[7]) / s; z = Real(0.25) * s; }
  Real nq = Num<Real>::sqrt(w * w + x * x + y * y + z * z); w /= nq; x /= nq; y /= nq; z /= nq;
  if (w < 0) { w = -w; x = -x; y = -y; z = -z; }
  Real sn = Num<Real>::sqrt(x * x + y * y + z * z), a = 2 * Num<Real>::atan2(sn, w);
  Real k = sn < Real(1e-12) ? Real(2) : a / sn;
  err[0] = k * x; err[1] = k * y; err[2] = k * z;
}

// cache layout: [0:3) tcp pos, [3:12) tcp mat, [12:48) J (6 rows: px,py,pz,rx,ry,rz) x 6 arm dofs, [48:54) qfrc_bias[:6]
template <typename Real, typename D>
UR3E_HD void update_cache(const DevModel<Real>& m, const EnvCfg<Real>& c, Arena<Real, D>& s) {
  int site = c.site_tcp;
  if (site < 0) return;
  int b = m.site_body[site];
  WARP_FOR(i, CACHE_SIZE) {
    Real v;
    if (i < 3) v = s.site_xpos[site][i];
    else if (i < 12) v = s.site_xmat[0][i - 3];   // the tcp is the first tracked site
    else if (i < 48) {
      int r = (i - 12) / 6, k = (i - 12) - 6 * r;
      if (r < 3) { Real col[3]; jac_col(m, s, k, s.site_xpos[site], b, col); v = col[r]; }
      else v = ((m.body_dofmask[b] >> k) & 1u) ? s.cdof[k][r - 3] : Real(0);
    } else v = s.qfrc_bias[i - 48];
    s.st.cache[i] = v;
  }
  WARP_SYNC();
}

template <typename Real, typename D>
UR3E_HD void pid_task(const DevModel<Real>& m, const EnvCfg<Real>& c, Arena<Real, D>& s, const Real* traj) {
  // controller_func.py:68-117: tau = J^T [Kp e - Kd J qvel] + qfrc_bias ; no clipping, no integral term (SURVEY F10)
  const Real* ch = s.st.cache;
  Real e[6], F[6];
  for (int k = 0; k < 3; ++k) e[k] = traj[k] - ch[k];
  rot_err(ch + 3, traj + 3, e + 3);
  for (int r = 0; r < 6; ++r) {
    Real v = 0; for (int k = 0; k < 6; ++k) v += ch[12 + 6 * r + k] * s.st.qvel[k];
    int g = r < 3 ? r : 3 + r;   // kp_pos[0:3] kd_pos[3:6] kp_rot[6:9] kd_rot[9:12]
    F[r] = c.gains[g] * e[r] - c.gains[g + 3] * v;
  }
  WARP_FOR(k, 6) { Real v = ch[48 + k]; for (int r = 0; r < 6; ++r) v += ch[12 + 6 * r + k] * F[r]; s.ctrl[k] = v; }
  IF_LANE0 s.ctrl[nu_<D>(m) - 1] = traj[6] * m.act_ctrlrange[nu_<D>(m) - 1][1];   // grip_ctrl, controller_func.py:183-186
}

template <typename Real, typename D>
UR3E_HD void controller(const DevModel<Real>& m, const EnvCfg<Real>& c, Arena<Real, D>& s, const Real* act) {
  switch (c.ctrl_mode) {
    case CTRL_RAW: { WARP_FOR(a, nu_<D>(m)) s.ctrl[a] = act[a]; break; }
    case CTRL_PD_JOINT: {
      // controller_func.py:128-167 with move_j.get_joint_delta (move_j.py:30-38)
      WARP_FOR(i, 6) {
        Real q = s.st.qpos[i], tq = q + (act[i] - q);
        tq = rmin(rmax(tq, m.dof_range[i][0]), m.dof_range[i][1]);
        Real u = c.gains[i] * (tq - q) + c.gains[6 + i] * -s.st.qvel[i];
        s.ctrl[i] = rmin(rmax(u, m.act_ctrlrange[i][0]), m.act_ctrlrange[i][1]);
      }
      if (nu_<D>(m) > 6) { IF_LANE0 s.ctrl[nu_<D>(m) - 1] = act[6] * m.act_ctrlrange[nu_<D>(m) - 1][1]; }
      break;
    }
    case CTRL_PID_TASK: { Real traj[7]; for (int k = 0; k < 7; ++k) traj[k] = act[k]; pid_task(m, c, s, traj); break; }
    case CTRL_PID_TASK_ENV: {
      // ur3e_env2.py:72-75: traj = [a0,a1,a2, tool rotvec, a3]
      Real traj[7] = {act[0], act[1], act[2], c.tool_rotvec[0], c.tool_rotvec[1], c.tool_rotvec[2], act[3]};
      pid_task(m, c, s, traj); break;
    }
    case CTRL_PINV: {
      // move_l.py:15-78: dtheta = pinv(Jp[:, :6]) e_p and pinv(Jr[:, :6]) e_r (pinv = J^T (J J^T)^-1 for the full-row-rank 3 x 6
      // blocks; numpy's SVD cut-off only differs at exact singularities), each through pd_joint_ctrl, summed; grip appended
      const Real* ch = s.st.cache;
      Real e[6], y[6];
      for (int k = 0; k < 3; ++k) e[k] = act[k] - ch[k];
      { Real rv[3] = {act[3], act[4], act[5]}; rot_err(ch + 3, rv, e + 3); }
      for (int blk = 0; blk < 2; ++blk) {
        const Real* J = ch + 12 + 18 * blk;   // 3 rows x 6 arm dofs
        Real A[6];                            // J J^T, symmetric: 00 01 02 11 12 22
        int idx = 0;
        for (int r = 0; r < 3; ++r) for (int c2 = r; c2 < 3; ++c2) { Real v = 0; for (int k = 0; k < 6; ++k) v += J[6 * r + k] * J[6 * c2 + k]; A[idx++] = v; }
        const Real c00 = A[3] * A[5] - A[4] * A[4], c01 = A[2] * A[4] - A[1] * A[5], c02 = A[1] * A[4] - A[2] * A[3];
        const Real det = A[0] * c00 + A[1] * c01 + A[2] * c02, id = Real(1) / det;
        const Real c11 = A[0] * A[5] - A[2] * A[2], c12 = A[1] * A[2] - A[0] * A[4], c22 = A[0] * A[3] - A[1] * A[1];
        const Real* b = e + 3 * blk;
        y[3 * blk + 0] = (c00 * b[0] + c01 * b[1] + c02 * b[2]) * id;
        y[3 * blk + 1] = (c01 * b[0] + c11 * b[1] + c12 * b[2]) * id;
        y[3 * blk + 2] = (c02 * b[0] + c12 * b[1] + c22 * b[2]) * id;
      }
      WARP_FOR(i, 6) {
        const Real q = s.st.qpos[i], qd = s.st.qvel[i];
        Real u = 0;
        for (int blk = 0; blk < 2; ++blk) {
          const Real* J = ch + 12 + 18 * blk;
          const Real dth = J[i] * y[3 * blk] + J[6 + i] * y[3 * blk + 1] + J[12 + i] * y[3 * blk + 2];
          Real tq = rmin(rmax(q + dth, m.dof_range[i][0]), m.dof_range[i][1]);
          Real ub = c.gains[12 * blk + i] * (tq - q) + c.gains[12 * blk + 6 + i] * -qd;
          u += rmin(rmax(ub, m.act_ctrlrange[i][0]), m.act_ctrlrange[i][1]);
        }
        s.ctrl[i] = u;
      }
      if (nu_<D>(m) > 6) { IF_LANE0 s.ctrl[nu_<D>(m) - 1] = act[6] * m.act_ctrlrange[nu_<D>(m) - 1][1]; }
      break;
    }
    default: break;
  }
  WARP_SYNC();
}

// ---------------------------------------------------------------- observation / reward / termination
struct ContactFlags { int grasp_count; int table_hit; int self_hit; };

// The contact predicates of the first s.ncon contacts as bits, the same in every lane: 1 mug - left pad, 2 mug - right pad,
// 4 gripper - table, 8 self-collision.  gym_utils.py:108-128 (distinct pad bodies touching the mug), :174-201 (gripper subtree vs
// table) and :146-172 (two bodies of the robot_base subtree that are not both in the gripper subtree); bodies as in the loaded
// model (GeomFlag)
template <typename Real, typename D>
UR3E_HD int contact_bits(const DevModel<Real>& m, const Arena<Real, D>& s) {
  int f = 0;
  if constexpr (D::HAS_CONTACT) {
    WARP_FOR(k, s.ncon) {
      const int p = s.con_pair[k], f1 = m.geom_flags[m.pair_g1[p]], f2 = m.geom_flags[m.pair_g2[p]], any = f1 | f2;
      if ((any & GF_MUG) && (any & GF_LPAD)) f |= 1;
      if ((any & GF_MUG) && (any & GF_RPAD)) f |= 2;
      if (((f1 & GF_TABLE) && (f2 & GF_GRIPPER)) || ((f2 & GF_TABLE) && (f1 & GF_GRIPPER))) f |= 4;
      if ((f1 & GF_ARM) && (f2 & GF_ARM) && !((f1 & GF_GRIPPER) && (f2 & GF_GRIPPER))) f |= 8;
    }
  }
  return warp_or(f);
}

template <typename Real, typename D>
UR3E_HD ContactFlags contact_flags(const DevModel<Real>& m, const EnvCfg<Real>& c, const Arena<Real, D>& s) {
  (void)c;
  const int f = contact_bits(m, s);
  ContactFlags r; r.grasp_count = (f & 1) + ((f >> 1) & 1); r.table_hit = (f >> 2) & 1; r.self_hit = (f >> 3) & 1;
  return r;
}

template <typename Real, typename D>
UR3E_HD void write_obs(const DevModel<Real>& m, const EnvCfg<Real>& c, Arena<Real, D>& s, const ContactFlags& cf) {
  if (c.obs_kind == OBS_STATE) {
    WARP_FOR(i, nq_<D>(m) + nv_<D>(m)) { if (i < 32) s.obs[i] = i < nq_<D>(m) ? s.st.qpos[i] : s.st.qvel[i - nq_<D>(m)]; }
  } else {
    const Real* tcp = s.site_xpos[c.site_tcp]; const Real* mug = s.site_xpos[c.site_mug]; const Real* ghost = s.xpos[c.body_ghost];
    IF_LANE0 {
      Real* o = s.obs;
      for (int k = 0; k < 3; ++k) { o[k] = tcp[k]; o[3 + k] = mug[k]; o[6 + k] = ghost[k]; }
      if (c.obs_kind == OBS_V2) {
        // ur3e_env2.py:111-123
        for (int k = 0; k < 3; ++k) {
          o[9 + k] = tcp[k] - mug[k]; o[12 + k] = mug[k] - ghost[k];
          o[15 + k] = s.site_velp[c.site_tcp][k]; o[18 + k] = s.site_velp[c.site_tcp][k] - s.site_velp[c.site_mug][k];
        }
        o[21] = s.st.qpos[c.finger_q]; o[22] = s.st.qvel[c.finger_q];
        // gym_utils.py:98-106
        bool robust = cf.grasp_count == 2 && Num<Real>::abs(tcp[0] - mug[0]) < Real(0.01) && Num<Real>::abs(tcp[1] - mug[1]) < Real(0.005) && Num<Real>::abs(tcp[2] - mug[2]) < Real(0.05);
        o[23] = robust ? Real(1) : Real(0);
      } else if (c.obs_kind == OBS_V0) {
        // ur3e_env.py:242-251
        o[9] = (Real)cf.grasp_count;
        for (int k = 0; k < 3; ++k) o[10 + k] = s.site_xpos[c.site_pad][k];
      } else {
        // imitation_env_direct.py:122-130
        o[9] = (Real)cf.grasp_count;
        for (int k = 0; k < 3; ++k) o[10 + k] = s.site_velp[c.site_tcp][k];
      }
    }
  }
  WARP_SYNC();
}

template <typename Real> UR3E_HD Real norm3(Real a, Real b, Real c) { return Num<Real>::sqrt(a * a + b * b + c * c); }

// reward_v2: ur3e_env2.py:150-228
template <typename Real> UR3E_HD Real reward_v2(const Real* o, Real grip) {
  Real mug_z = o[5], gx = o[9], gy = o[10], gz = o[11], grasped = o[23];
  Real xy = Num<Real>::sqrt(gx * gx + gy * gy), zerr = Num<Real>::abs(gz - Real(0.02)), place = norm3(o[12], o[13], o[14]);
  Real ready = Num<Real>::exp(-10 * xy) * Num<Real>::exp(-20 * zerr);
  Real r = Real(2) * ready + Real(2) * grip * ready + Real(10) * grasped * ready;
  r += Real(8) * grasped * Num<Real>::tanh(Real(8) * rmax(Real(0), mug_z));
  r += grasped * (Real(4) * Num<Real>::exp(-15 * place) - Real(1.5) * place);
  if (grasped != 0 && place < Real(0.05)) r += Real(50);
  r += Real(-1) * rmax(Real(0), -gz);
  r += Real(-0.01) * norm3(o[15], o[16], o[17]);
  return r;
}

// reward_v0: ur3e_env.py:256-393
template <typename Real> UR3E_HD Real reward_v0(const Real* o, Real grip, Real half_h, int table_hit, int toppled, int self_hit) {
  Real gs = o[9];
  Real top = o[5] + half_h, bot = o[5] - half_h, pad_top = o[12] - top, g2c = o[2] - o[5];
  Real hx = o[0] - o[3], hy = o[1] - o[4], herr = Num<Real>::sqrt(hx * hx + hy * hy);
  bool valid = gs == 2 && Num<Real>::abs(pad_top) < Real(0.04) && herr < Real(0.03);
  Real height_error = g2c - Real(0.5), z_tol = Real(0.1);
  Real descent = (1 / z_tol) * (height_error + z_tol) * Num<Real>::exp(-(1 / z_tol) * height_error);
  Real ready = Num<Real>::exp(-herr * herr) * Num<Real>::exp(-pad_top * pad_top) * Num<Real>::exp(-height_error * height_error) * 100 * Num<Real>::exp(-grip * grip);
  Real align = 4 * Num<Real>::exp(-60 * herr * herr);
  Real g1 = gs >= 1 ? Real(1) : Real(0), g2 = gs == 2 ? Real(1) : Real(0);
  Real grasp = Real(5.5) * g1 + Real(8.5) * g2 + Real(23.5) * grip * ready + Real(28.5) * g2 * ready + Real(11.5) * g2 * ready * Num<Real>::tanh(8 * grip);
  Real lift = 12 * g2 * Num<Real>::tanh(4 * bot);
  Real dplace = norm3(o[3] - o[6], o[4] - o[7], o[5] - o[8]);
  Real placement = -2 * dplace + 20 * Num<Real>::exp(-70 * dplace * dplace);
  if (dplace < Real(0.05) && valid) placement += 40;
  Real dh = o[5] - o[2] + Real(0.5);
  Real danger = rmin(Real(0), Real(-100000000000.0) * dh * dh * dh);
  Real pen = Real(-40) * self_hit + Real(-25) * table_hit + Real(-8) * toppled + Real(-4) * rmax(Real(0), pad_top) + danger;   // ur3e_env.py:339-345
  Real action_r = Real(700.5) * grip * ready, bonus = Real(1700.5) * g2 * ready * Num<Real>::tanh(10 * grip);
  return descent + align + grasp + lift + placement + action_r + bonus + pen;
}

template <typename Real> struct StepOut { Real reward; int terminated, truncated, reason; };

template <typename Real, typename D>
UR3E_HD StepOut<Real> reward_done(const DevModel<Real>& m, const EnvCfg<Real>& c, Arena<Real, D>& s, const ContactFlags& cf, const Real* act) {
  StepOut<Real> r; r.reward = 0; r.terminated = 0; r.truncated = 0; r.reason = 0;
  const Real* o = s.obs;
  int t = s.st.t;
  if (c.term_kind == TERM_V2) {
    // ur3e_env2.py:84-95, 230-261: reward, t += 1, termination, truncation (t >= max), success override
    r.reward = reward_v2(o, act[c.act_dim - 1]);
    t += 1;
    Real dpick = norm3(o[0] - o[3], o[1] - o[4], o[2] - o[5]);
    int toppled = o[5] <= c.topple_z;
    if (dpick > 1) { r.terminated = 1; r.reason = ST_TERM_REACH; }
    else if (cf.self_hit) { r.terminated = 1; r.reason = ST_TERM_COLLISION; }
    else if (toppled) { r.terminated = 1; r.reason = ST_TERM_TOPPLE; }
    if (t >= c.max_steps) r.truncated = 1;
    if (norm3(o[3] - o[6], o[4] - o[7], o[5] - o[8]) < Real(0.05)) { r.terminated = 1; r.reward += 50; r.reason = ST_SUCCESS; }
  } else if (c.term_kind == TERM_V0) {
    // ur3e_env.py:178-194, 397-462: checks use t before the increment
    int toppled = o[5] <= c.topple_z;
    r.reward = reward_v0(o, act[c.act_dim - 1], c.mug_size[2], cf.table_hit, toppled, cf.self_hit);
    Real dpick = norm3(o[0] - o[3], o[1] - o[4], o[2] - o[5]), dplace = norm3(o[3] - o[6], o[4] - o[7], o[5] - o[8]);
    if (dplace < Real(0.005)) { r.terminated = 1; r.reason = ST_SUCCESS; }
    else if (dpick > 1) { r.terminated = 1; r.reason = ST_TERM_REACH; }
    else if (cf.self_hit) { r.terminated = 1; r.reason = ST_TERM_COLLISION; }
    else if (toppled) { r.terminated = 1; r.reason = ST_TERM_TOPPLE; }
    if (t >= c.max_steps) r.truncated = 1;
    t += 1;
  } else {
    // imitation_env_indirect.py:97-101 / imitation_env_direct.py:99-103: reward -1, never terminates; controller demos: reward 0
    r.reward = c.reward_kind == REW_MINUS1 ? Real(-1) : Real(0);
    if (c.max_steps > 0 && t >= c.max_steps) r.truncated = 1;
    t += 1;
  }
  IF_LANE0 s.st.t = t;
  return r;
}

// ---------------------------------------------------------------- reset (ur3e_env2.py:101-109, gym_utils.py:48-79)
template <typename Real, typename D>
UR3E_PHASE void env_reset(const DevModel<Real>& m, const EnvCfg<Real>& c, Arena<Real, D>& s, const SolverOpts<Real>& opt, uint64_t seed, uint64_t env_id) {
  int key = c.reset_key;
  WARP_FOR(i, nq_<D>(m)) s.st.qpos[i] = key >= 0 ? m.key_qpos[key][i] : m.qpos0[i];
  WARP_FOR(i, nv_<D>(m)) { s.st.qvel[i] = key >= 0 ? m.key_qvel[key][i] : Real(0); s.st.qacc_ws[i] = 0; s.qacc[i] = 0; }
  WARP_FOR(i, nu_<D>(m)) s.ctrl[i] = 0;
  WARP_SYNC();
  if (c.reset_noise != NOISE_NONE && c.body_mug >= 0) {
    uint32_t r[4];
    philox4x32((uint32_t)env_id, (uint32_t)(env_id >> 32), (uint32_t)s.st.episode, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    Real ylo = c.reset_noise == NOISE_HIGH ? Real(-0.25) : c.reset_noise == NOISE_MED ? Real(-0.2) : Real(-0.1);
    Real yhi = c.reset_noise == NOISE_HIGH ? Real(0.2) : c.reset_noise == NOISE_MED ? Real(0.1) : Real(0.01);
    IF_LANE0 { int qa = m.body_qadr[c.body_mug]; s.st.qpos[qa] += Real(0.02) * u01<Real>(r[0]); s.st.qpos[qa + 1] += ylo + (yhi - ylo) * u01<Real>(r[1]); }
  }
  IF_LANE0 { s.st.t = 0; s.st.ep_return = 0; s.st.episode += 1; }
  WARP_SYNC();
  forward_cold(m, s, opt, false);   // set_state -> mj_forward: fresh kinematics, bias and contacts; warm start stays zero
  update_cache(m, c, s);
}

// ---------------------------------------------------------------- one environment step
template <typename Real, typename D>
UR3E_HD StepOut<Real> env_step(const DevModel<Real>& m, const EnvCfg<Real>& c, Arena<Real, D>& s, const SolverOpts<Real>& opt, const Real* act,
                               const SolverOpts<Real>& opt_cold, Real* sens_base = nullptr, long long env = 0) {
  IF_LANE0 { s.overflow = 0; }
#ifdef UR3E_CANARY
  canary_set(s);
#endif
  controller(m, c, s, act);
  // per-step counters live in the arena, not in registers: nothing but the loop counter stays live across the substep calls
  IF_LANE0 { s.max_ncon = 0; s.max_nefc = 0; s.sum_ncon = 0; s.sum_nefc = 0; s.sum_iter = 0; s.warn = 0; }
  for (int k = 0; k < c.frame_skip; ++k) {
    const int w = substep(m, s, opt, opt_cold, k == c.frame_skip - 1 ? sens_base : nullptr, env);   // sensors of the step's last mj_step
    IF_LANE0 {
      s.warn |= w; s.sum_nefc += s.nefc; s.sum_ncon += s.ncon; s.sum_iter += s.solver_iter;
      if (s.ncon > s.max_ncon) s.max_ncon = s.ncon;
      if (s.nefc > s.max_nefc) s.max_nefc = s.nefc;
    }
  }
  WARP_SYNC();
#ifdef UR3E_CANARY
  { const int bad = canary_bad(s); if (bad) { IF_LANE0 { printf("ur3e_b200: arena guard word clobbered (mask 0x%x, env %lld)\n", bad, env); s.warn |= 8; } } }
#endif
  const int warn = s.warn;
  const int sn = s.sum_nefc, sc = s.sum_ncon, si = s.sum_iter;
  update_cache(m, c, s);
  ContactFlags cf = contact_flags(m, c, s);
  write_obs(m, c, s, cf);
  StepOut<Real> r = reward_done(m, c, s, cf, act);
  IF_LANE0 {
    s.st.ep_return += r.reward;
    auto* st = s.st.stat;
    st[ST_NEFC].i += sn; st[ST_NCON].i += sc; st[ST_ITER].i += si; st[ST_SUBSTEPS].i += c.frame_skip;
    if (warn) st[ST_UNSTABLE].i += 1;
    if (s.overflow) st[ST_OVERFLOW].i += 1;
    st[ST_STEPS].i += 1;
    if (cf.grasp_count > 0) st[ST_PADCON].i += 1;
    if (r.terminated || r.truncated) {
      st[ST_EPISODES].i += 1; st[ST_RETURN].f += (float)s.st.ep_return; st[ST_LENGTH].i += s.st.t;
      if (r.terminated && r.reason) st[r.reason].i += 1;
      if (r.truncated && !r.terminated) st[ST_TRUNC].i += 1;
    }
  }
  WARP_SYNC();
  return r;
}

}  // namespace ur3e
