// TEST-ONLY: compiles the kernel source (ur3e_b200/csrc/engine.cuh, the query sources query.cuh + query_model.h and query_fwd.cuh)
// as plain C++ so that its arithmetic and its argument checks can be checked against the oracle without a GPU.  Not part of the
// package, never loaded by ur3e_b200: the product has no CPU path.
#include <cstdio>
#include <cstring>
#include <limits>
#include <map>
#include <memory>
#include <string>

#include "../../ur3e_b200/csrc/compile_model.h"
#include "../../ur3e_b200/csrc/merge_bodies.h"
#include "../../ur3e_b200/csrc/query.cuh"
#include "../../ur3e_b200/csrc/query_fwd.cuh"

using namespace ur3e;

static std::map<std::string, HostModel> g_models;
static const HostModel& get_model(const char* path) {
  auto it = g_models.find(path);
  if (it == g_models.end()) it = g_models.emplace(path, load_mjcf(path)).first;
  return it->second;
}

// f(D{}) with the generic size class the batch picks for the model at xml (capi.cu): raw without contacts, 2F85, main.
// -2 when the model cannot be loaded.
template <typename F>
static int with_dims(const char* name, const char* xml, F&& f) {
  try {
    const HostModel& h = get_model(xml);
    if (h.nv <= DimsRaw::NV && h.npair == 0) return f(h, DimsRaw{});
    if (h.nv <= DimsGrip::NV && h.nq <= DimsGrip::NQ) return f(h, DimsGrip{});
    return f(h, DimsMain{});
  } catch (const std::exception& e) { std::fprintf(stderr, "%s: %s\n", name, e.what()); return -2; }
}

template <typename Real, typename D>
static int run(const HostModel& h, const double* qpos, const double* qvel, const double* ctrl, const double* ws, int nsteps, int max_iter, double tol,
               double* oq, double* ov, double* oa, double* oM, double* obias, double* ofc, int* info) {
  std::vector<int> bmap;
  DevModel<Real> m = compile_model<Real>(merge_fixed_bodies(h, bmap));
  auto s = std::make_unique<Arena<Real, D>>();
  std::memset(s.get(), 0, sizeof(Arena<Real, D>));
  for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = (Real)qpos[i];
  for (int i = 0; i < h.nv; ++i) { s->st.qvel[i] = (Real)qvel[i]; s->st.qacc_ws[i] = (Real)ws[i]; }
  for (int i = 0; i < h.nu; ++i) s->ctrl[i] = (Real)ctrl[i];
  s->cap_con = D::MAXCON; s->cap_efc = D::MAXEFC;
  SolverOpts<Real> opt{max_iter, 50, (Real)tol, (Real)(sizeof(Real) == 8 ? 1e-14 : 1e-5), (Real)(sizeof(Real) == 8 ? 1e-15 : 2e-6), (Real)(sizeof(Real) == 8 ? 0.0 : 1e-8)};
  int w = 0;
  if (nsteps == 0) forward(m, *s, opt, true);
  for (int k = 0; k < nsteps; ++k) w |= substep(m, *s, opt, opt);
  for (int i = 0; i < h.nq; ++i) oq[i] = s->st.qpos[i];
  for (int i = 0; i < h.nv; ++i) { ov[i] = s->st.qvel[i]; oa[i] = nsteps == 0 ? s->qacc[i] : s->st.qacc_ws[i]; obias[i] = s->qfrc_bias[i]; ofc[i] = s->qfrc_constraint[i]; }
  for (int i = 0; i < h.nv; ++i) for (int j = 0; j < h.nv; ++j) { int hi = i > j ? i : j, lo = i > j ? j : i; oM[i * h.nv + j] = s->M[hi * (hi + 1) / 2 + lo]; }
  info[0] = s->ncon; info[1] = s->nefc; info[2] = s->solver_iter; info[3] = w; info[4] = s->overflow; info[5] = (int)sizeof(Arena<Real, D>);
  return 0;
}

extern "C" int hc_run(const char* xml, int use_float, const double* qpos, const double* qvel, const double* ctrl, const double* ws, int nsteps, int max_iter,
                      double tol, double* oq, double* ov, double* oa, double* oM, double* obias, double* ofc, int* info) {
  return with_dims("hc_run", xml, [&](const HostModel& h, auto d) {
    using D = decltype(d);
    return use_float ? run<float, D>(h, qpos, qvel, ctrl, ws, nsteps, max_iter, tol, oq, ov, oa, oM, obias, ofc, info)
                     : run<double, D>(h, qpos, qvel, ctrl, ws, nsteps, max_iter, tol, oq, ov, oa, oM, obias, ofc, info);
  });
}

// forward pass at (qpos, qvel, ctrl) followed by the logging-sensor cold path: the [NSENSOR] record the step kernel writes
extern "C" int hc_sensors(const char* xml, const double* qpos, const double* qvel, const double* ctrl, double* out) {
  return with_dims("hc_sensors", xml, [&](const HostModel& h, auto d) {
    using D = decltype(d);
    std::vector<int> bmap;
    DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
    auto s = std::make_unique<Arena<double, D>>();
    std::memset(s.get(), 0, sizeof(Arena<double, D>));
    for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
    for (int i = 0; i < h.nv; ++i) s->st.qvel[i] = qvel[i];
    for (int i = 0; i < h.nu; ++i) s->ctrl[i] = ctrl[i];
    s->cap_con = D::MAXCON; s->cap_efc = D::MAXEFC;
    SolverOpts<double> opt{50, 50, 1e-15, 1e-14, 1e-15, 0.0};
    forward(m, *s, opt, true);
    double rec[NSENSOR];
    sensors_cold(m, *s, rec);
    std::memcpy(out, rec, sizeof rec);
    return 0;
  });
}

extern "C" int hc_model_dims(const char* xml, int* out) {
  try {
    const HostModel& h = get_model(xml);
    int v[] = {h.nq, h.nv, h.nu, h.nbody, h.njnt, h.ngeom, h.nsite, h.neq, h.ntendon, h.npair, h.nkey};
    std::memcpy(out, v, sizeof v); return 0;
  } catch (const std::exception& e) { std::fprintf(stderr, "hc_model_dims: %s\n", e.what()); return -1; }
}
extern "C" int hc_model_array(const char* xml, const char* name, double* out, int cap) {
  try {
    const HostModel& h = get_model(xml);
    auto it = h.arr.find(name); if (it == h.arr.end()) return -1;
    int n = it->second.is_int ? (int)it->second.i.size() : (int)it->second.d.size();
    for (int k = 0; k < n && k < cap; ++k) out[k] = it->second.is_int ? it->second.i[k] : it->second.d[k];
    return n;
  } catch (const std::exception& e) { return -2; }
}

// k objects at (qpos, qvel): pos [k][3], mat [k][9], vel [k][6] (any may be null); -1 when the query is rejected
extern "C" int hc_query(const char* xml, const double* qpos, const double* qvel, const int32_t* objtype, const int32_t* objid, int k, int local,
                        double* pos, double* mat, double* vel) {
  return with_dims("hc_query", xml, [&](const HostModel& h, auto d) {
    using DK = QueryDims<decltype(d)>;
    std::vector<QueryEntry<double>> tab;
    const std::string err = compile_query<double>(h, objtype, objid, k, tab);
    if (!err.empty()) { std::fprintf(stderr, "hc_query: %s\n", err.c_str()); return -1; }
    std::vector<int> bmap;
    DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
    auto s = std::make_unique<Arena<double, DK>>();
    std::memset(s.get(), 0, sizeof(Arena<double, DK>));
    for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
    for (int i = 0; i < h.nv; ++i) s->st.qvel[i] = qvel[i];
    query_env(m, *s, tab.data(), k, pos, mat, vel, local);
    return 0;
  });
}

// Jacobians of k objects (query 0; k = 0: none), mass matrix and bias forces at (qpos, qvel) through query_id (0 or -1):
// jacp, jacr [k][3][nv], M [nv][nv], bias [nv] (any may be null); -1 when the call is rejected
extern "C" int hc_query_jac(const char* xml, const double* qpos, const double* qvel, const int32_t* objtype, const int32_t* objid, int k, int query_id,
                            double* jacp, double* jacr, double* M, double* bias) {
  return with_dims("hc_query_jac", xml, [&](const HostModel& h, auto d) {
    using DK = QueryDims<decltype(d)>;
    // the objects (k >= 1) are compiled as the batch's query 0; k = 0: the batch has no query
    std::vector<QueryEntry<double>> tab;
    if (k > 0) {
      const std::string err = compile_query<double>(h, objtype, objid, k, tab);
      if (!err.empty()) { std::fprintf(stderr, "hc_query_jac: %s\n", err.c_str()); return -1; }
    }
    const std::string err = query_jac_check(query_id, k > 0 ? 1 : 0, jacp || jacr, jacp || jacr || M || bias);
    if (!err.empty()) { std::fprintf(stderr, "hc_query_jac: %s\n", err.c_str()); return -1; }
    std::vector<int> bmap;
    DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
    auto s = std::make_unique<Arena<double, DK>>();
    std::memset(s.get(), 0xff, sizeof(Arena<double, DK>));   // NaN everywhere: whatever the query reads it must have written or loaded
    for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
    for (int i = 0; i < h.nv; ++i) s->st.qvel[i] = qvel[i];
    const bool objs = query_id >= 0;
    query_jac_env(m, *s, objs ? tab.data() : nullptr, objs ? k : 0, jacp, jacr, M, bias);
    return 0;
  });
}

// mj_forward at (qpos, qvel, warm start ws) with ctrl (null: zero).  fo = {qacc, qfrc_constraint, contact_dist, contact_pos,
// contact_frame, contact_force, sensordata}, io = {info, contact_geom, flags}: any may be null.  Returns -1 when the call is rejected.
extern "C" int hc_forward(const char* xml, const double* qpos, const double* qvel, const double* ws, const double* ctrl, double* const* fo, int32_t* const* io) {
  return with_dims("hc_forward", xml, [&](const HostModel& h, auto d) {
    using D = decltype(d);
    FwdOut<double> o{fo[0], fo[1], io[0], io[1], fo[2], fo[3], fo[4], fo[5], io[2], fo[6]};
    const bool con = o.contact_geom || o.contact_dist || o.contact_pos || o.contact_frame || o.contact_force;
    const bool any = con || o.qacc || o.qfrc_constraint || o.info || o.flags || o.sensordata;
    const std::string err = forward_query_check(true, con, any, D::HAS_CONTACT ? D::MAXCON : 0);
    if (!err.empty()) { std::fprintf(stderr, "hc_forward: %s\n", err.c_str()); return -1; }
    std::vector<int> bmap;
    DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
    set_geom_flags(h, m);
    auto s = std::make_unique<Arena<double, D>>();
    std::memset(s.get(), 0xff, sizeof(Arena<double, D>));   // NaN everywhere: whatever the query reads it must have written or loaded
    for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
    for (int i = 0; i < h.nv; ++i) { s->st.qvel[i] = qvel[i]; s->st.qacc_ws[i] = ws[i]; }
    // the float64 batch's solver options (batch_impl.cuh Batch::init)
    const SolverOpts<double> opt{50, 50, 1e-15, 1e-14, 1e-15, 0.0};
    forward_query_env(m, *s, opt, ctrl, o);
    return 0;
  });
}

// contacts stored per environment (ur3e_batch_max_contacts)
extern "C" int hc_max_contacts(const char* xml) {
  return with_dims("hc_max_contacts", xml, [](const HostModel&, auto d) { using D = decltype(d); return D::HAS_CONTACT ? D::MAXCON : 0; });
}

// forward_query_check itself: 0 when the combination is accepted, -1 when rejected
extern "C" int hc_forward_check(int out, int con, int any, int ncmax) { return forward_query_check(out != 0, con != 0, any != 0, ncmax).empty() ? 0 : -1; }

// The narrow phase's own functions in Real, called as collision() calls them: out is one STAGE_W staging row, filled with NaN first
// so that a value the function does not write shows, and returned whole (normal in [0, 3), then (pos 3, dist 1) per point).
template <typename Real>
static int box_box_row(const double* p1, const double* R1, const double* s1, const double* p2, const double* R2, const double* s2, double margin, double* out) {
  Real a1[3], a2[3], z1[3], z2[3], st[STAGE_W];
  for (int k = 0; k < 3; ++k) { a1[k] = (Real)p1[k]; a2[k] = (Real)p2[k]; z1[k] = (Real)s1[k]; z2[k] = (Real)s2[k]; }
  for (int k = 0; k < STAGE_W; ++k) st[k] = std::numeric_limits<Real>::quiet_NaN();
  for (int k = 0; k < 9; ++k) { st[k] = (Real)R1[k]; st[9 + k] = (Real)R2[k]; }   // the frames go in through the row
  const int n = box_box<Real>(a1, z1, a2, z2, (Real)margin, st);
  for (int k = 0; k < STAGE_W; ++k) out[k] = st[k];
  return n;
}
template <typename Real>
static int plane_box_row(const double* ppos, const double* pmat, const double* bpos, const double* bmat, const double* size, double margin, double* out) {
  Real pp[3], pm[9], bp[3], bm[9], sz[3], st[STAGE_W];
  for (int k = 0; k < 3; ++k) { pp[k] = (Real)ppos[k]; bp[k] = (Real)bpos[k]; sz[k] = (Real)size[k]; }
  for (int k = 0; k < 9; ++k) { pm[k] = (Real)pmat[k]; bm[k] = (Real)bmat[k]; }
  for (int k = 0; k < STAGE_W; ++k) st[k] = std::numeric_limits<Real>::quiet_NaN();
  const int n = plane_box<Real>(pp, pm, bp, bm, sz, (Real)margin, st);
  for (int k = 0; k < STAGE_W; ++k) out[k] = st[k];
  return n;
}
// box_box / plane_box in float (use_float) or double: the number of points; frames row-major [9], out [STAGE_W]
extern "C" int hc_box_box(int use_float, const double* p1, const double* R1, const double* s1, const double* p2, const double* R2, const double* s2, double margin,
                          double* out) {
  return use_float ? box_box_row<float>(p1, R1, s1, p2, R2, s2, margin, out) : box_box_row<double>(p1, R1, s1, p2, R2, s2, margin, out);
}
extern "C" int hc_plane_box(int use_float, const double* ppos, const double* pmat, const double* bpos, const double* bmat, const double* size, double margin,
                            double* out) {
  return use_float ? plane_box_row<float>(ppos, pmat, bpos, bmat, size, margin, out) : plane_box_row<double>(ppos, pmat, bpos, bmat, size, margin, out);
}
