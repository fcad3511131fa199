// TEST-ONLY: compiles the forward-dynamics query source (ur3e_b200/csrc/query_fwd.cuh forward_query_env, forward_query_check) as
// plain C++ so that its arithmetic and its argument checks can be tested against the oracle without a GPU.  Not part of the package.
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>

#include "../../ur3e_b200/csrc/compile_model.h"
#include "../../ur3e_b200/csrc/merge_bodies.h"
#include "../../ur3e_b200/csrc/query_fwd.cuh"

using namespace ur3e;

static std::map<std::string, HostModel> g_models;
static const HostModel& get_model(const char* path) {
  auto it = g_models.find(path);
  if (it == g_models.end()) it = g_models.emplace(path, load_mjcf(path)).first;
  return it->second;
}

template <typename D>
static int forward(const HostModel& h, const double* qpos, const double* qvel, const double* ws, const double* ctrl, double* const* fo, int32_t* const* io) {
  constexpr int C = D::HAS_CONTACT ? D::MAXCON : 0;
  FwdOut<double> o{fo[0], fo[1], io[0], io[1], fo[2], fo[3], fo[4], fo[5], io[2], fo[6]};
  const bool con = o.contact_geom || o.contact_dist || o.contact_pos || o.contact_frame || o.contact_force;
  const bool any = con || o.qacc || o.qfrc_constraint || o.info || o.flags || o.sensordata;
  const std::string err = forward_query_check(true, con, any, C);
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
}

// mj_forward at (qpos, qvel, warm start ws) with ctrl (null: zero).  fo = {qacc, qfrc_constraint, contact_dist, contact_pos,
// contact_frame, contact_force, sensordata}, io = {info, contact_geom, flags}: any may be null.  Returns -1 when the call is rejected.
extern "C" int hc_forward(const char* xml, const double* qpos, const double* qvel, const double* ws, const double* ctrl, double* const* fo, int32_t* const* io) {
  try {
    const HostModel& h = get_model(xml);
    if (h.nv <= DimsRaw::NV && h.npair == 0) return forward<DimsRaw>(h, qpos, qvel, ws, ctrl, fo, io);
    if (h.nv <= DimsGrip::NV) return forward<DimsGrip>(h, qpos, qvel, ws, ctrl, fo, io);
    return forward<DimsMain>(h, qpos, qvel, ws, ctrl, fo, io);
  } catch (const std::exception& e) { std::fprintf(stderr, "hc_forward: %s\n", e.what()); return -2; }
}

// contacts stored per environment (ur3e_batch_max_contacts)
extern "C" int hc_max_contacts(const char* xml) {
  try {
    const HostModel& h = get_model(xml);
    if (h.nv <= DimsRaw::NV && h.npair == 0) return DimsRaw::HAS_CONTACT ? DimsRaw::MAXCON : 0;
    if (h.nv <= DimsGrip::NV) return DimsGrip::MAXCON;
    return DimsMain::MAXCON;
  } catch (const std::exception& e) { std::fprintf(stderr, "hc_max_contacts: %s\n", e.what()); return -2; }
}

// forward_query_check itself: 0 when the combination is accepted, -1 when rejected
extern "C" int hc_forward_check(int out, int con, int any, int ncmax) { return forward_query_check(out != 0, con != 0, any != 0, ncmax).empty() ? 0 : -1; }
