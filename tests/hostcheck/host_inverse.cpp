// TEST-ONLY: compiles the inverse-dynamics query's source (ur3e_b200/csrc/query_inv.cuh, with the engine phases it runs) and its argument
// check as plain C++ so that both can be checked against the oracle without a GPU.  Not part of the package, never loaded by ur3e_b200:
// the product has no CPU path.  Bound by tests/hostcheck/inverse.py.
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>

#include "../../ur3e_b200/csrc/compile_model.h"
#include "../../ur3e_b200/csrc/merge_bodies.h"
#include "../../ur3e_b200/csrc/query_inv.cuh"

using namespace ur3e;

static std::map<std::string, HostModel> g_models;
static std::string g_err;   // the reason the latest call was rejected

// f(h, D{}) with the generic size class the batch picks for the model at xml (capi.cu); -2 when the model cannot be loaded
template <typename F>
static int with_dims(const char* xml, F&& f) {
  try {
    auto it = g_models.find(xml);
    if (it == g_models.end()) it = g_models.emplace(xml, load_mjcf(xml)).first;
    const HostModel& h = it->second;
    if (h.nv <= DimsRaw::NV && h.npair == 0) return f(h, DimsRaw{});
    if (h.nv <= DimsGrip::NV && h.nq <= DimsGrip::NQ) return f(h, DimsGrip{});
    return f(h, DimsMain{});
  } catch (const std::exception& e) { g_err = e.what(); return -2; }
}

extern "C" const char* hi_error() { return g_err.c_str(); }

// contacts stored per state (ur3e_batch_max_contacts)
extern "C" int hi_max_contacts(const char* xml) {
  return with_dims(xml, [](const HostModel&, auto d) { using D = decltype(d); return D::HAS_CONTACT ? D::MAXCON : 0; });
}

// mj_inverse of one state (qpos, qvel) at qacc, float64, as ur3e_batch_inverse computes it.  Outputs (any may be null): qfrc_inverse
// [nv], qfrc_constraint [nv], info [3], contact_geom [C][2], contact_force [C][6].  Returns -1 when the call is rejected (hi_error).
extern "C" int hi_inverse(const char* xml, const double* qpos, const double* qvel, const double* qacc, int discrete, double* qfrc_inverse,
                          double* qfrc_constraint, int32_t* info, int32_t* contact_geom, double* contact_force) {
  return with_dims(xml, [&](const HostModel& h, auto d) {
    using D = decltype(d);
    const bool con = contact_geom || contact_force;
    g_err = inverse_query_check(true, true, 1, 1, qacc != nullptr, true, con, con || qfrc_inverse || qfrc_constraint || info, D::HAS_CONTACT ? D::MAXCON : 0);
    if (!g_err.empty()) return -1;
    std::vector<int> bmap;
    DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
    set_geom_flags(h, m);
    auto s = std::make_unique<Arena<double, D>>();
    std::memset(s.get(), 0xff, sizeof(Arena<double, D>));   // NaN everywhere: whatever the pass reads it must have written or loaded
    for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
    for (int i = 0; i < h.nv; ++i) s->st.qvel[i] = qvel[i];
    inverse_query_env(m, *s, discrete != 0, qacc, InvOut<double>{qfrc_inverse, qfrc_constraint, info, contact_geom, contact_force});
    return 0;
  });
}

// inverse_query_check itself: 0 when the call is accepted, -1 when rejected (hi_error gives the reason)
extern "C" int hi_inverse_check(int qpos, int qvel, long long m, long long n, int qacc, int out, int con, int any, int ncmax) {
  g_err = inverse_query_check(qpos != 0, qvel != 0, m, n, qacc != 0, out != 0, con != 0, any != 0, ncmax);
  return g_err.empty() ? 0 : -1;
}
