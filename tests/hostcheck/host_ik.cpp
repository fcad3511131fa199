// TEST-ONLY: compiles the inverse-kinematics solve (ur3e_b200/csrc/ik.cuh, with the kinematics it runs), its table compiler and its
// argument check as plain C++ so that all three can be checked against the oracle without a GPU.  Not part of the package, never loaded
// by ur3e_b200: the product has no CPU path.  Bound by tests/hostcheck/ik.py.
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>

#include "../../ur3e_b200/csrc/compile_model.h"
#include "../../ur3e_b200/csrc/ik.cuh"
#include "../../ur3e_b200/csrc/merge_bodies.h"

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

// One IK problem, float64, as ur3e_batch_ik solves it: object (objtype, objid), joints [nj], start qpos [nq], targets (either may be
// null), options (null = the defaults).  Outputs (any may be null): qpos_out [nq], err_out [1], info [2].  Returns -1 when the family
// or the call is rejected (hi_error).
extern "C" int hi_ik(const char* xml, int objtype, int objid, const int32_t* joints, int nj, const double* qpos, const double* target_pos,
                     const double* target_quat, const ur3e_ik_options* opt, double* qpos_out, double* err_out, int32_t* info) {
  return with_dims(xml, [&](const HostModel& h, auto d) {
    using D = QueryDims<decltype(d)>;
    auto tab = std::make_unique<IkTable<double>>();
    g_err = compile_ik<double>(h, objtype, objid, joints, nj, *tab);
    if (!g_err.empty()) return -1;
    g_err = ik_check(0, 1, 1, 1, false, true, target_pos != nullptr, target_quat != nullptr, true, qpos_out || err_out || info, opt);
    if (!g_err.empty()) return -1;
    std::vector<int> bmap;
    DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
    auto s = std::make_unique<Arena<double, D>>();
    std::memset(s.get(), 0xff, sizeof(Arena<double, D>));   // NaN everywhere: whatever the solve reads it must have written or loaded
    for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
    const ur3e_ik_options o = opt ? *opt : ur3e_ik_options{ik_default_tol<double>(), 1.0, 0.1, 3e-2, 2.0, 20.0, 100, 0};
    const IkOpts<double> ko{o.tol, o.rot_weight, o.regularization_threshold, o.regularization_strength, o.max_update_norm, o.progress_thresh, o.max_steps};
    const IkResult<double> r = ik_env(m, *s, *tab, target_pos, target_quat, ko);
    if (qpos_out) for (int i = 0; i < h.nq; ++i) qpos_out[i] = s->st.qpos[i];
    if (err_out) *err_out = r.err_norm;
    if (info) { info[0] = r.steps; info[1] = r.status; }
    return 0;
  });
}

// compile_ik itself: 0 when the family is accepted, -1 when rejected (hi_error gives the reason)
extern "C" int hi_ik_compile(const char* xml, int objtype, int objid, const int32_t* joints, int nj) {
  return with_dims(xml, [&](const HostModel& h, auto) {
    auto tab = std::make_unique<IkTable<double>>();
    g_err = compile_ik<double>(h, objtype, objid, joints, nj, *tab);
    return g_err.empty() ? 0 : -1;
  });
}

// ik_check itself: 0 when the call is accepted, -1 when rejected (hi_error gives the reason)
extern "C" int hi_ik_check(int id, int nik, long long m, long long n, int env_ids, int qpos0, int pos, int quat, int out, int any,
                           const ur3e_ik_options* opt) {
  g_err = ik_check(id, nik, m, n, env_ids != 0, qpos0 != 0, pos != 0, quat != 0, out != 0, any != 0, opt);
  return g_err.empty() ? 0 : -1;
}
