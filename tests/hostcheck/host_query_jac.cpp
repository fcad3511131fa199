// TEST-ONLY: compiles the Jacobian / mass-matrix query source (ur3e_b200/csrc/query.cuh query_jac_env, query_jac_check) as plain
// C++ so that its arithmetic and its argument checks can be tested against the oracle without a GPU.  Not part of the package.
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>

#include "../../ur3e_b200/csrc/compile_model.h"
#include "../../ur3e_b200/csrc/merge_bodies.h"
#include "../../ur3e_b200/csrc/query.cuh"

using namespace ur3e;

static std::map<std::string, HostModel> g_models;
static const HostModel& get_model(const char* path) {
  auto it = g_models.find(path);
  if (it == g_models.end()) it = g_models.emplace(path, load_mjcf(path)).first;
  return it->second;
}

template <typename D>
static int query_jac(const HostModel& h, const double* qpos, const double* qvel, const int32_t* objtype, const int32_t* objid, int k, int query_id,
                     double* jacp, double* jacr, double* M, double* bias) {
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
  using DK = QueryDims<D>;
  auto s = std::make_unique<Arena<double, DK>>();
  std::memset(s.get(), 0xff, sizeof(Arena<double, DK>));   // NaN everywhere: whatever the query reads it must have written or loaded
  for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
  for (int i = 0; i < h.nv; ++i) s->st.qvel[i] = qvel[i];
  const bool objs = query_id >= 0;
  query_jac_env(m, *s, objs ? tab.data() : nullptr, objs ? k : 0, jacp, jacr, M, bias);
  return 0;
}

// Jacobians of k objects (query 0; k = 0: none), mass matrix and bias forces at (qpos, qvel) through query_id (0 or -1):
// jacp, jacr [k][3][nv], M [nv][nv], bias [nv] (any may be null); -1 when the call is rejected
extern "C" int hc_query_jac(const char* xml, const double* qpos, const double* qvel, const int32_t* objtype, const int32_t* objid, int k, int query_id,
                            double* jacp, double* jacr, double* M, double* bias) {
  try {
    const HostModel& h = get_model(xml);
    if (h.nv <= DimsRaw::NV && h.npair == 0) return query_jac<DimsRaw>(h, qpos, qvel, objtype, objid, k, query_id, jacp, jacr, M, bias);
    if (h.nv <= DimsGrip::NV) return query_jac<DimsGrip>(h, qpos, qvel, objtype, objid, k, query_id, jacp, jacr, M, bias);
    return query_jac<DimsMain>(h, qpos, qvel, objtype, objid, k, query_id, jacp, jacr, M, bias);
  } catch (const std::exception& e) { std::fprintf(stderr, "hc_query_jac: %s\n", e.what()); return -2; }
}
