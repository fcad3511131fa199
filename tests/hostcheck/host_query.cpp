// TEST-ONLY: compiles the kinematics-query source (ur3e_b200/csrc/query.cuh + query_model.h) as plain C++ so that the query
// kernel's arithmetic can be checked against the oracle without a GPU.  Not part of the package.
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
static int query(const HostModel& h, const double* qpos, const double* qvel, const int32_t* objtype, const int32_t* objid, int k, int local,
                 double* pos, double* mat, double* vel) {
  std::vector<QueryEntry<double>> tab;
  const std::string err = compile_query<double>(h, objtype, objid, k, tab);
  if (!err.empty()) { std::fprintf(stderr, "hc_query: %s\n", err.c_str()); return -1; }
  std::vector<int> bmap;
  DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
  using DK = QueryDims<D>;
  auto s = std::make_unique<Arena<double, DK>>();
  std::memset(s.get(), 0, sizeof(Arena<double, DK>));
  for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
  for (int i = 0; i < h.nv; ++i) s->st.qvel[i] = qvel[i];
  query_env(m, *s, tab.data(), k, pos, mat, vel, local);
  return 0;
}

// k objects at (qpos, qvel): pos [k][3], mat [k][9], vel [k][6] (any may be null); -1 when the query is rejected
extern "C" int hc_query(const char* xml, const double* qpos, const double* qvel, const int32_t* objtype, const int32_t* objid, int k, int local,
                        double* pos, double* mat, double* vel) {
  try {
    const HostModel& h = get_model(xml);
    if (h.nv <= DimsRaw::NV && h.npair == 0) return query<DimsRaw>(h, qpos, qvel, objtype, objid, k, local, pos, mat, vel);
    if (h.nv <= DimsGrip::NV) return query<DimsGrip>(h, qpos, qvel, objtype, objid, k, local, pos, mat, vel);
    return query<DimsMain>(h, qpos, qvel, objtype, objid, k, local, pos, mat, vel);
  } catch (const std::exception& e) { std::fprintf(stderr, "hc_query: %s\n", e.what()); return -2; }
}
