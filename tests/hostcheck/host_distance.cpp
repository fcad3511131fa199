// TEST-ONLY: compiles the geom-distance pass (ur3e_b200/csrc/distance.cuh, with the kinematics it runs), its pair-table compiler and
// its argument check as plain C++ in float64 and float32, so that they can be checked against an exact reference without a GPU.  Not
// part of the package, never loaded by ur3e_b200: the product has no CPU path.  Bound by tests/hostcheck/distance.py.
#include <cstring>
#include <limits>
#include <map>
#include <memory>
#include <string>

#include "../../ur3e_b200/csrc/compile_model.h"
#include "../../ur3e_b200/csrc/distance.cuh"
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

extern "C" const char* hd_error() { return g_err.c_str(); }

template <typename Real>
static void pair_row(int plane1, const double* p1, const double* R1, const double* s1, int plane2, const double* p2, const double* R2, const double* s2,
                     double distmax, double* out) {
  GeomPose<Real> g1, g2;
  DistGeom<Real> t1{}, t2{};
  for (int k = 0; k < 3; ++k) { g1.p[k] = (Real)p1[k]; g2.p[k] = (Real)p2[k]; t1.size[k] = (Real)s1[k]; t2.size[k] = (Real)s2[k]; }
  for (int k = 0; k < 9; ++k) { g1.R[k] = (Real)R1[k]; g2.R[k] = (Real)R2[k]; }
  t1.plane = plane1; t2.plane = plane2;
  Real row[DIST_ROW_W], o[7];
  for (Real& v : row) v = std::numeric_limits<Real>::quiet_NaN();
  geom_distance(g1, t1, g2, t2, distmax >= (double)Num<Real>::big ? Num<Real>::big : (Real)distmax, row, o);
  for (int k = 0; k < 7; ++k) out[k] = o[k];
}

// geom_distance of one pair at given world poses (centre, row-major frame, half-sizes; planeX = 1 for a plane) in float32 / float64:
// out = dist, fromto [6]
extern "C" void hd_pair(int use_float, int plane1, const double* p1, const double* R1, const double* s1, int plane2, const double* p2, const double* R2,
                        const double* s2, double distmax, double* out) {
  if (use_float) pair_row<float>(plane1, p1, R1, s1, plane2, p2, R2, s2, distmax, out);
  else pair_row<double>(plane1, p1, R1, s1, plane2, p2, R2, s2, distmax, out);
}

template <typename Real, typename D>
static int run(const HostModel& h, const int32_t* geom1, const int32_t* geom2, int k, const double* qpos, double distmax, double* dist, double* fromto) {
  std::vector<DistPair<Real>> tab;
  g_err = compile_distance<Real>(h, geom1, geom2, k, tab);
  if (!g_err.empty()) return -1;
  std::vector<int> bmap;
  DevModel<Real> m = compile_model<Real>(merge_fixed_bodies(h, bmap));
  auto s = std::make_unique<Arena<Real, D>>();
  std::memset(s.get(), 0xff, sizeof(Arena<Real, D>));   // NaN everywhere: whatever the pass reads it must have written or loaded
  for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = (Real)qpos[i];
  std::vector<Real> d(k), f(6 * k);
  const Real dm = distmax >= (double)Num<Real>::big ? Num<Real>::big : (Real)distmax;
  distance_env(m, *s, tab.data(), k, dm, dist ? d.data() : nullptr, fromto ? f.data() : nullptr);
  if (dist) for (int i = 0; i < k; ++i) dist[i] = d[i];
  if (fromto) for (int i = 0; i < 6 * k; ++i) fromto[i] = f[i];
  return 0;
}

// The whole per-state pass (kinematics, then every pair) as one warp of ur3e_batch_distance runs it, at qpos [nq]: dist [k],
// fromto [k, 6] (either may be null).  Returns -1 when the pair set is rejected (hd_error).
extern "C" int hd_distance(const char* xml, int use_float, const int32_t* geom1, const int32_t* geom2, int k, const double* qpos, double distmax,
                           double* dist, double* fromto) {
  return with_dims(xml, [&](const HostModel& h, auto d) {
    using D = QueryDims<decltype(d)>;
    return use_float ? run<float, D>(h, geom1, geom2, k, qpos, distmax, dist, fromto) : run<double, D>(h, geom1, geom2, k, qpos, distmax, dist, fromto);
  });
}

// compile_distance itself: 0 when the pair set is accepted, -1 when rejected (hd_error gives the reason)
extern "C" int hd_compile(const char* xml, const int32_t* geom1, const int32_t* geom2, int k) {
  return with_dims(xml, [&](const HostModel& h, auto) {
    std::vector<DistPair<double>> tab;
    g_err = compile_distance<double>(h, geom1, geom2, k, tab);
    return g_err.empty() ? 0 : -1;
  });
}

// distance_check itself: 0 when the call is accepted, -1 when rejected (hd_error gives the reason)
extern "C" int hd_check(int id, int ndist, long long m, long long n, int env_ids, int qpos, int any, double distmax) {
  g_err = distance_check(id, ndist, m, n, env_ids != 0, qpos != 0, any != 0, distmax);
  return g_err.empty() ? 0 : -1;
}

// Staging rows the overlapping path gets per warp, for the size class of the model at xml (float64 / float32)
extern "C" int hd_rows(const char* xml, int use_float) {
  return with_dims(xml, [&](const HostModel&, auto d) {
    using D = QueryDims<decltype(d)>;
    return use_float ? dist_rows<float, D>() : dist_rows<double, D>();
  });
}
