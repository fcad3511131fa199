// TEST-ONLY: compiles the renderer's source (ur3e_b200/csrc/render.cuh, with the kinematics it runs) as plain C++ so that its images
// and its argument checks can be checked without a GPU.  Not part of the package, never loaded by ur3e_b200: the product has no CPU
// path.  Bound by tests/hostcheck/render.py.
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>

#include "../../ur3e_b200/csrc/compile_model.h"
#include "../../ur3e_b200/csrc/merge_bodies.h"
#include "../../ur3e_b200/csrc/render.cuh"

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
    if (h.nv <= DimsGrip::NV) return f(h, DimsGrip{});
    return f(h, DimsMain{});
  } catch (const std::exception& e) { g_err = e.what(); return -2; }
}

extern "C" const char* hr_error() { return g_err.c_str(); }

// One environment rendered at qpos through the batch's two passes: rgb [H][W][3], depth [H][W], seg [H][W] (any may be null) and
// the pose scratch [k + 1][12] (may be null).  Returns -1 when the renderer is rejected (hr_error gives the reason).
extern "C" int hr_render(const char* xml, const double* qpos, const ur3e_camera* cam, const int32_t* geom_ids, int k, const float* rgba, int width,
                         int height, uint8_t* rgb, double* depth, int32_t* seg, double* pose_out) {
  return with_dims(xml, [&](const HostModel& h, auto d) {
    using DK = QueryDims<decltype(d)>;
    std::vector<QueryEntry<double>> q; std::vector<RenderGeom<double>> g; RenderCam<double> rc{};
    g_err = compile_render<double>(h, cam, geom_ids, k, rgba, width, height, q, g, rc);
    if (!g_err.empty()) return -1;
    std::vector<int> bmap;
    DevModel<double> m = compile_model<double>(merge_fixed_bodies(h, bmap));
    auto s = std::make_unique<Arena<double, DK>>();
    std::memset(s.get(), 0xff, sizeof(Arena<double, DK>));   // NaN everywhere: whatever the pass reads it must have written or loaded
    for (int i = 0; i < h.nq; ++i) s->st.qpos[i] = qpos[i];
    std::vector<double> pose(12 * (k + 1));
    render_pose_env(m, *s, q.data(), k, pose.data());
    if (pose_out) std::memcpy(pose_out, pose.data(), sizeof(double) * pose.size());
    for (int p = 0; p < width * height; ++p) {
      const RenderPixel<double> r = render_pixel(rc, pose.data(), g.data(), k, p % width, p / width);
      if (rgb) for (int c = 0; c < 3; ++c) rgb[3 * p + c] = r.rgb[c];
      if (depth) depth[p] = r.depth;
      if (seg) seg[p] = r.seg;
    }
    return 0;
  });
}

// render_check itself: 0 when the call is accepted, -1 when rejected (hr_error gives the reason)
extern "C" int hr_render_check(int id, int nrender, int any, long long m, long long n, int env_ids) {
  g_err = render_check(id, nrender, any != 0, m, n, env_ids != 0);
  return g_err.empty() ? 0 : -1;
}
