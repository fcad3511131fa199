// Offscreen rendering (ur3e_batch_render_create / ur3e_batch_render): RGB, depth and geom-segmentation images of a fixed list of
// box and plane geoms of the loaded model, seen from a camera anchored to the world, a body frame or a site.  Two passes: a warp per
// environment runs the step's kinematics and writes the world poses of the geoms and of the camera (render_pose_env), then one
// thread per pixel casts its ray against them (render_pixel).  Like query.cuh this file uses only warp_model.cuh constructs and
// plain arithmetic, so tests/hostcheck compiles it for the CPU.
//
// Semantics: the images are of the stored state, the state the kinematics queries see, i.e. MuJoCo's d.geom_xpos / d.geom_xmat after
// reset / set_state + mj_forward.  After mj_step MuJoCo's arrays still hold the last substep's pre-integration values (SURVEY F9);
// an image after a step is one substep newer than those.  The stored state is never written.
#pragma once
#include <algorithm>
#include <numeric>

#include "query.cuh"

namespace ur3e {

constexpr int RENDER_MAX_GEOMS = 256, RENDER_MAX_SIZE = 2048;

template <typename Real>
struct RenderGeom {
  Real size[3];   // box half sizes; plane (sx, sy, -): |x| <= sx, |y| <= sy, 0 = unbounded
  float rgb[3];
  int type, id;   // GEOM_BOX / GEOM_PLANE, geom id in the loaded model (the segmentation value)
};

template <typename Real>
struct RenderCam {
  Real tanx, tany;   // half extent of the image plane at unit distance: tan(fovy / 2) * W / H, tan(fovy / 2)
  Real znear, zfar;
  int width, height;
};

// Camera construction and argument checks of ur3e_batch_render_create.  The renderer's table `q` holds the k geoms (sorted by id, so
// that equal hit distances go to the lower geom id) followed by the camera: an entry whose frame is the camera's (x right, y up,
// view along -z) in its anchor body.  Returns "" on success, else the reason the renderer is rejected.
template <typename Real>
std::string compile_render(const HostModel& h, const ur3e_camera* cam, const int32_t* geom_ids, int k, const float* rgba, int width, int height,
                           std::vector<QueryEntry<Real>>& q, std::vector<RenderGeom<Real>>& geoms, RenderCam<Real>& rc) {
  if (!cam) return "null camera";
  if (cam->objtype != -1 && cam->objtype != UR3E_OBJ_XBODY && cam->objtype != UR3E_OBJ_SITE)
    return "camera anchor objtype " + std::to_string(cam->objtype) + " is not -1 (world), UR3E_OBJ_XBODY or UR3E_OBJ_SITE";
  if (!geom_ids) return "null geom list";
  if (k < 1 || k > RENDER_MAX_GEOMS) return "geom count k=" + std::to_string(k) + " is outside [1, " + std::to_string(RENDER_MAX_GEOMS) + "]";
  for (int i = 0; i < k; ++i) {
    if (geom_ids[i] < 0 || geom_ids[i] >= h.ngeom) return "geom " + std::to_string(i) + ": id " + std::to_string(geom_ids[i]) + " is out of range [0, " + std::to_string(h.ngeom) + ")";
    const int t = h.I("geom_type")[geom_ids[i]];
    if (t != GEOM_BOX && t != GEOM_PLANE) return "geom " + std::to_string(geom_ids[i]) + " has type " + std::to_string(t) + " (only box and plane are rendered)";
  }
  if (width < 1 || width > RENDER_MAX_SIZE || height < 1 || height > RENDER_MAX_SIZE)
    return "image size " + std::to_string(width) + " x " + std::to_string(height) + " is outside [1, " + std::to_string(RENDER_MAX_SIZE) + "]";
  if (!(cam->fovy > 0 && cam->fovy < 180)) return "fovy " + std::to_string(cam->fovy) + " is outside (0, 180) degrees";
  if (!(cam->znear > 0 && cam->znear < cam->zfar)) return "znear / zfar " + std::to_string(cam->znear) + " / " + std::to_string(cam->zfar) + " do not satisfy 0 < znear < zfar";
  // camera frame in its anchor: MJCF <camera xyaxes>, x normalised, y made orthogonal to x, z = x cross y
  double x[3] = {cam->xyaxes[0], cam->xyaxes[1], cam->xyaxes[2]}, y[3] = {cam->xyaxes[3], cam->xyaxes[4], cam->xyaxes[5]};
  const double nx = std::sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
  if (!(nx > 1e-12)) return "camera xyaxes: x axis is zero";
  for (double& v : x) v /= nx;
  const double xy = x[0] * y[0] + x[1] * y[1] + x[2] * y[2];
  for (int c = 0; c < 3; ++c) y[c] -= xy * x[c];
  const double ny = std::sqrt(y[0] * y[0] + y[1] * y[1] + y[2] * y[2]);
  if (!(ny > 1e-12)) return "camera xyaxes: y axis is zero or parallel to x";
  for (double& v : y) v /= ny;
  const double z[3] = {x[1] * y[2] - x[2] * y[1], x[2] * y[0] - x[0] * y[2], x[0] * y[1] - x[1] * y[0]};
  const double Rc[9] = {x[0], y[0], z[0], x[1], y[1], z[1], x[2], y[2], z[2]};   // columns x, y, z
  double ap[3] = {0, 0, 0}, aR[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  int abody = 0, aroot = 0;
  if (cam->objtype != -1) {
    std::vector<QueryEntry<double>> a;
    const std::string err = compile_query<double>(h, &cam->objtype, &cam->objid, 1, a);
    if (!err.empty()) return "camera anchor: " + err;
    for (int c = 0; c < 3; ++c) ap[c] = a[0].lpos[c];
    for (int c = 0; c < 9; ++c) aR[c] = a[0].lmat[c];
    abody = a[0].body; aroot = a[0].root;
  }
  // geoms in id order, each with its rgba
  std::vector<int> order(k);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return geom_ids[a] < geom_ids[b]; });
  std::vector<int32_t> types(k, UR3E_OBJ_GEOM), ids(k);
  for (int i = 0; i < k; ++i) ids[i] = geom_ids[order[i]];
  const std::string err = compile_query<Real>(h, types.data(), ids.data(), k, q);
  if (!err.empty()) return err;
  geoms.assign(k, RenderGeom<Real>{});
  for (int i = 0; i < k; ++i) {
    const int g = ids[i];
    RenderGeom<Real>& r = geoms[i];
    for (int c = 0; c < 3; ++c) r.size[c] = (Real)h.D("geom_size")[3 * g + c];
    for (int c = 0; c < 3; ++c) r.rgb[c] = rgba ? rgba[4 * order[i] + c] : (float)h.D("geom_rgba")[4 * g + c];
    r.type = h.I("geom_type")[g]; r.id = g;
  }
  QueryEntry<Real> ce{};
  for (int r = 0; r < 3; ++r) {
    double p = ap[r];
    for (int c = 0; c < 3; ++c) p += aR[3 * r + c] * cam->pos[c];
    ce.lpos[r] = (Real)p;
    for (int c = 0; c < 3; ++c) ce.lmat[3 * r + c] = (Real)(aR[3 * r] * Rc[c] + aR[3 * r + 1] * Rc[3 + c] + aR[3 * r + 2] * Rc[6 + c]);
  }
  ce.body = abody; ce.root = aroot;
  q.push_back(ce);
  const double ty = std::tan(cam->fovy * M_PI / 360.0);
  rc.tany = (Real)ty; rc.tanx = (Real)(ty * width / height); rc.znear = (Real)cam->znear; rc.zfar = (Real)cam->zfar;
  rc.width = width; rc.height = height;
  return "";
}

// Arguments of a render call: renderer `id` of `nrender`, `any` = some output given, m environments of a batch of n, env_ids given or
// not.  Returns "" when valid, else the reason the call is rejected.
inline std::string render_check(int id, int nrender, bool any, long long m, long long n, bool env_ids) {
  if (id < 0 || id >= nrender) return "unknown render id " + std::to_string(id);
  if (!any) return "all outputs are null";
  if (m < 1) return "m=" + std::to_string(m) + " environments (at least 1)";
  if (!env_ids && m != n) return "env_ids is null (all environments) but m=" + std::to_string(m) + " is not the batch size " + std::to_string(n);
  return "";
}

// Pose pass of one environment (qpos loaded): pose [k + 1][12].  Geom j < k: its world -> local transform, R^T row-major (9) and
// -R^T p (3); entry k, the camera: camera -> world, R row-major (9) and p (3).
template <typename Real, typename D>
UR3E_HD void render_pose_env(const DevModel<Real>& m, Arena<Real, D>& s, const QueryEntry<Real>* q, int k, Real* pose) {
  kinematics(m, s);
  WARP_FOR(i, 12 * (k + 1)) {
    const int j = i / 12, e = i - 12 * j;
    const QueryEntry<Real>& o = q[j];
    Real v;
    if (e < 9) {
      const int r = e / 3, c = e - 3 * r;
      v = j < k ? entry_rot(s, o, c, r) : entry_rot(s, o, r, c);
    } else {
      const int r = e - 9;
      Real p[3]; entry_point(s, o, p);
      if (j == k) v = r == 0 ? p[0] : (r == 1 ? p[1] : p[2]);   // selects, not a dynamically indexed (local-memory) array
      else v = -(entry_rot(s, o, 0, r) * p[0] + entry_rot(s, o, 1, r) * p[1] + entry_rot(s, o, 2, r) * p[2]);
    }
    pose[i] = v;
  }
}

template <typename Real>
struct RenderPixel { Real depth; int seg; unsigned char rgb[3]; };

// The ray of pixel (px, py) (row 0 at the top) against the k geoms of pose / g: nearest front-facing hit with znear <= t <= zfar,
// t the z-depth (distance along the view axis).  Boxes: the slab entry point; planes: front side only (ray . normal < 0), inside
// |x| <= sx, |y| <= sy where those are nonzero.  Equal t: the earlier geom (lower id).  Headlight shading
// rgb * (0.3 + 0.7 max(0, -n . d)) with d the unit ray, rounded to the nearest uint8.  No hit: depth zfar, seg -1, black.
template <typename Real>
UR3E_HD RenderPixel<Real> render_pixel(const RenderCam<Real>& cam, const Real* pose, const RenderGeom<Real>* g, int k, int px, int py) {
  const Real* C = pose + 12 * k;
  const Real xs = (Real(2) * (Real(px) + Real(0.5)) / Real(cam.width) - Real(1)) * cam.tanx;
  const Real ys = (Real(1) - Real(2) * (Real(py) + Real(0.5)) / Real(cam.height)) * cam.tany;
  // world ray o + t d with d = R (xs, ys, -1): t is the z-depth
  const Real d[3] = {C[0] * xs + C[1] * ys - C[2], C[3] * xs + C[4] * ys - C[5], C[6] * xs + C[7] * ys - C[8]};
  const Real o[3] = {C[9], C[10], C[11]};
  Real best = cam.zfar, cosang = 0;
  int hit = -1;
  for (int j = 0; j < k; ++j) {
    const Real* T = pose + 12 * j;
    Real ol[3], dl[3];
    for (int r = 0; r < 3; ++r) {
      ol[r] = T[3 * r] * o[0] + T[3 * r + 1] * o[1] + T[3 * r + 2] * o[2] + T[9 + r];
      dl[r] = T[3 * r] * d[0] + T[3 * r + 1] * d[1] + T[3 * r + 2] * d[2];
    }
    Real t, nd;   // hit distance and -n . d (unnormalised)
    if (g[j].type == GEOM_PLANE) {
      if (!(dl[2] < 0)) continue;
      t = -ol[2] / dl[2];
      if (!(t >= cam.znear && t <= best && (hit < 0 || t < best))) continue;
      const Real sx = g[j].size[0], sy = g[j].size[1];
      const Real x = ol[0] + t * dl[0], y = ol[1] + t * dl[1];
      if ((sx > 0 && !(x >= -sx && x <= sx)) || (sy > 0 && !(y >= -sy && y <= sy))) continue;
      nd = -dl[2];
    } else {
      Real tn = 0, tf = 0; bool first = true, miss = false;
      nd = 0;
      for (int a = 0; a < 3; ++a) {
        const Real h = g[j].size[a];
        if (dl[a] == 0) { if (ol[a] < -h || ol[a] > h) miss = true; continue; }
        const Real t1 = (-h - ol[a]) / dl[a], t2 = (h - ol[a]) / dl[a];
        const Real lo = t1 < t2 ? t1 : t2, hi = t1 < t2 ? t2 : t1;
        if (first || lo > tn) { tn = lo; nd = dl[a] < 0 ? -dl[a] : dl[a]; }
        if (first || hi < tf) tf = hi;
        first = false;
      }
      t = tn;
      if (miss || !(tn <= tf) || !(t >= cam.znear && t <= best && (hit < 0 || t < best))) continue;
    }
    best = t; hit = j; cosang = nd;
  }
  RenderPixel<Real> out;
  out.depth = best; out.seg = -1; out.rgb[0] = out.rgb[1] = out.rgb[2] = 0;
  if (hit >= 0) {
    const Real len = Num<Real>::sqrt(xs * xs + ys * ys + Real(1));
    const Real shade = Real(0.3) + Real(0.7) * (cosang / len);
    out.seg = g[hit].id;
    for (int c = 0; c < 3; ++c) {
      Real v = Real(g[hit].rgb[c]) * shade;
      v = v < 0 ? Real(0) : (v > 1 ? Real(1) : v);
      out.rgb[c] = (unsigned char)(int)(Real(255) * v + Real(0.5));   // v >= 0: truncation is floor
    }
  }
  return out;
}

}  // namespace ur3e
