// Kinematics queries (ur3e_batch_query_create): a fixed list of objects of the loaded model compiled into uniform table entries
// for query.cuh.  The kernel model has merged fixed bodies (merge_bodies.h) and tracks only a few sites and the collidable geoms,
// so every object -- body, body inertial frame, geom or site -- becomes a constant frame in one body of the merged model.
#pragma once
#include <cmath>
#include <string>
#include <vector>

#include "../../include/ur3e_b200.h"
#include "host_model.h"
#include "merge_bodies.h"

namespace ur3e {

constexpr int QUERY_MAX_OBJECTS = 256;

template <typename Real>
struct QueryEntry {
  Real lpos[3], lmat[9];   // the object's frame in its anchor body: position, row-major rotation
  int body, root;          // anchor body of the merged model, and the root of its kinematic tree (reference point of cvel)
  int pad_[2];
};

// Compiles `k` (objtype, id) pairs of the loaded model `h`.  Object kinds follow mj_objectVelocity: UR3E_OBJ_BODY = inertial
// frame (d.xipos / d.ximat), UR3E_OBJ_XBODY = body frame (d.xpos / d.xmat), UR3E_OBJ_GEOM, UR3E_OBJ_SITE.  Returns "" on success,
// else the reason the query is invalid.
template <typename Real>
std::string compile_query(const HostModel& h, const int32_t* objtype, const int32_t* objid, int k, std::vector<QueryEntry<Real>>& out) {
  if (!objtype || !objid) return "null object list";
  if (k < 1 || k > QUERY_MAX_OBJECTS) return "query size k=" + std::to_string(k) + " is outside [1, " + std::to_string(QUERY_MAX_OBJECTS) + "]";
  for (int i = 0; i < k; ++i) {
    const int t = objtype[i], n = t == UR3E_OBJ_BODY || t == UR3E_OBJ_XBODY ? h.nbody : t == UR3E_OBJ_GEOM ? h.ngeom : t == UR3E_OBJ_SITE ? h.nsite : -1;
    if (n < 0) return "object " + std::to_string(i) + ": objtype " + std::to_string(t) + " is not UR3E_OBJ_BODY, UR3E_OBJ_XBODY, UR3E_OBJ_GEOM or UR3E_OBJ_SITE";
    if (objid[i] < 0 || objid[i] >= n) return "object " + std::to_string(i) + ": id " + std::to_string(objid[i]) + " is out of range [0, " + std::to_string(n) + ")";
  }
  using namespace merge_detail;
  std::vector<int> bmap;
  const HostModel hm = merge_fixed_bodies(h, bmap);
  // frame of every loaded body in its anchor (the kept ancestor it was merged into), composed the way merge_fixed_bodies does
  // it: a body shares its parent's anchor exactly when it was merged away
  const auto& par = h.I("body_parentid");
  std::vector<double> rp(3 * h.nbody, 0.0), rq(4 * h.nbody, 0.0);
  for (int b = 0; b < h.nbody; ++b) {
    if (b > 0 && bmap[b] == bmap[par[b]]) compose(&rp[3 * b], &rq[4 * b], &rp[3 * par[b]], &rq[4 * par[b]], &h.D("body_pos")[3 * b], &h.D("body_quat")[4 * b]);
    else rq[4 * b] = 1;
  }
  out.assign(k, QueryEntry<Real>{});
  for (int i = 0; i < k; ++i) {
    const int t = objtype[i], id = objid[i];
    double p[3], q[4];
    int a;
    if (t == UR3E_OBJ_XBODY || t == UR3E_OBJ_BODY) {
      a = bmap[id];
      for (int c = 0; c < 3; ++c) p[c] = rp[3 * id + c];
      for (int c = 0; c < 4; ++c) q[c] = rq[4 * id + c];
      if (t == UR3E_OBJ_BODY) {
        const double p0[3] = {p[0], p[1], p[2]}, q0[4] = {q[0], q[1], q[2], q[3]};
        compose(p, q, p0, q0, &h.D("body_ipos")[3 * id], &h.D("body_iquat")[4 * id]);
      }
    } else {   // geoms and sites were re-attached to their anchor by merge_fixed_bodies
      const char* pre = t == UR3E_OBJ_GEOM ? "geom_" : "site_";
      a = hm.I(std::string(pre) + "bodyid")[id];
      for (int c = 0; c < 3; ++c) p[c] = hm.D(std::string(pre) + "pos")[3 * id + c];
      for (int c = 0; c < 4; ++c) q[c] = hm.D(std::string(pre) + "quat")[4 * id + c];
    }
    const double nq = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    for (int c = 0; c < 4; ++c) q[c] = nq < 1e-15 ? (c == 0 ? 1.0 : 0.0) : q[c] / nq;
    double R[9]; q2m(R, q);
    QueryEntry<Real>& e = out[i];
    for (int c = 0; c < 3; ++c) e.lpos[c] = (Real)p[c];
    for (int c = 0; c < 9; ++c) e.lmat[c] = (Real)R[c];
    e.body = a; e.root = hm.I("body_rootid")[a];
  }
  return "";
}

}  // namespace ur3e
