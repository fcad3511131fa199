// Geom distances (mj_geomDistance): the signed distance and the closest points of k fixed pairs of box / plane geoms of the loaded
// model, for one state per warp, off the step path.  Read-only: the caller loads qpos into the arena; nothing is written back to a
// record.  Like engine.cuh this file uses only warp_model.cuh constructs, so tests/hostcheck compiles it for the CPU.
//
// Semantics, per pair (geom1, geom2), capped at distmax:
//   box-box, disjoint (some SAT axis separates): the exact Euclidean distance of the two solids, fromto = the closest points: the
//     minimum of the 16 vertex-to-solid-box distances (closed form: clamp in the box's frame) and the 144 edge-edge segment
//     distances, which between them reach every closest feature pair of two disjoint boxes;
//   box-box, overlapping: what the collider returns, as mj_geomDistance does: the contact of box_box(..., margin = 0, ...) with the
//     smallest dist, fromto = pos -/+ dist/2 normal (on geom1, on geom2).  When box_box finds no point (a touching pair that rounding
//     puts on the overlapping side) the exact path gives the value, near 0, so that the two regimes meet at zero;
//   plane-box: the plane is the infinite half-space below its z axis, as in collision(): dist = the smallest signed height of the
//     8 vertices (plane_box keeps only 4 points and not always the deepest), fromto = that vertex projected onto the plane, and the
//     vertex (swapped when the plane is geom2);
//   dist >= distmax: dist = distmax, fromto = 0.
#pragma once
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "query.cuh"

namespace ur3e {

constexpr int DIST_MAX_PAIRS = 256;

template <typename Real>
struct DistGeom {
  QueryEntry<Real> e;   // the geom's frame in its anchor body
  Real size[3];         // box half-sizes (a plane's are not used: it is infinite)
  int plane, pad_;      // 1: plane, 0: box
};
template <typename Real> struct DistPair { DistGeom<Real> g[2]; };

// Compiles the k pairs (geom1[i], geom2[i]) of the loaded model h.  Returns "" on success, else the reason.
template <typename Real>
std::string compile_distance(const HostModel& h, const int32_t* geom1, const int32_t* geom2, int k, std::vector<DistPair<Real>>& out) {
  if (!geom1 || !geom2) return "null geom list";
  if (k < 1 || k > DIST_MAX_PAIRS) return "pair count k=" + std::to_string(k) + " is outside [1, " + std::to_string(DIST_MAX_PAIRS) + "]";
  const auto& gt = h.I("geom_type");
  const auto& gs = h.D("geom_size");
  std::vector<int32_t> type(2 * k, UR3E_OBJ_GEOM), id(2 * k);
  for (int i = 0; i < k; ++i) {
    const int g[2] = {geom1[i], geom2[i]};
    for (int c = 0; c < 2; ++c) {
      if (g[c] < 0 || g[c] >= h.ngeom) return "pair " + std::to_string(i) + ": geom id " + std::to_string(g[c]) + " is out of range [0, " + std::to_string(h.ngeom) + ")";
      if (gt[g[c]] != GEOM_BOX && gt[g[c]] != GEOM_PLANE) return "pair " + std::to_string(i) + ": geom " + std::to_string(g[c]) + " has type " + std::to_string(gt[g[c]]) + " (only box and plane geoms are supported)";
      id[2 * i + c] = g[c];
    }
    if (g[0] == g[1]) return "pair " + std::to_string(i) + ": geom " + std::to_string(g[0]) + " is paired with itself";
    if (gt[g[0]] == GEOM_PLANE && gt[g[1]] == GEOM_PLANE) return "pair " + std::to_string(i) + ": two planes (" + std::to_string(g[0]) + ", " + std::to_string(g[1]) + ")";
  }
  std::vector<QueryEntry<Real>> q, part;
  for (int c = 0; c < 2 * k; c += QUERY_MAX_OBJECTS) {   // compile_query takes at most QUERY_MAX_OBJECTS objects at a time
    const std::string err = compile_query<Real>(h, type.data() + c, id.data() + c, std::min(2 * k - c, QUERY_MAX_OBJECTS), part);
    if (!err.empty()) return err;
    q.insert(q.end(), part.begin(), part.end());
  }
  out.assign(k, DistPair<Real>{});
  for (int i = 0; i < 2 * k; ++i) {
    DistGeom<Real>& d = out[i / 2].g[i % 2];
    d.e = q[i]; d.plane = gt[id[i]] == GEOM_PLANE;
    for (int c = 0; c < 3; ++c) d.size[c] = (Real)gs[3 * id[i] + c];
  }
  return "";
}

// Arguments of a distance call (ur3e_batch_distance): pair set `id` of `ndist`, m states, the batch's n, which source is given,
// `any` = some output requested.  Returns "" when valid, else the reason.
inline std::string distance_check(int id, int ndist, long long m, long long n, bool env_ids, bool qpos, bool any, double distmax) {
  if (id < 0 || id >= ndist) return "unknown distance id " + std::to_string(id);
  if (m < 1 || m > 2147483647LL) return "m=" + std::to_string(m) + " states (1 .. 2^31 - 1)";
  if (env_ids && qpos) return "give env_ids or qpos, not both";
  if (!env_ids && !qpos && m != n) return "m=" + std::to_string(m) + " for the stored state of n=" + std::to_string(n) + " environments (m must equal n)";
  if (!any) return "all outputs are null";
  if (distmax != distmax) return "distmax is NaN";
  return "";
}

// world frame of a geom: position p, row-major rotation R (column a = the geom's axis a)
template <typename Real> struct GeomPose { Real p[3], R[9]; };

template <typename Real, typename D>
UR3E_HD GeomPose<Real> geom_pose(const Arena<Real, D>& s, const QueryEntry<Real>& e) {
  GeomPose<Real> g;
  entry_point(s, e, g.p);
  for (int c = 0; c < 9; ++c) g.R[c] = entry_rot(s, e, c / 3, c - 3 * (c / 3));
  return g;
}

// A candidate closest pair: squared distance d2 (or signed distance d, see geom_distance), point a on geom1, point b on geom2
template <typename Real> struct DistPts { Real d, a[3], b[3]; };

// Element k of a 3-vector, selected (not a dynamically indexed, local-memory array), and column c of a row-major 3 x 3 matrix
template <typename Real> UR3E_HD Real sel3(const Real* v, int k) { return k == 0 ? v[0] : (k == 1 ? v[1] : v[2]); }
template <typename Real> UR3E_HD void col3(const Real* R, int c, Real* o) { o[0] = sel3(R, c); o[1] = sel3(R + 3, c); o[2] = sel3(R + 6, c); }

// True when one of the 15 SAT axes separates the boxes (some projected gap > 0).  Edge-edge axes of nearly parallel edges
// (|u x v| < 1e-6) are skipped as in box_box; the face axes then decide.
template <typename Real>
UR3E_HD bool box_separated(const GeomPose<Real>& g1, const Real* s1, const GeomPose<Real>& g2, const Real* s2) {
  const Real d[3] = {g2.p[0] - g1.p[0], g2.p[1] - g1.p[1], g2.p[2] - g1.p[2]};
  bool sep = false;
  for (int ax = 0; ax < 15; ++ax) {
    Real n[3];
    if (ax < 3) col3(g1.R, ax, n);
    else if (ax < 6) col3(g2.R, ax - 3, n);
    else {
      Real u[3], v[3]; col3(g1.R, (ax - 6) / 3, u); col3(g2.R, (ax - 6) % 3, v);
      cross3(n, u, v);
      const Real l = Num<Real>::sqrt(dot3(n, n));
      if (l < Real(1e-6)) continue;
      for (int k = 0; k < 3; ++k) n[k] /= l;
    }
    Real r = 0;
    for (int k = 0; k < 3; ++k) {
      Real a[3], b[3]; col3(g1.R, k, a); col3(g2.R, k, b);
      r += s1[k] * Num<Real>::abs(dot3(a, n)) + s2[k] * Num<Real>::abs(dot3(b, n));
    }
    sep |= Num<Real>::abs(dot3(d, n)) - r > 0;
  }
  return sep;
}

// Vertex i (bit c = sign of axis c) of a box
template <typename Real>
UR3E_HD void box_vertex(const GeomPose<Real>& g, const Real* s, int i, Real* v) {
  const Real x = (i & 1) ? s[0] : -s[0], y = (i & 2) ? s[1] : -s[1], z = (i & 4) ? s[2] : -s[2];
  for (int k = 0; k < 3; ++k) v[k] = g.p[k] + g.R[3 * k] * x + g.R[3 * k + 1] * y + g.R[3 * k + 2] * z;
}

// Exact distance of two disjoint boxes: r.d = the squared distance, r.a on box 1, r.b on box 2.  For overlapping boxes the value
// is not the penetration (a vertex inside the other box gives 0).
template <typename Real>
UR3E_HD DistPts<Real> box_box_exact(const GeomPose<Real>& g1, const Real* s1, const GeomPose<Real>& g2, const Real* s2) {
  DistPts<Real> r; r.d = Num<Real>::big;
  for (int k = 0; k < 3; ++k) r.a[k] = r.b[k] = 0;
  // the 16 vertices against the other solid box: clamp the vertex's coordinates in the box's frame (called with fixed roles, so that
  // no frame is selected at run time)
  auto vertices = [&](const GeomPose<Real>& gv, const Real* sv, const GeomPose<Real>& gb, const Real* sb, bool first) {
    for (int i = 0; i < 8; ++i) {
      Real v[3], w[3], q[3]; box_vertex(gv, sv, i, v);
      for (int k = 0; k < 3; ++k) w[k] = v[k] - gb.p[k];
      Real d2 = 0;
      for (int c = 0; c < 3; ++c) {
        const Real l = gb.R[c] * w[0] + gb.R[3 + c] * w[1] + gb.R[6 + c] * w[2], h = sb[c], cl = rmin(rmax(l, -h), h);
        d2 += (l - cl) * (l - cl);
        q[c] = cl;
      }
      if (d2 < r.d) {
        r.d = d2;
        for (int k = 0; k < 3; ++k) {
          const Real on = gb.p[k] + gb.R[3 * k] * q[0] + gb.R[3 * k + 1] * q[1] + gb.R[3 * k + 2] * q[2];
          r.a[k] = first ? v[k] : on; r.b[k] = first ? on : v[k];
        }
      }
    }
  };
  vertices(g1, s1, g2, s2, true);
  vertices(g2, s2, g1, s1, false);
  // the 12 x 12 edge pairs: edge e of a box runs along axis a = e / 4 through the centre offset by +-size along the other two axes;
  // closest points of the segments c1 + s u, c2 + t v (|s| <= h1, |t| <= h2) by the clamped normal equations (Ericson 5.1.9)
  for (int e1 = 0; e1 < 12; ++e1) {
    const int a1 = e1 >> 2, b1 = a1 == 2 ? 0 : a1 + 1, c1 = b1 == 2 ? 0 : b1 + 1;
    Real u[3], ob[3], oc[3]; col3(g1.R, a1, u); col3(g1.R, b1, ob); col3(g1.R, c1, oc);
    const Real h1 = sel3(s1, a1), fb = (e1 & 1) ? sel3(s1, b1) : -sel3(s1, b1), fc = (e1 & 2) ? sel3(s1, c1) : -sel3(s1, c1);
    Real p1[3]; for (int k = 0; k < 3; ++k) p1[k] = g1.p[k] + fb * ob[k] + fc * oc[k];
    for (int e2 = 0; e2 < 12; ++e2) {
      const int a2 = e2 >> 2, b2 = a2 == 2 ? 0 : a2 + 1, c2 = b2 == 2 ? 0 : b2 + 1;
      Real v[3], pb[3], pc[3]; col3(g2.R, a2, v); col3(g2.R, b2, pb); col3(g2.R, c2, pc);
      const Real h2 = sel3(s2, a2), gb = (e2 & 1) ? sel3(s2, b2) : -sel3(s2, b2), gc = (e2 & 2) ? sel3(s2, c2) : -sel3(s2, c2);
      Real p2[3], w[3];
      for (int k = 0; k < 3; ++k) { p2[k] = g2.p[k] + gb * pb[k] + gc * pc[k]; w[k] = p1[k] - p2[k]; }
      const Real b = dot3(u, v), d = dot3(u, w), e = dot3(v, w), den = 1 - b * b;
      Real s = den > Real(1e-12) ? rmin(rmax((b * e - d) / den, -h1), h1) : Real(0);
      Real t = e + b * s;
      if (t < -h2 || t > h2) { t = rmin(rmax(t, -h2), h2); s = rmin(rmax(t * b - d, -h1), h1); }
      Real d2 = 0, x[3], y[3];
      for (int k = 0; k < 3; ++k) { x[k] = p1[k] + s * u[k]; y[k] = p2[k] + t * v[k]; d2 += (x[k] - y[k]) * (x[k] - y[k]); }
      if (d2 < r.d) { r.d = d2; for (int k = 0; k < 3; ++k) { r.a[k] = x[k]; r.b[k] = y[k]; } }
    }
  }
  return r;
}

// Plane (geom pl) and box (gb, half-sizes s): the smallest signed height of the 8 vertices above the plane, r.a = that vertex projected
// onto the plane, r.b = the vertex
template <typename Real>
UR3E_HD DistPts<Real> plane_box_exact(const GeomPose<Real>& pl, const GeomPose<Real>& gb, const Real* s) {
  const Real n[3] = {pl.R[2], pl.R[5], pl.R[8]};
  DistPts<Real> r; r.d = Num<Real>::big;
  for (int k = 0; k < 3; ++k) r.a[k] = r.b[k] = 0;
  for (int i = 0; i < 8; ++i) {
    Real v[3]; box_vertex(gb, s, i, v);
    const Real h = n[0] * (v[0] - pl.p[0]) + n[1] * (v[1] - pl.p[1]) + n[2] * (v[2] - pl.p[2]);
    if (h < r.d) { r.d = h; for (int k = 0; k < 3; ++k) { r.b[k] = v[k]; r.a[k] = v[k] - h * n[k]; } }
  }
  return r;
}

// Staging row of the overlapping path: box_box's row (frames in, contacts out), then the two centres
constexpr int DIST_ROW_W = STAGE_W + 6;

// The no-staging part of one pair: the plane-box result, or the exact result of a disjoint box pair.  Returns false (r unset) when
// the boxes overlap, which needs box_box and a staging row (geom_distance).  r.d is the signed distance.
template <typename Real>
UR3E_HD bool geom_distance_direct(const GeomPose<Real>& g1, const DistGeom<Real>& t1, const GeomPose<Real>& g2, const DistGeom<Real>& t2,
                                  bool force_exact, DistPts<Real>& r) {
  if (t1.plane || t2.plane) {
    const bool p1 = t1.plane != 0;
    const DistPts<Real> q = p1 ? plane_box_exact(g1, g2, t2.size) : plane_box_exact(g2, g1, t1.size);
    r.d = q.d;
    for (int k = 0; k < 3; ++k) { r.a[k] = p1 ? q.a[k] : q.b[k]; r.b[k] = p1 ? q.b[k] : q.a[k]; }
    return true;
  }
  if (!force_exact && !box_separated(g1, t1.size, g2, t2.size)) return false;
  r = box_box_exact(g1, t1.size, g2, t2.size);
  r.d = Num<Real>::sqrt(r.d);
  return true;
}

// The overlapping box pair: the smallest-dist contact of box_box(margin 0) on the staging row `row` (DIST_ROW_W values, shared
// memory on the GPU), fromto = pos -/+ dist/2 normal.  Returns false when box_box finds no point.
template <typename Real>
UR3E_HD bool box_box_contact(const GeomPose<Real>& g1, const DistGeom<Real>& t1, const GeomPose<Real>& g2, const DistGeom<Real>& t2, Real* row,
                             DistPts<Real>& r) {
  // the out-of-line box_box takes everything through the row: arrays passed by address would live on the stack
  for (int k = 0; k < 9; ++k) { row[k] = g1.R[k]; row[9 + k] = g2.R[k]; }
  for (int k = 0; k < 3; ++k) { row[STAGE_W + k] = g1.p[k]; row[STAGE_W + 3 + k] = g2.p[k]; }
  const int n = box_box(row + STAGE_W, t1.size, row + STAGE_W + 3, t2.size, Real(0), row);
  if (n == 0) return false;
  int best = 0;
  for (int c = 1; c < n; ++c) if (row[3 + 4 * c + 3] < row[3 + 4 * best + 3]) best = c;
  const Real* pt = row + 3 + 4 * best;
  r.d = pt[3];
  for (int k = 0; k < 3; ++k) { r.a[k] = pt[k] - Real(0.5) * r.d * row[k]; r.b[k] = pt[k] + Real(0.5) * r.d * row[k]; }
  return true;
}

// mj_geomDistance of one pair at the given world poses, every regime: out = dist, fromto (7 values).  `row` is a staging row of
// DIST_ROW_W values.  distance_env runs the same pieces, with the overlapping pairs batched into the arena's rows.
template <typename Real>
UR3E_HD void geom_distance(const GeomPose<Real>& g1, const DistGeom<Real>& t1, const GeomPose<Real>& g2, const DistGeom<Real>& t2, Real distmax,
                           Real* row, Real* out) {
  DistPts<Real> r;
  if (!geom_distance_direct(g1, t1, g2, t2, false, r) && !box_box_contact(g1, t1, g2, t2, row, r)) geom_distance_direct(g1, t1, g2, t2, true, r);
  const bool keep = r.d < distmax;
  out[0] = keep ? r.d : distmax;
  for (int k = 0; k < 3; ++k) { out[1 + k] = keep ? r.a[k] : Real(0); out[4 + k] = keep ? r.b[k] : Real(0); }
}

// Lower bounds of a pair's distance: the box centre's height over the plane minus its bounding radius; the centre distance minus
// both bounding radii
template <typename Real> UR3E_HD Real plane_box_bound(const GeomPose<Real>& pl, const GeomPose<Real>& bx, const Real* s) {
  return pl.R[2] * (bx.p[0] - pl.p[0]) + pl.R[5] * (bx.p[1] - pl.p[1]) + pl.R[8] * (bx.p[2] - pl.p[2]) - Num<Real>::sqrt(dot3(s, s));
}
template <typename Real> UR3E_HD Real box_box_bound(const GeomPose<Real>& g1, const Real* s1, const GeomPose<Real>& g2, const Real* s2) {
  const Real d[3] = {g2.p[0] - g1.p[0], g2.p[1] - g1.p[1], g2.p[2] - g1.p[2]};
  return Num<Real>::sqrt(dot3(d, d)) - Num<Real>::sqrt(dot3(s1, s1)) - Num<Real>::sqrt(dot3(s2, s2));
}

// Rows of the arena's union u available to the overlapping path (after kinematics() its kinematics view is dead)
template <typename Real, typename D> constexpr int dist_rows() {
  constexpr int r = (int)(sizeof(Arena<Real, D>::u) / (sizeof(Real) * DIST_ROW_W));
  return r < 32 ? r : 32;
}

// The k pairs of table t for this warp's state (qpos loaded by the caller): dist [k], fromto [k][6], either may be null.
// Pass 1, lane = pair: a bounding-sphere / plane-height bound at distmax, the plane-box pairs, SAT, and the disjoint box pairs in
// registers; overlapping box pairs are marked.  Pass 2 ballot-compacts the marked pairs of each group of 32 into the staging rows
// laid over the union u, at most dist_rows() at a time, and runs box_box on them; a pair where box_box finds no point is sent
// back through pass 1 with the exact path forced.
template <typename Real, typename D>
UR3E_HD void distance_env(const DevModel<Real>& m, Arena<Real, D>& s, const DistPair<Real>* t, int k, Real distmax, Real* dist, Real* fromto) {
  constexpr int NROW = dist_rows<Real, D>();
  static_assert(NROW >= 1, "one staging row fits the arena's union u");
  kinematics(m, s);
  Real* const rows = reinterpret_cast<Real*>(&s.u);
  auto put = [&](int j, const DistPts<Real>& r) {
    const bool keep = r.d < distmax;
    if (dist) dist[j] = keep ? r.d : distmax;
    if (fromto) for (int c = 0; c < 3; ++c) { fromto[6 * j + c] = keep ? r.a[c] : Real(0); fromto[6 * j + 3 + c] = keep ? r.b[c] : Real(0); }
  };
  for (int base = 0; base < k; base += 32) {
    const int cnt = k - base < 32 ? k - base : 32;
    int todo = cnt == 32 ? -1 : (int)((1u << cnt) - 1u), forced = 0;
    while (todo) {
      int ovl = 0;
      WARP_FOR(i, cnt) {
        if ((todo >> i) & 1) {
          const int j = base + i;
          const DistPair<Real>& pr = t[j];
          const GeomPose<Real> g1 = geom_pose(s, pr.g[0].e), g2 = geom_pose(s, pr.g[1].e);
          const Real lb = pr.g[0].plane ? plane_box_bound(g1, g2, pr.g[1].size)
                          : pr.g[1].plane ? plane_box_bound(g2, g1, pr.g[0].size)
                                          : box_box_bound(g1, pr.g[0].size, g2, pr.g[1].size);
          DistPts<Real> r;
          if (lb >= distmax) { r.d = distmax; put(j, r); }
          else if (geom_distance_direct(g1, pr.g[0], g2, pr.g[1], ((forced >> i) & 1) != 0, r)) put(j, r);
          else ovl |= (int)(1u << i);
        }
      }
      ovl = warp_or(ovl);
      int back = 0;
      const int nov = popcount32(ovl);
      for (int r0 = 0; r0 < nov; r0 += NROW) {
        WARP_FOR(i, nov - r0 < NROW ? nov - r0 : NROW) {
          const int b = nth_set_bit(ovl, r0 + i), j = base + b;
          const DistPair<Real>& pr = t[j];
          const GeomPose<Real> g1 = geom_pose(s, pr.g[0].e), g2 = geom_pose(s, pr.g[1].e);
          DistPts<Real> r;
          if (box_box_contact(g1, pr.g[0], g2, pr.g[1], rows + i * DIST_ROW_W, r)) put(j, r);
          else back |= (int)(1u << b);
        }
        WARP_SYNC();
      }
      todo = forced = warp_or(back);
    }
  }
}

}  // namespace ur3e
