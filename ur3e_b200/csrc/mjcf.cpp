// C++ MJCF loader + model-constant pass (replaces MjModel.from_xml_path for the reference's
// scenes: reference utils/utils.py:9-12 -> assets/main.xml, ur3e_2f85.xml, ur3e_raw.xml).
// Supports exactly the MJCF subset those files use (SURVEY §7 step 1); anything else throws.
#include "host_model.h"
#include "xml_mini.h"

#include <cmath>
#include <cstring>
#include <fstream>
#include <set>
#include <sstream>

namespace ur3e {
namespace {

constexpr double kMinVal = 1e-15;
using Attr = std::map<std::string, std::string>;
using V = std::vector<double>;

[[noreturn]] void fail(const std::string& m) { throw std::runtime_error("mjcf: " + m); }

V floats(const Attr& a, const char* key, size_t n, const V& dflt) {
  V out;
  auto it = a.find(key);
  if (it != a.end()) { std::istringstream is(it->second); double x; while (is >> x) out.push_back(x); }
  for (size_t k = out.size(); k < n && k < dflt.size(); ++k) out.push_back(dflt[k]);
  if (n && out.size() < n) fail(std::string("attribute '") + key + "' needs " + std::to_string(n) + " numbers");
  if (n && out.size() > n) out.resize(n);
  return out;
}
double num(const Attr& a, const char* key, double dflt) { auto it = a.find(key); return it == a.end() ? dflt : std::stod(it->second); }
std::string str(const Attr& a, const char* key, const std::string& dflt = "") { auto it = a.find(key); return it == a.end() ? dflt : it->second; }
bool has(const Attr& a, const char* key) { return a.count(key) != 0; }

// ---- small rigid-body math (host, float64)
void quat_norm(double* q) { double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]); if (n < kMinVal) { q[0] = 1; q[1] = q[2] = q[3] = 0; } else for (int i = 0; i < 4; ++i) q[i] /= n; }
void quat_mul(double* r, const double* a, const double* b) {
  double t[4] = {a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                 a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]};
  std::memcpy(r, t, sizeof t);
}
void quat2mat(double* m, const double* q) {
  double w = q[0], x = q[1], y = q[2], z = q[3];
  m[0] = w * w + x * x - y * y - z * z; m[1] = 2 * (x * y - w * z); m[2] = 2 * (x * z + w * y);
  m[3] = 2 * (x * y + w * z); m[4] = w * w - x * x + y * y - z * z; m[5] = 2 * (y * z - w * x);
  m[6] = 2 * (x * z - w * y); m[7] = 2 * (y * z + w * x); m[8] = w * w - x * x - y * y + z * z;
}
void mat_vec(double* r, const double* m, const double* v) { double t[3] = {m[0] * v[0] + m[1] * v[1] + m[2] * v[2], m[3] * v[0] + m[4] * v[1] + m[5] * v[2], m[6] * v[0] + m[7] * v[1] + m[8] * v[2]}; std::memcpy(r, t, sizeof t); }
void matT_vec(double* r, const double* m, const double* v) { double t[3] = {m[0] * v[0] + m[3] * v[1] + m[6] * v[2], m[1] * v[0] + m[4] * v[1] + m[7] * v[2], m[2] * v[0] + m[5] * v[1] + m[8] * v[2]}; std::memcpy(r, t, sizeof t); }
void cross(double* r, const double* a, const double* b) { double t[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]}; std::memcpy(r, t, sizeof t); }

// ---- <default> class tree
struct Defaults {
  std::map<std::string, std::map<std::string, Attr>> cls;  // class -> tag -> attrs
  std::map<std::string, std::string> parent;
  Defaults() { cls["main"]; parent["main"] = ""; }
  void load(const XmlNode& e, const std::string& c) {
    for (auto& ch : e.children) {
      if (ch->tag == "default") {
        const std::string* n = ch->find("class");
        if (!n) fail("nested <default> without class");
        cls[*n]; parent[*n] = c; load(*ch, *n);
      } else {
        for (auto& kv : ch->attrs) cls[c][ch->tag][kv.first] = kv.second;
      }
    }
  }
  Attr resolve(const std::string& tag, const XmlNode& e, const std::string& childclass) const {
    std::string c = "main";
    if (const std::string* k = e.find("class")) c = *k; else if (!childclass.empty()) c = childclass;
    if (!cls.count(c)) fail("unknown default class '" + c + "'");
    std::vector<std::string> chain;
    for (std::string x = c; !x.empty(); x = parent.at(x)) chain.push_back(x);
    Attr out;
    for (auto it = chain.rbegin(); it != chain.rend(); ++it) {
      const auto& tags = cls.at(*it);
      if (tag == "motor") { auto g = tags.find("general"); if (g != tags.end()) for (auto& kv : g->second) out[kv.first] = kv.second; }
      auto t = tags.find(tag);
      if (t != tags.end()) for (auto& kv : t->second) out[kv.first] = kv.second;
    }
    for (auto& kv : e.attrs) out[kv.first] = kv.second;
    return out;
  }
};

const V kSolref = {0.02, 1.0};
const V kSolimp = {0.9, 0.95, 0.001, 0.5, 2.0};

struct Builder {
  HostModel m;
  Defaults dfl;
  bool autolimits = true;
  // body
  std::vector<std::string> bname; std::vector<int> bparent, bjntadr, bjntnum;
  V bpos, bquat, bipos, biquat, bmass, binertia;
  // joint
  std::vector<std::string> jname; std::vector<int> jtype, jbody, jlimited;
  V jpos, jaxis, jrange, jarm, jdamp, jfl, jstiff, jspringref, jref, jmargin, jsolref, jsolimp;
  // geom
  std::vector<std::string> gname; std::vector<int> gtype, gbody, gcontype, gconaff, gcondim, gprio;
  V gpos, gquat, gsize, gfriction, gsolref, gsolimp, gsolmix, gmargin, ggap, grgba;
  // site
  std::vector<std::string> sname; std::vector<int> sbody; V spos, squat, ssize;

  static void push(V& dst, const V& src) { dst.insert(dst.end(), src.begin(), src.end()); }

  int add_body(const XmlNode& e, int parent, const std::string& childclass) {
    int bid = (int)bname.size();
    Attr ba; for (auto& kv : e.attrs) ba[kv.first] = kv.second;
    bname.push_back(str(ba, "name", parent < 0 ? "world" : "body" + std::to_string(bid)));
    bparent.push_back(parent < 0 ? 0 : parent);
    push(bpos, floats(ba, "pos", 3, {0, 0, 0}));
    V q = floats(ba, "quat", 4, {1, 0, 0, 0}); quat_norm(q.data()); push(bquat, q);
    std::string cc = has(ba, "childclass") ? ba["childclass"] : childclass;
    bjntadr.push_back((int)jname.size());
    int nj = 0;
    struct GM { double mass; double pos[3]; double quat[4]; double I[3]; };
    std::vector<GM> gm;
    const XmlNode* inertial = nullptr;
    for (auto& chp : e.children) {
      const XmlNode& ch = *chp;
      if (ch.tag == "inertial") inertial = &ch;
      else if (ch.tag == "joint" || ch.tag == "freejoint") {
        Attr a;
        if (ch.tag == "joint") a = dfl.resolve("joint", ch, cc); else { for (auto& kv : ch.attrs) a[kv.first] = kv.second; a["type"] = "free"; }
        std::string t = str(a, "type", "hinge");
        int jt = t == "free" ? JNT_FREE : t == "hinge" ? JNT_HINGE : t == "slide" ? JNT_SLIDE : -1;
        if (jt < 0 || jt == JNT_SLIDE) fail("joint type '" + t + "' is not supported (hinge and free only)");
        jname.push_back(str(a, "name")); jtype.push_back(jt); jbody.push_back(bid);
        push(jpos, floats(a, "pos", 3, {0, 0, 0}));
        V ax = floats(a, "axis", 3, {0, 0, 1});
        double n = std::sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]); if (n < kMinVal) fail("zero joint axis"); for (auto& x : ax) x /= n;
        push(jaxis, ax);
        push(jrange, floats(a, "range", 2, {0, 0}));
        std::string lim = str(a, "limited", "auto");
        bool limited = lim == "true" || (lim == "auto" && autolimits && has(a, "range"));
        jlimited.push_back(limited && jt != JNT_FREE ? 1 : 0);
        jarm.push_back(num(a, "armature", 0)); jdamp.push_back(num(a, "damping", 0)); jfl.push_back(num(a, "frictionloss", 0));
        jstiff.push_back(num(a, "stiffness", 0)); jspringref.push_back(num(a, "springref", 0)); jref.push_back(num(a, "ref", 0));
        jmargin.push_back(num(a, "margin", 0));
        push(jsolref, floats(a, "solreflimit", 2, kSolref)); push(jsolimp, floats(a, "solimplimit", 5, kSolimp));
        ++nj;
      } else if (ch.tag == "geom") {
        Attr a = dfl.resolve("geom", ch, cc);
        std::string t = str(a, "type", "sphere");
        if (has(a, "mesh")) t = "mesh";
        if (t == "mesh") { m.warnings.push_back("mesh geom '" + str(a, "name") + "' on body '" + bname[bid] + "' ignored (no mesh collision / mesh mass)"); continue; }
        int gt = t == "plane" ? GEOM_PLANE : t == "box" ? GEOM_BOX : -1;
        if (gt < 0) fail("geom type '" + t + "' is not supported (plane, box; mesh ignored)");
        gname.push_back(str(a, "name")); gtype.push_back(gt); gbody.push_back(bid);
        V gp = floats(a, "pos", 3, {0, 0, 0}); V gq = floats(a, "quat", 4, {1, 0, 0, 0}); quat_norm(gq.data());
        push(gpos, gp); push(gquat, gq);
        V sz = floats(a, "size", 3, {0, 0, 0}); push(gsize, sz);
        gcontype.push_back((int)num(a, "contype", 1)); gconaff.push_back((int)num(a, "conaffinity", 1));
        gcondim.push_back((int)num(a, "condim", 3)); gprio.push_back((int)num(a, "priority", 0));
        push(gfriction, floats(a, "friction", 3, {1, 0.005, 0.0001}));
        push(gsolref, floats(a, "solref", 2, kSolref)); push(gsolimp, floats(a, "solimp", 5, kSolimp));
        gsolmix.push_back(num(a, "solmix", 1)); gmargin.push_back(num(a, "margin", 0)); ggap.push_back(num(a, "gap", 0));
        push(grgba, floats(a, "rgba", 4, {0.5, 0.5, 0.5, 1}));   // MuJoCo's default; offscreen rendering only
        if (gt == GEOM_BOX) {
          double vol = 8 * sz[0] * sz[1] * sz[2];
          double mass = has(a, "mass") ? num(a, "mass", 0) : num(a, "density", 1000) * vol;
          if (mass > 0) {
            GM g; g.mass = mass; std::memcpy(g.pos, gp.data(), 24); std::memcpy(g.quat, gq.data(), 32);
            g.I[0] = mass / 3 * (sz[1] * sz[1] + sz[2] * sz[2]); g.I[1] = mass / 3 * (sz[0] * sz[0] + sz[2] * sz[2]); g.I[2] = mass / 3 * (sz[0] * sz[0] + sz[1] * sz[1]);
            gm.push_back(g);
          }
        }
      } else if (ch.tag == "site") {
        Attr a = dfl.resolve("site", ch, cc);
        sname.push_back(str(a, "name")); sbody.push_back(bid);
        push(spos, floats(a, "pos", 3, {0, 0, 0}));
        V sq = floats(a, "quat", 4, {1, 0, 0, 0}); quat_norm(sq.data()); push(squat, sq);
        push(ssize, floats(a, "size", 3, {0.005, 0.005, 0.005}));   // MuJoCo's default site size; box sites give three half-sizes
      } else if (ch.tag == "body" || ch.tag == "light" || ch.tag == "camera") {
      } else fail("unsupported element <" + ch.tag + "> in body '" + bname[bid] + "'");
    }
    bjntnum.push_back(nj);
    if (nj > 1) fail("body '" + bname[bid] + "' has more than one joint (unsupported)");
    if (inertial) {
      Attr a; for (auto& kv : inertial->attrs) a[kv.first] = kv.second;
      if (!has(a, "mass") || !has(a, "diaginertia")) fail("<inertial> needs mass and diaginertia");
      bmass.push_back(num(a, "mass", 0)); push(bipos, floats(a, "pos", 3, {0, 0, 0}));
      V iq = floats(a, "quat", 4, {1, 0, 0, 0}); quat_norm(iq.data()); push(biquat, iq);
      push(binertia, floats(a, "diaginertia", 3, {}));
    } else if (!gm.empty()) {
      double mt = 0, com[3] = {0, 0, 0};
      for (auto& g : gm) { mt += g.mass; for (int k = 0; k < 3; ++k) com[k] += g.mass * g.pos[k]; }
      for (int k = 0; k < 3; ++k) com[k] /= mt;
      double I[9] = {0};
      for (auto& g : gm) {
        double R[9]; quat2mat(R, g.quat);
        double d[3] = {g.pos[0] - com[0], g.pos[1] - com[1], g.pos[2] - com[2]}, dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
        for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) {
          double v = 0; for (int k = 0; k < 3; ++k) v += R[3 * i + k] * g.I[k] * R[3 * j + k];
          I[3 * i + j] += v + g.mass * ((i == j ? dd : 0) - d[i] * d[j]);
        }
      }
      double off = std::fabs(I[1]) + std::fabs(I[2]) + std::fabs(I[5]);
      if (off > 1e-15) fail("body '" + bname[bid] + "': geom-derived inertia is not axis-aligned; add an explicit <inertial>");
      bmass.push_back(mt); push(bipos, {com[0], com[1], com[2]}); push(biquat, {1, 0, 0, 0}); push(binertia, {I[0], I[4], I[8]});
    } else {
      if (parent >= 0 && nj > 0) m.warnings.push_back("body '" + bname[bid] + "' has no mass");
      bmass.push_back(0); push(bipos, {0, 0, 0}); push(biquat, {1, 0, 0, 0}); push(binertia, {0, 0, 0});
    }
    for (auto& chp : e.children) if (chp->tag == "body") add_body(*chp, bid, cc);
    return bid;
  }
};

template <class T> int index_of(const std::vector<T>& v, const T& x, const char* what) {
  for (size_t i = 0; i < v.size(); ++i) if (v[i] == x) return (int)i;
  fail(std::string("unknown ") + what + " '" + x + "'");
}

void set_array(HostModel& m, const std::string& n, const V& v, std::vector<long long> shape) { auto& a = m.arr[n]; a.d = v; a.shape = shape; a.is_int = false; }
void set_array(HostModel& m, const std::string& n, const std::vector<int>& v, std::vector<long long> shape) { auto& a = m.arr[n]; a.i = v; a.shape = shape; a.is_int = true; }

// forward kinematics at qpos (host; used for the model-constant pass)
struct HostFK { V xpos, xquat, xmat, xipos, ximat, xanchor, xaxis; };
HostFK host_fk(const HostModel& m, const V& qpos) {
  HostFK f; int nb = m.nbody;
  f.xpos.assign(3 * nb, 0); f.xquat.assign(4 * nb, 0); f.xmat.assign(9 * nb, 0); f.xipos.assign(3 * nb, 0); f.ximat.assign(9 * nb, 0);
  f.xanchor.assign(3 * m.njnt + 3, 0); f.xaxis.assign(3 * m.njnt + 3, 0);
  const auto &par = m.I("body_parentid"), &ja = m.I("body_jntadr"), &jn = m.I("body_jntnum"), &jt = m.I("jnt_type"), &qa = m.I("jnt_qposadr");
  const auto &bp = m.D("body_pos"), &bq = m.D("body_quat"), &ip = m.D("body_ipos"), &iq = m.D("body_iquat"), &jp = m.D("jnt_pos"), &jax = m.D("jnt_axis"), &q0 = m.D("qpos0");
  f.xquat[0] = 1; quat2mat(&f.xmat[0], &f.xquat[0]); quat2mat(&f.ximat[0], &f.xquat[0]);
  for (int b = 1; b < nb; ++b) {
    int p = par[b]; double pos[3], quat[4];
    if (jn[b] == 1 && jt[ja[b]] == JNT_FREE) {
      int a = qa[ja[b]]; std::memcpy(pos, &qpos[a], 24); std::memcpy(quat, &qpos[a + 3], 32); quat_norm(quat);
      std::memcpy(&f.xanchor[3 * ja[b]], pos, 24); f.xaxis[3 * ja[b] + 2] = 1;
    } else {
      double v[3]; mat_vec(v, &f.xmat[9 * p], &bp[3 * b]);
      for (int k = 0; k < 3; ++k) pos[k] = f.xpos[3 * p + k] + v[k];
      quat_mul(quat, &f.xquat[4 * p], &bq[4 * b]);
      if (jn[b] == 1) {
        int j = ja[b]; double R[9], vec[3], anchor[3];
        quat2mat(R, quat); mat_vec(vec, R, &jp[3 * j]);
        for (int k = 0; k < 3; ++k) anchor[k] = pos[k] + vec[k];
        mat_vec(&f.xaxis[3 * j], R, &jax[3 * j]); std::memcpy(&f.xanchor[3 * j], anchor, 24);
        double ang = qpos[qa[j]] - q0[qa[j]], s = std::sin(ang / 2), ql[4] = {std::cos(ang / 2), jax[3 * j] * s, jax[3 * j + 1] * s, jax[3 * j + 2] * s};
        quat_mul(quat, quat, ql); quat2mat(R, quat); mat_vec(vec, R, &jp[3 * j]);
        for (int k = 0; k < 3; ++k) pos[k] = anchor[k] - vec[k];
      }
    }
    quat_norm(quat);
    std::memcpy(&f.xpos[3 * b], pos, 24); std::memcpy(&f.xquat[4 * b], quat, 32); quat2mat(&f.xmat[9 * b], quat);
    double v[3]; mat_vec(v, &f.xmat[9 * b], &ip[3 * b]);
    for (int k = 0; k < 3; ++k) f.xipos[3 * b + k] = pos[k] + v[k];
    double qi[4]; quat_mul(qi, quat, &iq[4 * b]); quat2mat(&f.ximat[9 * b], qi);
  }
  return f;
}

// world-frame point jacobian columns for the dof chain of `body` (3 x nv each)
void host_jac(const HostModel& m, const HostFK& f, const double* point, int body, V& jp, V& jr) {
  int nv = m.nv; jp.assign(3 * nv, 0); jr.assign(3 * nv, 0);
  const auto &par = m.I("body_parentid"), &ja = m.I("body_jntadr"), &jn = m.I("body_jntnum"), &jt = m.I("jnt_type"), &da = m.I("jnt_dofadr");
  for (int b = body; b > 0; b = par[b]) {
    if (jn[b] == 0) continue;
    int j = ja[b];
    if (jt[j] == JNT_FREE) {
      for (int i = 0; i < 3; ++i) jp[i * nv + da[j] + i] = 1;
      for (int i = 0; i < 3; ++i) {
        double ax[3] = {f.xmat[9 * b + i], f.xmat[9 * b + 3 + i], f.xmat[9 * b + 6 + i]}, r[3] = {point[0] - f.xpos[3 * b], point[1] - f.xpos[3 * b + 1], point[2] - f.xpos[3 * b + 2]}, c[3];
        cross(c, ax, r);
        for (int k = 0; k < 3; ++k) { jr[k * nv + da[j] + 3 + i] = ax[k]; jp[k * nv + da[j] + 3 + i] = c[k]; }
      }
    } else {
      const double* ax = &f.xaxis[3 * j]; double r[3] = {point[0] - f.xanchor[3 * j], point[1] - f.xanchor[3 * j + 1], point[2] - f.xanchor[3 * j + 2]}, c[3];
      cross(c, ax, r);
      for (int k = 0; k < 3; ++k) { jr[k * nv + da[j]] = ax[k]; jp[k * nv + da[j]] = c[k]; }
    }
  }
}

// dense symmetric solve helpers
bool chol(V& A, int n) {
  for (int j = 0; j < n; ++j) {
    double s = A[j * n + j]; for (int k = 0; k < j; ++k) s -= A[j * n + k] * A[j * n + k];
    if (!(s > 0)) return false;
    double d = std::sqrt(s); A[j * n + j] = d;
    for (int i = j + 1; i < n; ++i) { double t = A[i * n + j]; for (int k = 0; k < j; ++k) t -= A[i * n + k] * A[j * n + k]; A[i * n + j] = t / d; }
  }
  return true;
}
void chol_solve(const V& L, double* x, int n) {
  for (int i = 0; i < n; ++i) { double t = x[i]; for (int k = 0; k < i; ++k) t -= L[i * n + k] * x[k]; x[i] = t / L[i * n + i]; }
  for (int i = n - 1; i >= 0; --i) { double t = x[i]; for (int k = i + 1; k < n; ++k) t -= L[k * n + i] * x[k]; x[i] = t / L[i * n + i]; }
}

void set_const(HostModel& m) {
  // mj_setConst restated: connect anchors on body 2, dof/body/tendon invweight0, meaninertia, all at qpos0
  int nv = m.nv, nb = m.nbody;
  HostFK f = host_fk(m, m.D("qpos0"));
  auto& eqd = m.D("eq_data");
  for (int e = 0; e < m.neq; ++e) if (m.I("eq_type")[e] == EQ_CONNECT) {
    int b1 = m.I("eq_obj1id")[e], b2 = m.I("eq_obj2id")[e]; double v[3], p[3];
    mat_vec(v, &f.xmat[9 * b1], &eqd[11 * e]);
    for (int k = 0; k < 3; ++k) p[k] = f.xpos[3 * b1 + k] + v[k] - f.xpos[3 * b2 + k];
    matT_vec(&eqd[11 * e + 3], &f.xmat[9 * b2], p);
  }
  V M(nv * nv, 0.0), jp, jr;
  for (int b = 1; b < nb; ++b) {
    double mass = m.D("body_mass")[b]; const double* I = &m.D("body_inertia")[3 * b]; const double* R = &f.ximat[9 * b];
    if (mass <= 0 && I[0] <= 0) continue;
    host_jac(m, f, &f.xipos[3 * b], b, jp, jr);
    double Iw[9];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { double v = 0; for (int k = 0; k < 3; ++k) v += R[3 * i + k] * I[k] * R[3 * j + k]; Iw[3 * i + j] = v; }
    for (int a = 0; a < nv; ++a) for (int c = 0; c < nv; ++c) {
      double v = 0;
      for (int k = 0; k < 3; ++k) v += mass * jp[k * nv + a] * jp[k * nv + c];
      for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) v += jr[i * nv + a] * Iw[3 * i + j] * jr[j * nv + c];
      M[a * nv + c] += v;
    }
  }
  for (int i = 0; i < nv; ++i) M[i * nv + i] += m.D("dof_armature")[i];
  double tr = 0; for (int i = 0; i < nv; ++i) tr += M[i * nv + i];
  m.meaninertia = nv ? tr / nv : 1;
  V L = M;
  if (nv && !chol(L, nv)) fail("mass matrix at qpos0 is not positive definite (massless moving body?)");
  V Minv(nv * nv, 0.0);
  for (int c = 0; c < nv; ++c) { V col(nv, 0.0); col[c] = 1; chol_solve(L, col.data(), nv); for (int r = 0; r < nv; ++r) Minv[r * nv + c] = col[r]; }
  V biw(2 * nb, 0.0), diw(nv, 0.0), tiw(m.ntendon, 0.0);
  for (int b = 1; b < nb; ++b) {
    if (m.I("body_weldid")[b] == 0) continue;
    host_jac(m, f, &f.xipos[3 * b], b, jp, jr);
    double tp = 0, trr = 0;
    for (int r = 0; r < 3; ++r) for (int a = 0; a < nv; ++a) for (int c = 0; c < nv; ++c) { tp += jp[r * nv + a] * Minv[a * nv + c] * jp[r * nv + c]; trr += jr[r * nv + a] * Minv[a * nv + c] * jr[r * nv + c]; }
    biw[2 * b] = tp / 3; biw[2 * b + 1] = trr / 3;
  }
  for (int j = 0; j < m.njnt; ++j) {
    int da = m.I("jnt_dofadr")[j];
    if (m.I("jnt_type")[j] == JNT_FREE) {
      double a = 0, b = 0; for (int i = 0; i < 3; ++i) { a += Minv[(da + i) * nv + da + i]; b += Minv[(da + 3 + i) * nv + da + 3 + i]; }
      for (int i = 0; i < 3; ++i) { diw[da + i] = a / 3; diw[da + 3 + i] = b / 3; }
    } else diw[da] = Minv[da * nv + da];
  }
  for (int t = 0; t < m.ntendon; ++t) {
    V J(nv, 0.0);
    for (int w = m.I("tendon_adr")[t]; w < m.I("tendon_adr")[t] + m.I("tendon_num")[t]; ++w) J[m.I("jnt_dofadr")[m.I("wrap_jnt")[w]]] = m.D("wrap_coef")[w];
    double v = 0; for (int a = 0; a < nv; ++a) for (int c = 0; c < nv; ++c) v += J[a] * Minv[a * nv + c] * J[c];
    tiw[t] = v;
  }
  set_array(m, "body_invweight0", biw, {nb, 2}); set_array(m, "dof_invweight0", diw, {nv}); set_array(m, "tendon_invweight0", tiw, {m.ntendon});
  // per-geom / per-equality constraint weights, so that later model passes (fixed-body merging) cannot change them
  V giw(m.ngeom, 0.0), eiw(m.neq, 0.0);
  for (int g = 0; g < m.ngeom; ++g) giw[g] = biw[2 * m.I("geom_bodyid")[g]];
  for (int e = 0; e < m.neq; ++e) {
    int o1 = m.I("eq_obj1id")[e], o2 = m.I("eq_obj2id")[e];
    if (m.I("eq_type")[e] == EQ_CONNECT) eiw[e] = biw[2 * o1] + biw[2 * o2];
    else eiw[e] = diw[m.I("jnt_dofadr")[o1]] + (o2 >= 0 ? diw[m.I("jnt_dofadr")[o2]] : 0.0);
  }
  set_array(m, "geom_invweight0", giw, {m.ngeom}); set_array(m, "eq_invweight0", eiw, {m.neq});
}

}  // namespace

HostModel load_mjcf(const std::string& path) {
  std::ifstream in(path);
  if (!in) fail("cannot open '" + path + "'");
  std::stringstream ss; ss << in.rdbuf();
  std::string text = ss.str();
  std::unique_ptr<XmlNode> root;
  try { root = XmlParser(text).parse(); } catch (const std::exception& e) { fail(std::string(e.what()) + " in '" + path + "'"); }
  if (root->tag != "mujoco") fail("root element must be <mujoco>");
  Builder B; HostModel& m = B.m;
  if (const XmlNode* c = root->child("compiler")) {
    Attr a; for (auto& kv : c->attrs) a[kv.first] = kv.second;
    if (str(a, "angle", "degree") != "radian") fail("only <compiler angle=\"radian\"> models are supported");
    B.autolimits = str(a, "autolimits", "true") == "true";
  } else fail("missing <compiler angle=\"radian\">");
  if (const XmlNode* o = root->child("option")) {
    Attr a; for (auto& kv : o->attrs) a[kv.first] = kv.second;
    m.timestep = num(a, "timestep", 0.002); m.impratio = num(a, "impratio", 1);
    V g = floats(a, "gravity", 3, {0, 0, -9.81}); std::memcpy(m.gravity, g.data(), 24);
    std::string cone = str(a, "cone", "pyramidal"); m.cone_elliptic = cone == "elliptic";
    for (const char* k : {"integrator", "solver"}) if (has(a, k)) fail(std::string("<option ") + k + "> is not supported (Euler + Newton only)");
  }
  for (auto& ch : root->children) if (ch->tag == "default") B.dfl.load(*ch, "main");
  const XmlNode* wb = root->child("worldbody");
  if (!wb) fail("missing <worldbody>");
  B.add_body(*wb, -1, "");

  int nb = (int)B.bname.size(), nj = (int)B.jname.size(), ng = (int)B.gname.size(), ns = (int)B.sname.size();
  m.nbody = nb; m.njnt = nj; m.ngeom = ng; m.nsite = ns;
  m.names[OBJ_BODY] = B.bname; m.names[OBJ_JOINT] = B.jname; m.names[OBJ_GEOM] = B.gname; m.names[OBJ_SITE] = B.sname;
  std::vector<int> qadr, dadr; int nq = 0, nv = 0;
  for (int j = 0; j < nj; ++j) { qadr.push_back(nq); dadr.push_back(nv); nq += B.jtype[j] == JNT_FREE ? 7 : 1; nv += B.jtype[j] == JNT_FREE ? 6 : 1; }
  m.nq = nq; m.nv = nv;
  std::vector<int> bjadr = B.bjntadr; for (int b = 0; b < nb; ++b) if (B.bjntnum[b] == 0) bjadr[b] = -1;
  set_array(m, "body_parentid", B.bparent, {nb}); set_array(m, "body_jntadr", bjadr, {nb}); set_array(m, "body_jntnum", B.bjntnum, {nb});
  set_array(m, "body_pos", B.bpos, {nb, 3}); set_array(m, "body_quat", B.bquat, {nb, 4}); set_array(m, "body_ipos", B.bipos, {nb, 3});
  set_array(m, "body_iquat", B.biquat, {nb, 4}); set_array(m, "body_mass", B.bmass, {nb}); set_array(m, "body_inertia", B.binertia, {nb, 3});
  set_array(m, "jnt_type", B.jtype, {nj}); set_array(m, "jnt_bodyid", B.jbody, {nj}); set_array(m, "jnt_qposadr", qadr, {nj}); set_array(m, "jnt_dofadr", dadr, {nj});
  set_array(m, "jnt_pos", B.jpos, {nj, 3}); set_array(m, "jnt_axis", B.jaxis, {nj, 3}); set_array(m, "jnt_range", B.jrange, {nj, 2}); set_array(m, "jnt_limited", B.jlimited, {nj});
  set_array(m, "jnt_stiffness", B.jstiff, {nj}); set_array(m, "jnt_margin", B.jmargin, {nj}); set_array(m, "jnt_solref", B.jsolref, {nj, 2}); set_array(m, "jnt_solimp", B.jsolimp, {nj, 5});
  V qpos0(nq, 0.0), qspring(nq, 0.0), darm, ddamp, dfl; std::vector<int> dbody, djnt, dpar, bdofadr(nb, -1), bdofnum(nb, 0), lastdof(nb, -1);
  for (int j = 0; j < nj; ++j) {
    int b = B.jbody[j], nd = 1;
    if (B.jtype[j] == JNT_FREE) {
      for (int k = 0; k < 3; ++k) qpos0[qadr[j] + k] = B.bpos[3 * b + k];
      for (int k = 0; k < 4; ++k) qpos0[qadr[j] + 3 + k] = B.bquat[4 * b + k];
      for (int k = 0; k < 7; ++k) qspring[qadr[j] + k] = qpos0[qadr[j] + k];
      nd = 6;
    } else { qpos0[qadr[j]] = B.jref[j]; qspring[qadr[j]] = B.jspringref[j]; }
    for (int k = 0; k < nd; ++k) {
      int d = dadr[j] + k;
      if (bdofadr[b] < 0) bdofadr[b] = d;
      bdofnum[b]++;
      int par = -1;
      if (lastdof[b] >= 0) par = lastdof[b];
      else for (int a = B.bparent[b];; a = B.bparent[a]) { if (lastdof[a] >= 0) { par = lastdof[a]; break; } if (a == 0) break; }
      dpar.push_back(par); lastdof[b] = d; dbody.push_back(b); djnt.push_back(j);
      darm.push_back(B.jarm[j]); ddamp.push_back(B.jdamp[j]); dfl.push_back(B.jfl[j]);
    }
  }
  set_array(m, "qpos0", qpos0, {nq}); set_array(m, "qpos_spring", qspring, {nq});
  set_array(m, "dof_bodyid", dbody, {nv}); set_array(m, "dof_jntid", djnt, {nv}); set_array(m, "dof_parentid", dpar, {nv});
  set_array(m, "dof_armature", darm, {nv}); set_array(m, "dof_damping", ddamp, {nv}); set_array(m, "dof_frictionloss", dfl, {nv});
  V dsr, dsi; for (int i = 0; i < nv; ++i) { Builder::push(dsr, kSolref); Builder::push(dsi, kSolimp); }
  set_array(m, "dof_solref", dsr, {nv, 2}); set_array(m, "dof_solimp", dsi, {nv, 5});
  set_array(m, "body_dofadr", bdofadr, {nb}); set_array(m, "body_dofnum", bdofnum, {nb});
  std::vector<int> rootid(nb, 0), weldid(nb, 0);
  for (int b = 1; b < nb; ++b) { int p = B.bparent[b]; rootid[b] = p == 0 ? b : rootid[p]; weldid[b] = B.bjntnum[b] > 0 ? b : weldid[p]; }
  set_array(m, "body_rootid", rootid, {nb}); set_array(m, "body_weldid", weldid, {nb});
  set_array(m, "geom_type", B.gtype, {ng}); set_array(m, "geom_bodyid", B.gbody, {ng}); set_array(m, "geom_pos", B.gpos, {ng, 3});
  set_array(m, "geom_quat", B.gquat, {ng, 4}); set_array(m, "geom_size", B.gsize, {ng, 3}); set_array(m, "geom_contype", B.gcontype, {ng});
  set_array(m, "geom_conaffinity", B.gconaff, {ng}); set_array(m, "geom_condim", B.gcondim, {ng}); set_array(m, "geom_priority", B.gprio, {ng});
  set_array(m, "geom_friction", B.gfriction, {ng, 3}); set_array(m, "geom_solref", B.gsolref, {ng, 2}); set_array(m, "geom_solimp", B.gsolimp, {ng, 5});
  set_array(m, "geom_solmix", B.gsolmix, {ng}); set_array(m, "geom_margin", B.gmargin, {ng}); set_array(m, "geom_gap", B.ggap, {ng});
  set_array(m, "geom_rgba", B.grgba, {ng, 4});
  set_array(m, "site_bodyid", B.sbody, {ns}); set_array(m, "site_pos", B.spos, {ns, 3}); set_array(m, "site_quat", B.squat, {ns, 4}); set_array(m, "site_size", B.ssize, {ns, 3});

  // tendons (fixed)
  std::vector<std::string> tname; std::vector<int> tadr, tnum, wjnt; V wcoef;
  if (const XmlNode* t = root->child("tendon")) for (auto& fx : t->children) {
    if (fx->tag != "fixed") fail("only <tendon><fixed> is supported");
    const std::string* n = fx->find("name"); tname.push_back(n ? *n : ""); tadr.push_back((int)wjnt.size()); int c = 0;
    for (auto& jj : fx->children) if (jj->tag == "joint") {
      const std::string *jn = jj->find("joint"), *cf = jj->find("coef");
      if (!jn || !cf) fail("<fixed><joint> needs joint and coef");
      wjnt.push_back(index_of(B.jname, *jn, "joint")); wcoef.push_back(std::stod(*cf)); ++c;
    }
    tnum.push_back(c);
  }
  m.ntendon = (int)tname.size(); m.nwrap = (int)wjnt.size(); m.names[OBJ_TENDON] = tname;
  set_array(m, "tendon_adr", tadr, {m.ntendon}); set_array(m, "tendon_num", tnum, {m.ntendon}); set_array(m, "wrap_jnt", wjnt, {m.nwrap}); set_array(m, "wrap_coef", wcoef, {m.nwrap});

  // equality
  std::vector<int> etype, eo1, eo2; V edata, esolref, esolimp;
  if (const XmlNode* eq = root->child("equality")) for (auto& e : eq->children) {
    Attr a; for (auto& kv : e->attrs) a[kv.first] = kv.second;
    V data(11, 0.0);
    if (e->tag == "connect") {
      etype.push_back(EQ_CONNECT); eo1.push_back(index_of(B.bname, str(a, "body1"), "body"));
      eo2.push_back(has(a, "body2") ? index_of(B.bname, str(a, "body2"), "body") : 0);
      V an = floats(a, "anchor", 3, {}); std::memcpy(data.data(), an.data(), 24);
    } else if (e->tag == "joint") {
      etype.push_back(EQ_JOINT); eo1.push_back(index_of(B.jname, str(a, "joint1"), "joint"));
      eo2.push_back(has(a, "joint2") ? index_of(B.jname, str(a, "joint2"), "joint") : -1);
      V pc = floats(a, "polycoef", 5, {0, 1, 0, 0, 0}); std::memcpy(data.data(), pc.data(), 40);
    } else fail("equality <" + e->tag + "> is not supported (connect, joint)");
    Builder::push(edata, data); Builder::push(esolref, floats(a, "solref", 2, kSolref)); Builder::push(esolimp, floats(a, "solimp", 5, kSolimp));
  }
  m.neq = (int)etype.size();
  set_array(m, "eq_type", etype, {m.neq}); set_array(m, "eq_obj1id", eo1, {m.neq}); set_array(m, "eq_obj2id", eo2, {m.neq});
  set_array(m, "eq_data", edata, {m.neq, 11}); set_array(m, "eq_solref", esolref, {m.neq, 2}); set_array(m, "eq_solimp", esolimp, {m.neq, 5});

  // actuators
  std::vector<std::string> aname; std::vector<int> atrntype, atrnid, actrllim, afrclim; V again, abias, actrlr, afrcr, agear;
  if (const XmlNode* act = root->child("actuator")) for (auto& e : act->children) {
    if (e->tag != "motor" && e->tag != "general") fail("actuator <" + e->tag + "> is not supported (motor, general)");
    Attr a = B.dfl.resolve(e->tag, *e, "");
    aname.push_back(str(a, "name"));
    if (has(a, "joint")) { atrntype.push_back(TRN_JOINT); atrnid.push_back(index_of(B.jname, str(a, "joint"), "joint")); }
    else if (has(a, "tendon")) { atrntype.push_back(TRN_TENDON); atrnid.push_back(index_of(tname, str(a, "tendon"), "tendon")); }
    else fail("actuator needs joint or tendon transmission");
    if (e->tag == "motor") { again.push_back(1); Builder::push(abias, {0, 0, 0}); }
    else {
      again.push_back(floats(a, "gainprm", 1, {1})[0]);
      V bp = floats(a, "biasprm", 3, {0, 0, 0});
      if (str(a, "biastype", "none") != "affine") bp = {0, 0, 0};
      Builder::push(abias, bp);
    }
    Builder::push(actrlr, floats(a, "ctrlrange", 2, {0, 0})); Builder::push(afrcr, floats(a, "forcerange", 2, {0, 0}));
    std::string cl = str(a, "ctrllimited", "auto"), fl = str(a, "forcelimited", "auto");
    actrllim.push_back(cl == "true" || (cl == "auto" && B.autolimits && has(a, "ctrlrange")) ? 1 : 0);
    afrclim.push_back(fl == "true" || (fl == "auto" && B.autolimits && has(a, "forcerange")) ? 1 : 0);
    agear.push_back(floats(a, "gear", 1, {1})[0]);
  }
  m.nu = (int)aname.size(); m.names[OBJ_ACTUATOR] = aname;
  set_array(m, "actuator_trntype", atrntype, {m.nu}); set_array(m, "actuator_trnid", atrnid, {m.nu}); set_array(m, "actuator_gainprm", again, {m.nu});
  set_array(m, "actuator_biasprm", abias, {m.nu, 3}); set_array(m, "actuator_ctrlrange", actrlr, {m.nu, 2}); set_array(m, "actuator_ctrllimited", actrllim, {m.nu});
  set_array(m, "actuator_forcerange", afrcr, {m.nu, 2}); set_array(m, "actuator_forcelimited", afrclim, {m.nu}); set_array(m, "actuator_gear", agear, {m.nu});

  // collision pair candidates (SURVEY B.9 filter), explicit <pair>s override the mixing
  std::set<std::pair<int, int>> excl; std::map<std::pair<int, int>, Attr> expl; std::map<std::pair<int, int>, std::pair<int, int>> expl_order;
  if (const XmlNode* c = root->child("contact")) for (auto& e : c->children) {
    Attr a; for (auto& kv : e->attrs) a[kv.first] = kv.second;
    if (e->tag == "exclude") { int b1 = index_of(B.bname, str(a, "body1"), "body"), b2 = index_of(B.bname, str(a, "body2"), "body"); excl.insert({std::min(b1, b2), std::max(b1, b2)}); }
    else if (e->tag == "pair") {
      int g1 = -1, g2 = -1;
      for (int g = 0; g < ng; ++g) { if (B.gname[g] == str(a, "geom1")) g1 = g; if (B.gname[g] == str(a, "geom2")) g2 = g; }
      if (g1 < 0 || g2 < 0) { m.warnings.push_back("<pair " + str(a, "geom1") + "," + str(a, "geom2") + "> names a geom that is not in the model (mesh?) - skipped"); continue; }
      expl[{std::min(g1, g2), std::max(g1, g2)}] = a; expl_order[{std::min(g1, g2), std::max(g1, g2)}] = {g1, g2};
    }
  }
  std::vector<int> pg1, pg2, pcondim; V pfric, psolref, psolimp, pmargin, pgap;
  for (int g1 = 0; g1 < ng; ++g1) for (int g2 = g1 + 1; g2 < ng; ++g2) {
    int t1 = B.gtype[g1], t2 = B.gtype[g2];
    if (t1 == GEOM_PLANE && t2 == GEOM_PLANE) continue;
    int b1 = B.gbody[g1], b2 = B.gbody[g2];
    int a = g1, b = g2, condim; V fr, sr, si; double margin, gap;
    auto key = std::make_pair(g1, g2);
    const bool is_expl = expl.count(key) != 0;
    if (!is_expl) {
      int w1 = weldid[b1], w2 = weldid[b2];
      if (w1 == w2) continue;
      if (!((B.gcontype[g1] & B.gconaff[g2]) || (B.gcontype[g2] & B.gconaff[g1]))) continue;
      int pw1 = w1 != 0 ? weldid[B.bparent[w1]] : -1, pw2 = w2 != 0 ? weldid[B.bparent[w2]] : -1;
      if (w1 != 0 && w2 != 0 && (pw1 == w2 || pw2 == w1)) continue;
      if (excl.count({std::min(b1, b2), std::max(b1, b2)})) continue;
    }
    // contact parameters mixed from the two geoms (priority, else max friction / solmix-weighted solref, solimp)
    if (B.gprio[g1] != B.gprio[g2]) {
      int gw = B.gprio[g1] > B.gprio[g2] ? g1 : g2;
      fr = {B.gfriction[3 * gw], B.gfriction[3 * gw], B.gfriction[3 * gw + 1], B.gfriction[3 * gw + 2], B.gfriction[3 * gw + 2]};
      sr = {B.gsolref[2 * gw], B.gsolref[2 * gw + 1]}; si.assign(B.gsolimp.begin() + 5 * gw, B.gsolimp.begin() + 5 * gw + 5); condim = B.gcondim[gw];
    } else {
      double f[3]; for (int k = 0; k < 3; ++k) f[k] = std::max(B.gfriction[3 * g1 + k], B.gfriction[3 * g2 + k]);
      fr = {f[0], f[0], f[1], f[2], f[2]};
      double s1 = B.gsolmix[g1], s2 = B.gsolmix[g2], mix = (s1 + s2) > kMinVal ? s1 / (s1 + s2) : 0.5;
      for (int k = 0; k < 2; ++k) sr.push_back(mix * B.gsolref[2 * g1 + k] + (1 - mix) * B.gsolref[2 * g2 + k]);
      for (int k = 0; k < 5; ++k) si.push_back(mix * B.gsolimp[5 * g1 + k] + (1 - mix) * B.gsolimp[5 * g2 + k]);
      condim = std::max(B.gcondim[g1], B.gcondim[g2]);
    }
    margin = std::max(B.gmargin[g1], B.gmargin[g2]); gap = std::max(B.ggap[g1], B.ggap[g2]);
    if (is_expl) {
      // explicit <pair>: always tested (no filtering); attributes it leaves out are inferred from its geoms as above
      // (MuJoCo's compiler, mjCPair::Compile), the ones it sets override
      const Attr& at = expl[key]; a = expl_order[key].first; b = expl_order[key].second;
      if (has(at, "condim")) condim = (int)num(at, "condim", 3);
      if (has(at, "friction")) fr = floats(at, "friction", 5, fr);
      if (has(at, "solref")) sr = floats(at, "solref", 2, sr);
      if (has(at, "solimp")) si = floats(at, "solimp", 5, si);
      if (has(at, "margin")) margin = num(at, "margin", 0);
      if (has(at, "gap")) gap = num(at, "gap", 0);
    }
    if (condim != 3) fail("only condim=3 contacts are supported");
    if (B.gtype[b] == GEOM_PLANE) std::swap(a, b);  // plane first
    pg1.push_back(a); pg2.push_back(b); pcondim.push_back(condim);
    Builder::push(pfric, fr); Builder::push(psolref, sr); Builder::push(psolimp, si); pmargin.push_back(margin); pgap.push_back(gap);
  }
  m.npair = (int)pg1.size();
  set_array(m, "pair_geom1", pg1, {m.npair}); set_array(m, "pair_geom2", pg2, {m.npair}); set_array(m, "pair_condim", pcondim, {m.npair});
  set_array(m, "pair_friction", pfric, {m.npair, 5}); set_array(m, "pair_solref", psolref, {m.npair, 2}); set_array(m, "pair_solimp", psolimp, {m.npair, 5});
  set_array(m, "pair_margin", pmargin, {m.npair}); set_array(m, "pair_gap", pgap, {m.npair});

  // torque sensors (reference assets/main.xml:384-391): the sites they are attached to, in sensor order
  std::vector<int> tqsite;
  if (const XmlNode* sn = root->child("sensor")) for (auto& e : sn->children) if (e->tag == "torque") {
    Attr a; for (auto& kv : e->attrs) a[kv.first] = kv.second;
    tqsite.push_back(index_of(B.sname, str(a, "site"), "site"));
  }
  set_array(m, "sensor_torque_site", tqsite, {(long long)tqsite.size()});

  // keyframes
  std::vector<std::string> kname; V kqpos, kqvel;
  if (const XmlNode* kf = root->child("keyframe")) for (auto& e : kf->children) if (e->tag == "key") {
    Attr a; for (auto& kv : e->attrs) a[kv.first] = kv.second;
    kname.push_back(str(a, "name"));
    Builder::push(kqpos, has(a, "qpos") ? floats(a, "qpos", nq, qpos0) : qpos0);
    Builder::push(kqvel, has(a, "qvel") ? floats(a, "qvel", nv, V(nv, 0.0)) : V(nv, 0.0));
  }
  m.nkey = (int)kname.size(); m.names[OBJ_KEY] = kname;
  set_array(m, "key_qpos", kqpos, {m.nkey, nq}); set_array(m, "key_qvel", kqvel, {m.nkey, nv});

  set_const(m);
  return m;
}

}  // namespace ur3e
