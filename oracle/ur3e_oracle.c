/* ORACLE (test infrastructure, NOT product code) -- see ur3e_oracle.h for the header note.
 *
 * Scalar float64 restatement of mujoco==3.3.3 mj_forward / mj_step (reference
 * requirements.txt:58; call sites gymnasium_env/envs/ur3e_env2.py:83, controller/move_j.py:83)
 * for the feature subset the reference's three scenes use, following SURVEY App. B item by
 * item, plus the reference controllers (controller/controller_func.py).
 * Dense matrices everywhere (nv <= 20): only the mathematics is restated, not MuJoCo's
 * sparse storage.  Parity status: UNPINNED against a real MuJoCo build (header note).
 */
#include "ur3e_oracle.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define MINVAL 1e-15
#define MINIMP 0.0001
#define MAXIMP 0.9999
enum { JNT_FREE = 0, JNT_BALL = 1, JNT_SLIDE = 2, JNT_HINGE = 3 };
enum { GEOM_PLANE = 0, GEOM_BOX = 6 };
enum { EQ_CONNECT = 0, EQ_JOINT = 2 };
enum { TRN_JOINT = 0, TRN_TENDON = 3 };

/* ------------------------------------------------------------------ small math */
static double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static void cross3(double* r, const double* a, const double* b) {
  double x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
static double norm3(const double* a) { return sqrt(dot3(a, a)); }
static double normalize3(double* a) {
  double n = norm3(a);
  if (n < MINVAL) { a[0] = 1; a[1] = 0; a[2] = 0; } else { a[0] /= n; a[1] /= n; a[2] /= n; }
  return n;
}
static void normalize4(double* q) {
  double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < MINVAL) { q[0] = 1; q[1] = q[2] = q[3] = 0; } else { for (int i = 0; i < 4; i++) q[i] /= n; }
}
static void mul_quat(double* r, const double* a, const double* b) {
  double t[4] = {a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                 a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]};
  memcpy(r, t, sizeof t);
}
static void quat2mat(double* m, const double* q) {
  double w = q[0], x = q[1], y = q[2], z = q[3];
  m[0] = w * w + x * x - y * y - z * z; m[1] = 2 * (x * y - w * z); m[2] = 2 * (x * z + w * y);
  m[3] = 2 * (x * y + w * z); m[4] = w * w - x * x + y * y - z * z; m[5] = 2 * (y * z - w * x);
  m[6] = 2 * (x * z - w * y); m[7] = 2 * (y * z + w * x); m[8] = w * w - x * x - y * y + z * z;
}
static void rot_vec_quat(double* r, const double* v, const double* q) {
  double m[9]; quat2mat(m, q);
  double t[3] = {m[0] * v[0] + m[1] * v[1] + m[2] * v[2], m[3] * v[0] + m[4] * v[1] + m[5] * v[2], m[6] * v[0] + m[7] * v[1] + m[8] * v[2]};
  memcpy(r, t, sizeof t);
}
static void axis_angle2quat(double* q, const double* axis, double angle) {
  if (angle == 0) { q[0] = 1; q[1] = q[2] = q[3] = 0; return; }
  double s = sin(angle * 0.5); q[0] = cos(angle * 0.5); q[1] = axis[0] * s; q[2] = axis[1] * s; q[3] = axis[2] * s;
}
static void mat_vec3(double* r, const double* m, const double* v) {
  double t[3] = {m[0] * v[0] + m[1] * v[1] + m[2] * v[2], m[3] * v[0] + m[4] * v[1] + m[5] * v[2], m[6] * v[0] + m[7] * v[1] + m[8] * v[2]};
  memcpy(r, t, sizeof t);
}
static void matT_vec3(double* r, const double* m, const double* v) {
  double t[3] = {m[0] * v[0] + m[3] * v[1] + m[6] * v[2], m[1] * v[0] + m[4] * v[1] + m[7] * v[2], m[2] * v[0] + m[5] * v[1] + m[8] * v[2]};
  memcpy(r, t, sizeof t);
}
static void mat_mul3(double* r, const double* a, const double* b) {
  double t[9];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) t[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
  memcpy(r, t, sizeof t);
}
/* spatial vectors are [rotational(3); translational(3)] (MuJoCo convention) */
static void inert_com(double* res, const double* inert, const double* mat, const double* dif, double mass) {
  double t[9];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) t[3 * i + j] = mat[3 * i] * inert[0] * mat[3 * j] + mat[3 * i + 1] * inert[1] * mat[3 * j + 1] + mat[3 * i + 2] * inert[2] * mat[3 * j + 2];
  res[0] = t[0] + mass * (dif[1] * dif[1] + dif[2] * dif[2]);
  res[1] = t[4] + mass * (dif[0] * dif[0] + dif[2] * dif[2]);
  res[2] = t[8] + mass * (dif[0] * dif[0] + dif[1] * dif[1]);
  res[3] = t[1] - mass * dif[0] * dif[1]; res[4] = t[2] - mass * dif[0] * dif[2]; res[5] = t[5] - mass * dif[1] * dif[2];
  res[6] = mass * dif[0]; res[7] = mass * dif[1]; res[8] = mass * dif[2]; res[9] = mass;
}
static void mul_inert_vec(double* res, const double* i, const double* v) {
  double r[6];
  r[0] = i[0] * v[0] + i[3] * v[1] + i[4] * v[2] - i[8] * v[4] + i[7] * v[5];
  r[1] = i[3] * v[0] + i[1] * v[1] + i[5] * v[2] + i[8] * v[3] - i[6] * v[5];
  r[2] = i[4] * v[0] + i[5] * v[1] + i[2] * v[2] - i[7] * v[3] + i[6] * v[4];
  r[3] = i[8] * v[1] - i[7] * v[2] + i[9] * v[3];
  r[4] = i[6] * v[2] - i[8] * v[0] + i[9] * v[4];
  r[5] = i[7] * v[0] - i[6] * v[1] + i[9] * v[5];
  memcpy(res, r, sizeof r);
}
static void cross_motion(double* res, const double* vel, const double* v) {
  double r[6]; cross3(r, vel, v); double a[3], b[3]; cross3(a, vel, v + 3); cross3(b, vel + 3, v);
  r[3] = a[0] + b[0]; r[4] = a[1] + b[1]; r[5] = a[2] + b[2]; memcpy(res, r, sizeof r);
}
static void cross_force(double* res, const double* vel, const double* f) {
  double r[6], a[3], b[3]; cross3(a, vel, f); cross3(b, vel + 3, f + 3);
  r[0] = a[0] + b[0]; r[1] = a[1] + b[1]; r[2] = a[2] + b[2]; cross3(r + 3, vel, f + 3); memcpy(res, r, sizeof r);
}

/* dense Cholesky A = L L^T (lower, row-major n x n); returns 0 ok, -1 not PD */
static int chol_factor(double* L, const double* A, int n) {
  memcpy(L, A, sizeof(double) * n * n);
  for (int j = 0; j < n; j++) {
    double s = L[j * n + j];
    for (int k = 0; k < j; k++) s -= L[j * n + k] * L[j * n + k];
    if (!(s > MINVAL)) { s = MINVAL; }
    double d = sqrt(s); L[j * n + j] = d;
    for (int i = j + 1; i < n; i++) {
      double t = L[i * n + j];
      for (int k = 0; k < j; k++) t -= L[i * n + k] * L[j * n + k];
      L[i * n + j] = t / d;
    }
  }
  return 0;
}
static void chol_solve(const double* L, double* x, int n) {
  for (int i = 0; i < n; i++) { double t = x[i]; for (int k = 0; k < i; k++) t -= L[i * n + k] * x[k]; x[i] = t / L[i * n + i]; }
  for (int i = n - 1; i >= 0; i--) { double t = x[i]; for (int k = i + 1; k < n; k++) t -= L[k * n + i] * x[k]; x[i] = t / L[i * n + i]; }
}

/* ------------------------------------------------------------------ model / data plumbing */
static int sizes_of_int(const OModel* m, const char* n) {
#define S(name, expr) if (!strcmp(n, #name)) return (expr);
  S(body_parentid, m->nbody) S(body_rootid, m->nbody) S(body_weldid, m->nbody) S(body_jntadr, m->nbody) S(body_jntnum, m->nbody)
  S(body_dofadr, m->nbody) S(body_dofnum, m->nbody) S(jnt_type, m->njnt) S(jnt_bodyid, m->njnt) S(jnt_qposadr, m->njnt)
  S(jnt_dofadr, m->njnt) S(jnt_limited, m->njnt) S(dof_bodyid, m->nv) S(dof_jntid, m->nv) S(dof_parentid, m->nv)
  S(geom_type, m->ngeom) S(geom_bodyid, m->ngeom) S(site_bodyid, m->nsite) S(tendon_adr, m->ntendon) S(tendon_num, m->ntendon)
  S(wrap_jnt, m->nwrap) S(eq_type, m->neq) S(eq_obj1id, m->neq) S(eq_obj2id, m->neq) S(actuator_trntype, m->nu)
  S(actuator_trnid, m->nu) S(actuator_ctrllimited, m->nu) S(actuator_forcelimited, m->nu) S(pair_geom1, m->npair)
  S(pair_geom2, m->npair) S(pair_condim, m->npair)
  return -1;
}
static int sizes_of_dbl(const OModel* m, const char* n) {
  S(body_pos, 3 * m->nbody) S(body_quat, 4 * m->nbody) S(body_ipos, 3 * m->nbody) S(body_iquat, 4 * m->nbody) S(body_mass, m->nbody)
  S(body_inertia, 3 * m->nbody) S(body_invweight0, 2 * m->nbody) S(jnt_pos, 3 * m->njnt) S(jnt_axis, 3 * m->njnt) S(jnt_range, 2 * m->njnt)
  S(jnt_stiffness, m->njnt) S(jnt_margin, m->njnt) S(jnt_solref, 2 * m->njnt) S(jnt_solimp, 5 * m->njnt) S(qpos0, m->nq) S(qpos_spring, m->nq)
  S(dof_armature, m->nv) S(dof_damping, m->nv) S(dof_frictionloss, m->nv) S(dof_invweight0, m->nv) S(dof_solref, 2 * m->nv) S(dof_solimp, 5 * m->nv)
  S(geom_pos, 3 * m->ngeom) S(geom_quat, 4 * m->ngeom) S(geom_size, 3 * m->ngeom) S(site_pos, 3 * m->nsite) S(site_quat, 4 * m->nsite)
  S(wrap_coef, m->nwrap) S(tendon_invweight0, m->ntendon) S(eq_data, 11 * m->neq) S(eq_solref, 2 * m->neq) S(eq_solimp, 5 * m->neq)
  S(actuator_gainprm, m->nu) S(actuator_biasprm, 3 * m->nu) S(actuator_ctrlrange, 2 * m->nu) S(actuator_forcerange, 2 * m->nu) S(actuator_gear, m->nu)
  S(pair_friction, 5 * m->npair) S(pair_solref, 2 * m->npair) S(pair_solimp, 5 * m->npair) S(pair_margin, m->npair) S(pair_gap, m->npair)
  S(key_qpos, m->nq * m->nkey) S(key_qvel, m->nv * m->nkey)
#undef S
  return -1;
}

OModel* o_model_new(const int* s, const double* opt) {
  OModel* m = (OModel*)calloc(1, sizeof(OModel));
  m->nq = s[0]; m->nv = s[1]; m->nu = s[2]; m->nbody = s[3]; m->njnt = s[4]; m->ngeom = s[5]; m->nsite = s[6];
  m->neq = s[7]; m->ntendon = s[8]; m->nwrap = s[9]; m->npair = s[10]; m->nkey = s[11];
  m->timestep = opt[0]; m->gravity[0] = opt[1]; m->gravity[1] = opt[2]; m->gravity[2] = opt[3]; m->impratio = opt[4];
  m->tolerance = opt[5]; m->ls_tolerance = opt[6]; m->cone_elliptic = (int)opt[7]; m->iterations = (int)opt[8]; m->ls_iterations = (int)opt[9];
#define X(n) { int c = sizes_of_int(m, #n); m->n = (int*)calloc(c > 0 ? c : 1, sizeof(int)); }
  O_MODEL_INT_FIELDS(X)
#undef X
#define X(n) { int c = sizes_of_dbl(m, #n); m->n = (double*)calloc(c > 0 ? c : 1, sizeof(double)); }
  O_MODEL_DBL_FIELDS(X)
#undef X
  return m;
}
int o_model_set_int(OModel* m, const char* name, const int* src, int n) {
#define X(f) if (!strcmp(name, #f)) { if (n != sizes_of_int(m, #f)) return -2; memcpy(m->f, src, sizeof(int) * n); return 0; }
  O_MODEL_INT_FIELDS(X)
#undef X
  return -1;
}
int o_model_set_dbl(OModel* m, const char* name, const double* src, int n) {
#define X(f) if (!strcmp(name, #f)) { if (n != sizes_of_dbl(m, #f)) return -2; memcpy(m->f, src, sizeof(double) * n); return 0; }
  O_MODEL_DBL_FIELDS(X)
#undef X
  return -1;
}
int o_model_get_dbl(OModel* m, const char* name, double** ptr) {
#define X(f) if (!strcmp(name, #f)) { *ptr = m->f; return sizes_of_dbl(m, #f); }
  O_MODEL_DBL_FIELDS(X)
#undef X
  return -1;
}
void o_model_free(OModel* m) {
#define X(n) free(m->n);
  O_MODEL_INT_FIELDS(X) O_MODEL_DBL_FIELDS(X)
#undef X
  free(m);
}
double o_model_meaninertia(const OModel* m) { return m->meaninertia; }

OData* o_data_new(const OModel* m) {
  OData* d = (OData*)calloc(1, sizeof(OData));
#define X(n, c) d->n = (double*)calloc((c) > 0 ? (c) : 1, sizeof(double));
  O_DATA_DBL_FIELDS(X)
#undef X
#define X(n, c) d->n = (int*)calloc((c) > 0 ? (c) : 1, sizeof(int));
  O_DATA_INT_FIELDS(X)
#undef X
  o_reset_data(m, d);
  return d;
}
void o_data_free(OData* d) {
#define X(n, c) free(d->n);
  O_DATA_DBL_FIELDS(X) O_DATA_INT_FIELDS(X)
#undef X
  free(d);
}
int o_data_get_dbl(const OModel* m, OData* d, const char* name, double** ptr, int* n) {
#define X(f, c) if (!strcmp(name, #f)) { *ptr = d->f; *n = (c); return 0; }
  O_DATA_DBL_FIELDS(X)
#undef X
  return -1;
}
int o_data_get_int(const OModel* m, OData* d, const char* name, int** ptr, int* n) {
  (void)m;
#define X(f, c) if (!strcmp(name, #f)) { *ptr = d->f; *n = (c); return 0; }
  O_DATA_INT_FIELDS(X)
#undef X
  return -1;
}
OContact* o_data_contacts(OData* d) { return d->contact; }
int o_data_info(OData* d, int w) {
  switch (w) { case 0: return d->ncon; case 1: return d->nefc; case 2: return d->solver_iter; case 3: return d->warn_bad;
    case 4: return d->ne; case 5: return d->nf; case 6: return d->nl; } return -1;
}
double o_data_time(OData* d) { return d->time; }

void o_reset_data(const OModel* m, OData* d) {
  /* mj_resetData: qpos = qpos0, everything else zero */
#define X(n, c) memset(d->n, 0, sizeof(double) * ((c) > 0 ? (c) : 1));
  O_DATA_DBL_FIELDS(X)
#undef X
  memcpy(d->qpos, m->qpos0, sizeof(double) * m->nq);
  d->time = 0; d->ncon = d->nefc = d->solver_iter = d->warn_bad = d->ne = d->nf = d->nl = 0; d->solver_cost = 0;
}

/* ------------------------------------------------------------------ position stage */
static void kinematics(const OModel* m, OData* d) {
  /* SURVEY B.1 (mj_kinematics) */
  for (int j = 0; j < m->njnt; j++) if (m->jnt_type[j] == JNT_FREE) normalize4(d->qpos + m->jnt_qposadr[j] + 3);
  double* xp = d->xpos; double* xq = d->xquat;
  xp[0] = xp[1] = xp[2] = 0; xq[0] = 1; xq[1] = xq[2] = xq[3] = 0; quat2mat(d->xmat, xq);
  memcpy(d->xipos, xp, 24); quat2mat(d->ximat, xq);
  for (int b = 1; b < m->nbody; b++) {
    int p = m->body_parentid[b];
    double pos[3], quat[4];
    int jn = m->body_jntnum[b], ja = m->body_jntadr[b];
    if (jn == 1 && m->jnt_type[ja] == JNT_FREE) {
      int qa = m->jnt_qposadr[ja];
      memcpy(pos, d->qpos + qa, 24); memcpy(quat, d->qpos + qa + 3, 32);
      memcpy(d->xanchor + 3 * ja, pos, 24); d->xaxis[3 * ja] = 0; d->xaxis[3 * ja + 1] = 0; d->xaxis[3 * ja + 2] = 1;
    } else {
      double v[3]; mat_vec3(v, d->xmat + 9 * p, m->body_pos + 3 * b);
      for (int k = 0; k < 3; k++) pos[k] = d->xpos[3 * p + k] + v[k];
      mul_quat(quat, d->xquat + 4 * p, m->body_quat + 4 * b);
      for (int j = ja; j < ja + jn; j++) {
        int qa = m->jnt_qposadr[j];
        double anchor[3], vec[3];
        rot_vec_quat(vec, m->jnt_pos + 3 * j, quat);
        for (int k = 0; k < 3; k++) anchor[k] = pos[k] + vec[k];
        rot_vec_quat(d->xaxis + 3 * j, m->jnt_axis + 3 * j, quat);
        memcpy(d->xanchor + 3 * j, anchor, 24);
        if (m->jnt_type[j] == JNT_HINGE) {
          double ql[4]; axis_angle2quat(ql, m->jnt_axis + 3 * j, d->qpos[qa] - m->qpos0[qa]);
          mul_quat(quat, quat, ql);
          rot_vec_quat(vec, m->jnt_pos + 3 * j, quat);
          for (int k = 0; k < 3; k++) pos[k] = anchor[k] - vec[k];
        } else if (m->jnt_type[j] == JNT_SLIDE) {
          for (int k = 0; k < 3; k++) pos[k] += d->xaxis[3 * j + k] * (d->qpos[qa] - m->qpos0[qa]);
        }
      }
    }
    normalize4(quat);
    memcpy(d->xpos + 3 * b, pos, 24); memcpy(d->xquat + 4 * b, quat, 32); quat2mat(d->xmat + 9 * b, quat);
    double v[3]; mat_vec3(v, d->xmat + 9 * b, m->body_ipos + 3 * b);
    for (int k = 0; k < 3; k++) d->xipos[3 * b + k] = pos[k] + v[k];
    double qi[4]; mul_quat(qi, quat, m->body_iquat + 4 * b); quat2mat(d->ximat + 9 * b, qi);
  }
  for (int g = 0; g < m->ngeom; g++) {
    int b = m->geom_bodyid[g]; double v[3], q[4];
    mat_vec3(v, d->xmat + 9 * b, m->geom_pos + 3 * g);
    for (int k = 0; k < 3; k++) d->geom_xpos[3 * g + k] = d->xpos[3 * b + k] + v[k];
    mul_quat(q, d->xquat + 4 * b, m->geom_quat + 4 * g); quat2mat(d->geom_xmat + 9 * g, q);
  }
  for (int s = 0; s < m->nsite; s++) {
    int b = m->site_bodyid[s]; double v[3], q[4];
    mat_vec3(v, d->xmat + 9 * b, m->site_pos + 3 * s);
    for (int k = 0; k < 3; k++) d->site_xpos[3 * s + k] = d->xpos[3 * b + k] + v[k];
    mul_quat(q, d->xquat + 4 * b, m->site_quat + 4 * s); quat2mat(d->site_xmat + 9 * s, q);
  }
}

static void com_pos(const OModel* m, OData* d) {
  /* SURVEY B.2 (mj_comPos): subtree COM, cinert, cdof about the tree root's subtree COM */
  int nb = m->nbody;
  double* mass = (double*)calloc(nb, sizeof(double));
  for (int b = 0; b < nb; b++) { mass[b] = m->body_mass[b]; for (int k = 0; k < 3; k++) d->subtree_com[3 * b + k] = m->body_mass[b] * d->xipos[3 * b + k]; }
  for (int b = nb - 1; b > 0; b--) { int p = m->body_parentid[b]; mass[p] += mass[b]; for (int k = 0; k < 3; k++) d->subtree_com[3 * p + k] += d->subtree_com[3 * b + k]; }
  for (int b = 0; b < nb; b++) {
    if (mass[b] < MINVAL) memcpy(d->subtree_com + 3 * b, d->xipos + 3 * b, 24);
    else for (int k = 0; k < 3; k++) d->subtree_com[3 * b + k] /= mass[b];
  }
  free(mass);
  memset(d->cinert, 0, sizeof(double) * 10);
  for (int b = 1; b < nb; b++) {
    double off[3]; const double* com = d->subtree_com + 3 * m->body_rootid[b];
    for (int k = 0; k < 3; k++) off[k] = d->xipos[3 * b + k] - com[k];
    inert_com(d->cinert + 10 * b, m->body_inertia + 3 * b, d->ximat + 9 * b, off, m->body_mass[b]);
  }
  for (int j = 0; j < m->njnt; j++) {
    int b = m->jnt_bodyid[j], da = m->jnt_dofadr[j];
    double off[3]; const double* com = d->subtree_com + 3 * m->body_rootid[b];
    for (int k = 0; k < 3; k++) off[k] = com[k] - d->xanchor[3 * j + k];
    if (m->jnt_type[j] == JNT_FREE) {
      memset(d->cdof + 6 * da, 0, sizeof(double) * 18);
      for (int i = 0; i < 3; i++) d->cdof[6 * (da + i) + 3 + i] = 1;
      for (int i = 0; i < 3; i++) {
        double ax[3] = {d->xmat[9 * b + i], d->xmat[9 * b + 3 + i], d->xmat[9 * b + 6 + i]};
        double* c = d->cdof + 6 * (da + 3 + i); memcpy(c, ax, 24); cross3(c + 3, ax, off);
      }
    } else if (m->jnt_type[j] == JNT_HINGE) {
      double* c = d->cdof + 6 * da; memcpy(c, d->xaxis + 3 * j, 24); cross3(c + 3, d->xaxis + 3 * j, off);
    } else { /* slide */
      double* c = d->cdof + 6 * da; c[0] = c[1] = c[2] = 0; memcpy(c + 3, d->xaxis + 3 * j, 24);
    }
  }
}

static void tendon(const OModel* m, OData* d) {
  for (int t = 0; t < m->ntendon; t++) {
    d->ten_length[t] = 0; memset(d->ten_J + t * m->nv, 0, sizeof(double) * m->nv);
    for (int w = m->tendon_adr[t]; w < m->tendon_adr[t] + m->tendon_num[t]; w++) {
      int j = m->wrap_jnt[w];
      d->ten_length[t] += m->wrap_coef[w] * d->qpos[m->jnt_qposadr[j]];
      d->ten_J[t * m->nv + m->jnt_dofadr[j]] = m->wrap_coef[w];
    }
  }
}

static void crb(const OModel* m, OData* d) {
  /* SURVEY B.3 (mj_crb): composite inertias, M_ij = cdof_j . (crb_body(i) cdof_i), + armature */
  int nv = m->nv;
  memcpy(d->crb, d->cinert, sizeof(double) * 10 * m->nbody);
  for (int b = m->nbody - 1; b > 0; b--) { int p = m->body_parentid[b]; if (p > 0) for (int k = 0; k < 10; k++) d->crb[10 * p + k] += d->crb[10 * b + k]; }
  memset(d->qM, 0, sizeof(double) * nv * nv);
  for (int i = 0; i < nv; i++) {
    double buf[6]; mul_inert_vec(buf, d->crb + 10 * m->dof_bodyid[i], d->cdof + 6 * i);
    d->qM[i * nv + i] = m->dof_armature[i];
    for (int j = i; j >= 0; j = m->dof_parentid[j]) {
      double v = 0; for (int k = 0; k < 6; k++) v += d->cdof[6 * j + k] * buf[k];
      d->qM[i * nv + j] += v; if (j != i) d->qM[j * nv + i] = d->qM[i * nv + j];
    }
  }
}

void o_fullM(const OModel* m, const OData* d, double* dst) { memcpy(dst, d->qM, sizeof(double) * m->nv * m->nv); }

/* jacobian of a world point attached to body (mj_jac): jacp/jacr are 3 x nv, may be NULL */
void o_jac(const OModel* m, const OData* d, double* jacp, double* jacr, const double* point, int body) {
  int nv = m->nv;
  if (jacp) memset(jacp, 0, sizeof(double) * 3 * nv);
  if (jacr) memset(jacr, 0, sizeof(double) * 3 * nv);
  while (body > 0 && m->body_dofnum[body] == 0) body = m->body_parentid[body];
  if (body <= 0) return;
  double off[3]; const double* com = d->subtree_com + 3 * m->body_rootid[body];
  for (int k = 0; k < 3; k++) off[k] = point[k] - com[k];
  int i = m->body_dofadr[body] + m->body_dofnum[body] - 1;
  while (i >= 0) {
    const double* c = d->cdof + 6 * i;
    if (jacr) for (int k = 0; k < 3; k++) jacr[k * nv + i] = c[k];
    if (jacp) { double t[3]; cross3(t, c, off); for (int k = 0; k < 3; k++) jacp[k * nv + i] = c[3 + k] + t[k]; }
    i = m->dof_parentid[i];
  }
}
void o_jac_site(const OModel* m, const OData* d, double* jacp, double* jacr, int site) {
  o_jac(m, d, jacp, jacr, d->site_xpos + 3 * site, m->site_bodyid[site]);
}
void o_object_velocity_site(const OModel* m, const OData* d, int site, double* res, int flg_local) {
  /* mj_objectVelocity(mjOBJ_SITE): [omega; v at the site point] */
  int b = m->site_bodyid[site];
  const double* cv = d->cvel + 6 * b; const double* com = d->subtree_com + 3 * m->body_rootid[b];
  double off[3], t[3];
  for (int k = 0; k < 3; k++) off[k] = d->site_xpos[3 * site + k] - com[k];
  cross3(t, cv, off);
  double w[3] = {cv[0], cv[1], cv[2]}, v[3] = {cv[3] + t[0], cv[4] + t[1], cv[5] + t[2]};
  if (flg_local) { matT_vec3(res, d->site_xmat + 9 * site, w); matT_vec3(res + 3, d->site_xmat + 9 * site, v); }
  else { memcpy(res, w, 24); memcpy(res + 3, v, 24); }
}

/* ------------------------------------------------------------------ collision (SURVEY B.9) */
static void make_frame(double* f) {
  normalize3(f);
  double* y = f + 3;
  y[0] = y[1] = y[2] = 0;
  if (f[1] < 0.5 && f[1] > -0.5) y[1] = 1; else y[2] = 1;
  double t = dot3(f, y); for (int k = 0; k < 3; k++) y[k] -= t * f[k];
  normalize3(y); cross3(f + 6, f, y);
}

static int plane_box(const double* ppos, const double* pmat, const double* bpos, const double* bmat, const double* size,
                     double margin, double* dist, double* pos, double* normal) {
  /* mjc_PlaneBox: corners below the plane (and not pointing up), first 4 in corner-index order */
  double n[3] = {pmat[2], pmat[5], pmat[8]}, dif[3];
  for (int k = 0; k < 3; k++) dif[k] = bpos[k] - ppos[k];
  double cd = dot3(dif, n); int cnt = 0;
  for (int i = 0; i < 8; i++) {
    double v[3] = {(i & 1 ? size[0] : -size[0]), (i & 2 ? size[1] : -size[1]), (i & 4 ? size[2] : -size[2])}, c[3];
    mat_vec3(c, bmat, v);
    double ld = dot3(n, c);
    if (cd + ld > margin || ld > 0) continue;
    dist[cnt] = cd + ld;
    for (int k = 0; k < 3; k++) { pos[3 * cnt + k] = c[k] + bpos[k] - n[k] * dist[cnt] * 0.5; normal[3 * cnt + k] = n[k]; }
    if (++cnt >= 4) break;
  }
  return cnt;
}

/* clip polygon (2-D points) against half-plane  a*x + b*y <= c */
static int clip_poly(double* px, double* py, int n, double a, double b, double c) {
  double ox[16], oy[16]; int k = 0;
  for (int i = 0; i < n; i++) {
    int j = (i + 1) % n;
    double di = a * px[i] + b * py[i] - c, dj = a * px[j] + b * py[j] - c;
    if (di <= 0) { ox[k] = px[i]; oy[k] = py[i]; k++; }
    if ((di < 0 && dj > 0) || (di > 0 && dj < 0)) { double t = di / (di - dj); ox[k] = px[i] + t * (px[j] - px[i]); oy[k] = py[i] + t * (py[j] - py[i]); k++; }
    if (k >= 15) break;
  }
  memcpy(px, ox, sizeof(double) * k); memcpy(py, oy, sizeof(double) * k);
  return k;
}

#define EDGE_END_SLACK 1e-5   /* csrc/engine.cuh EDGE_END_SLACK */
static int box_box(const double* p1, const double* R1, const double* s1, const double* p2, const double* R2, const double* s2,
                   double margin, double* dist, double* pos, double* normal) {
  /* This repo's box-box manifold (stands in for mjc_BoxBox, whose exact point selection is not
   * reproducible from memory, SURVEY hard-part 4): 15-axis SAT -> face case: incident face clipped
   * against the reference face's side planes, points kept where depth > -margin, contact at
   * mid-penetration; edge case: closest points of the two edges.  Normal points from box1 to box2.
   * The edge case stands only when the closest points lie within both edges (up to EDGE_END_SLACK): outside them the edge-edge
   * axis was degenerate (nearly parallel edges, or an axis within rounding of a face normal) and the face case decides.
   * Kernel (csrc/engine.cuh box_box) implements the same rules. */
  double d[3], A1[3][3], A2[3][3];
  for (int k = 0; k < 3; k++) d[k] = p2[k] - p1[k];
  for (int i = 0; i < 3; i++) for (int k = 0; k < 3; k++) { A1[i][k] = R1[3 * k + i]; A2[i][k] = R2[3 * k + i]; } /* axis i = column i */
  double C[3][3], AC[3][3];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { C[i][j] = dot3(A1[i], A2[j]); AC[i][j] = fabs(C[i][j]); }
  double best = -1e30; int code = -1; double bn[3] = {0, 0, 0};
  /* face axes of box1, then box2 */
  for (int i = 0; i < 3; i++) {
    double t = dot3(d, A1[i]); double ra = s1[i], rb = s2[0] * AC[i][0] + s2[1] * AC[i][1] + s2[2] * AC[i][2];
    double sep = fabs(t) - ra - rb;
    if (sep > margin) return 0;
    if (sep > best) { best = sep; code = i; double sg = t < 0 ? -1 : 1; for (int k = 0; k < 3; k++) bn[k] = sg * A1[i][k]; }
  }
  for (int j = 0; j < 3; j++) {
    double t = dot3(d, A2[j]); double ra = s1[0] * AC[0][j] + s1[1] * AC[1][j] + s1[2] * AC[2][j], rb = s2[j];
    double sep = fabs(t) - ra - rb;
    if (sep > margin) return 0;
    if (sep > best + 1e-6 * (s1[0] + s1[1] + s1[2])) { best = sep; code = 3 + j; double sg = t < 0 ? -1 : 1; for (int k = 0; k < 3; k++) bn[k] = sg * A2[j][k]; }
  }
  /* edge-edge axes: only win when clearly better than the best face axis */
  double ebest = -1e30; int ei = -1, ej = -1; double en[3] = {0, 0, 0};
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) {
    double ax[3]; cross3(ax, A1[i], A2[j]);
    double l = norm3(ax); if (l < 1e-6) continue;
    for (int k = 0; k < 3; k++) ax[k] /= l;
    double t = dot3(d, ax);
    double ra = 0, rb = 0;
    for (int k = 0; k < 3; k++) { ra += s1[k] * fabs(dot3(A1[k], ax)); rb += s2[k] * fabs(dot3(A2[k], ax)); }
    double sep = fabs(t) - ra - rb;
    if (sep > margin) return 0;
    if (sep > ebest) { ebest = sep; ei = i; ej = j; double sg = t < 0 ? -1 : 1; for (int k = 0; k < 3; k++) en[k] = sg * ax[k]; }
  }
  if (ei >= 0 && ebest > best + 1e-3 * fabs(best) + 1e-9) {
    /* edge-edge: pick the supporting edges, closest points between the two lines */
    double c1[3], c2[3];
    for (int k = 0; k < 3; k++) { c1[k] = p1[k]; c2[k] = p2[k]; }
    for (int a = 0; a < 3; a++) if (a != ei) { double sg = dot3(A1[a], en) > 0 ? 1 : -1; for (int k = 0; k < 3; k++) c1[k] += sg * s1[a] * A1[a][k]; }
    for (int a = 0; a < 3; a++) if (a != ej) { double sg = dot3(A2[a], en) > 0 ? -1 : 1; for (int k = 0; k < 3; k++) c2[k] += sg * s2[a] * A2[a][k]; }
    const double* u = A1[ei]; const double* v = A2[ej];
    double w[3]; for (int k = 0; k < 3; k++) w[k] = c1[k] - c2[k];
    double b = dot3(u, v), dd = dot3(u, w), e = dot3(v, w), den = 1 - b * b;
    double sa = (b * e - dd) / den, sb = (e - b * dd) / den;
    /* a real edge-edge contact meets within both edges; otherwise the axis was degenerate and the face case decides */
    if (fabs(sa) <= s1[ei] * (1 + EDGE_END_SLACK) && fabs(sb) <= s2[ej] * (1 + EDGE_END_SLACK)) {
      if (sa > s1[ei]) sa = s1[ei]; if (sa < -s1[ei]) sa = -s1[ei];
      if (sb > s2[ej]) sb = s2[ej]; if (sb < -s2[ej]) sb = -s2[ej];
      double q1[3], q2[3];
      for (int k = 0; k < 3; k++) { q1[k] = c1[k] + sa * u[k]; q2[k] = c2[k] + sb * v[k]; }
      dist[0] = ebest;
      for (int k = 0; k < 3; k++) { pos[k] = 0.5 * (q1[k] + q2[k]); normal[k] = en[k]; }
      return 1;
    }
  }
  /* face case */
  int ref_is_1 = code < 3; int ra = ref_is_1 ? code : code - 3;
  const double *rp = ref_is_1 ? p1 : p2, *ip = ref_is_1 ? p2 : p1, *rs = ref_is_1 ? s1 : s2, *is = ref_is_1 ? s2 : s1;
  double(*RA)[3] = ref_is_1 ? A1 : A2; double(*IA)[3] = ref_is_1 ? A2 : A1;
  double nref[3]; /* outward normal of the reference face (towards the incident box) */
  for (int k = 0; k < 3; k++) nref[k] = ref_is_1 ? bn[k] : -bn[k];
  /* incident face: the face of the other box most anti-parallel to nref */
  int ia = 0; double mind = 1e30, isg = 1;
  for (int a = 0; a < 3; a++) { double t = dot3(IA[a], nref); if (-fabs(t) < mind) { mind = -fabs(t); ia = a; isg = t > 0 ? -1 : 1; } }
  int iu = (ia + 1) % 3, iv = (ia + 2) % 3, ru = (ra + 1) % 3, rv = (ra + 2) % 3;
  double fc[3]; for (int k = 0; k < 3; k++) fc[k] = ip[k] + isg * is[ia] * IA[ia][k];
  double rc[3]; for (int k = 0; k < 3; k++) rc[k] = rp[k] + rs[ra] * nref[k];  /* centre of the reference face */
  static const double sgu[4] = {1, -1, -1, 1}, sgv[4] = {1, 1, -1, -1};
  double px[16], py[16], vtx[4][3];
  for (int c = 0; c < 4; c++) {
    for (int k = 0; k < 3; k++) vtx[c][k] = fc[k] + sgu[c] * is[iu] * IA[iu][k] + sgv[c] * is[iv] * IA[iv][k];
    double r[3]; for (int k = 0; k < 3; k++) r[k] = vtx[c][k] - rc[k];
    px[c] = dot3(r, RA[ru]); py[c] = dot3(r, RA[rv]);
  }
  /* incident face plane expressed in reference 2-D coords: depth(x,y) = h0 + hx*x + hy*y (along nref, positive = outside) */
  int n = 4;
  n = clip_poly(px, py, n, 1, 0, rs[ru]); n = clip_poly(px, py, n, -1, 0, rs[ru]);
  n = clip_poly(px, py, n, 0, 1, rs[rv]); n = clip_poly(px, py, n, 0, -1, rs[rv]);
  if (n == 0) return 0;
  /* plane of the incident face: normal ni, through fc */
  double ni[3]; for (int k = 0; k < 3; k++) ni[k] = isg * IA[ia][k];
  double nn = dot3(ni, nref);
  int cnt = 0;
  for (int c = 0; c < n && cnt < 8; c++) {
    /* 3-D point on the incident face above reference coords (px,py): rc + x*U + y*V + h*nref with ni.(P - fc) = 0 */
    double base[3]; for (int k = 0; k < 3; k++) base[k] = rc[k] + px[c] * RA[ru][k] + py[c] * RA[rv][k];
    double r[3]; for (int k = 0; k < 3; k++) r[k] = fc[k] - base[k];
    double h = fabs(nn) > 1e-12 ? dot3(ni, r) / nn : 0;   /* signed height above the reference face */
    if (h > margin) continue;
    dist[cnt] = h;
    for (int k = 0; k < 3; k++) { pos[3 * cnt + k] = base[k] + 0.5 * h * nref[k]; normal[3 * cnt + k] = bn[k]; }
    cnt++;
  }
  return cnt;
}

static void collision(const OModel* m, OData* d) {
  d->ncon = 0;
  for (int p = 0; p < m->npair; p++) {
    int g1 = m->pair_geom1[p], g2 = m->pair_geom2[p];
    double margin = m->pair_margin[p];
    double dist[8], pos[24], nrm[24]; int n = 0;
    int t1 = m->geom_type[g1], t2 = m->geom_type[g2];
    if (t1 == GEOM_PLANE && t2 == GEOM_BOX)
      n = plane_box(d->geom_xpos + 3 * g1, d->geom_xmat + 9 * g1, d->geom_xpos + 3 * g2, d->geom_xmat + 9 * g2, m->geom_size + 3 * g2, margin, dist, pos, nrm);
    else if (t1 == GEOM_BOX && t2 == GEOM_BOX)
      n = box_box(d->geom_xpos + 3 * g1, d->geom_xmat + 9 * g1, m->geom_size + 3 * g1, d->geom_xpos + 3 * g2, d->geom_xmat + 9 * g2, m->geom_size + 3 * g2, margin, dist, pos, nrm);
    for (int c = 0; c < n && d->ncon < O_MAXCON; c++) {
      if (!(dist[c] < margin)) continue;
      OContact* con = d->contact + d->ncon++;
      memset(con, 0, sizeof *con);
      con->dist = dist[c]; memcpy(con->pos, pos + 3 * c, 24); memcpy(con->frame, nrm + 3 * c, 24);
      make_frame(con->frame);
      con->geom1 = g1; con->geom2 = g2; con->dim = m->pair_condim[p];
      memcpy(con->friction, m->pair_friction + 5 * p, 40); memcpy(con->solref, m->pair_solref + 2 * p, 16);
      memcpy(con->solimp, m->pair_solimp + 5 * p, 40);
      con->includemargin = m->pair_margin[p] - m->pair_gap[p];
    }
  }
}

/* ------------------------------------------------------------------ constraints (SURVEY B.6) */
static int add_row(const OModel* m, OData* d, int type, int id, double pos, double margin, double frictionloss) {
  int i = d->nefc;
  if (i >= O_MAXEFC) return -1;
  d->nefc++;
  memset(d->efc_J + i * m->nv, 0, sizeof(double) * m->nv);
  d->efc_type[i] = type; d->efc_id[i] = id; d->efc_pos[i] = pos; d->efc_margin[i] = margin; d->efc_frictionloss[i] = frictionloss;
  return i;
}

static double impedance(const double* solimp_in, double pos, double margin) {
  double s[5]; memcpy(s, solimp_in, 40);
  for (int k = 0; k < 2; k++) { if (s[k] < MINIMP) s[k] = MINIMP; if (s[k] > MAXIMP) s[k] = MAXIMP; }
  if (s[2] < 0) s[2] = 0;
  if (s[3] < MINIMP) s[3] = MINIMP; if (s[3] > MAXIMP) s[3] = MAXIMP;
  if (s[4] < 1) s[4] = 1;
  if (s[0] == s[1] || s[2] <= MINVAL) return 0.5 * (s[0] + s[1]);
  double x = (pos - margin) / s[2]; if (x < 0) x = -x;
  if (x >= 1 || x <= 0) return x >= 1 ? s[1] : s[0];
  double y;
  if (s[4] == 1) y = x;
  else if (x <= s[3]) y = pow(x, s[4]) / pow(s[3], s[4] - 1);
  else y = 1 - pow(1 - x, s[4]) / pow(1 - s[3], s[4] - 1);
  return s[0] + y * (s[1] - s[0]);
}

static void make_constraint(const OModel* m, OData* d) {
  int nv = m->nv;
  d->nefc = 0;
  double* jp1 = (double*)malloc(sizeof(double) * 3 * nv); double* jp2 = (double*)malloc(sizeof(double) * 3 * nv);
  /* equality */
  for (int e = 0; e < m->neq; e++) {
    if (m->eq_type[e] == EQ_CONNECT) {
      int b1 = m->eq_obj1id[e], b2 = m->eq_obj2id[e];
      double a1[3], a2[3], v[3];
      mat_vec3(v, d->xmat + 9 * b1, m->eq_data + 11 * e); for (int k = 0; k < 3; k++) a1[k] = d->xpos[3 * b1 + k] + v[k];
      mat_vec3(v, d->xmat + 9 * b2, m->eq_data + 11 * e + 3); for (int k = 0; k < 3; k++) a2[k] = d->xpos[3 * b2 + k] + v[k];
      o_jac(m, d, jp1, NULL, a1, b1); o_jac(m, d, jp2, NULL, a2, b2);
      for (int r = 0; r < 3; r++) {
        int i = add_row(m, d, O_CNSTR_EQUALITY, e, a1[r] - a2[r], 0, 0);
        for (int c = 0; c < nv; c++) d->efc_J[i * nv + c] = jp1[r * nv + c] - jp2[r * nv + c];
        d->efc_diagApprox[i] = m->body_invweight0[2 * b1] + m->body_invweight0[2 * b2];
      }
    } else if (m->eq_type[e] == EQ_JOINT) {
      int j1 = m->eq_obj1id[e], j2 = m->eq_obj2id[e];
      const double* c = m->eq_data + 11 * e;
      double p1 = d->qpos[m->jnt_qposadr[j1]] - m->qpos0[m->jnt_qposadr[j1]];
      double pos, deriv = 0;
      if (j2 >= 0) {
        double p2 = d->qpos[m->jnt_qposadr[j2]] - m->qpos0[m->jnt_qposadr[j2]];
        pos = p1 - (c[0] + c[1] * p2 + c[2] * p2 * p2 + c[3] * p2 * p2 * p2 + c[4] * p2 * p2 * p2 * p2);
        deriv = c[1] + 2 * c[2] * p2 + 3 * c[3] * p2 * p2 + 4 * c[4] * p2 * p2 * p2;
      } else pos = p1 - c[0];
      int i = add_row(m, d, O_CNSTR_EQUALITY, e, pos, 0, 0);
      d->efc_J[i * nv + m->jnt_dofadr[j1]] = 1;
      d->efc_diagApprox[i] = m->dof_invweight0[m->jnt_dofadr[j1]];
      if (j2 >= 0) { d->efc_J[i * nv + m->jnt_dofadr[j2]] = -deriv; d->efc_diagApprox[i] += m->dof_invweight0[m->jnt_dofadr[j2]]; }
    }
  }
  d->ne = d->nefc;
  /* dof friction loss */
  for (int i = 0; i < nv; i++) if (m->dof_frictionloss[i] > 0) {
    int r = add_row(m, d, O_CNSTR_FRICTION_DOF, i, 0, 0, m->dof_frictionloss[i]);
    d->efc_J[r * nv + i] = 1; d->efc_diagApprox[r] = m->dof_invweight0[i];
  }
  d->nf = d->nefc - d->ne;
  /* joint limits */
  for (int j = 0; j < m->njnt; j++) if (m->jnt_limited[j] && (m->jnt_type[j] == JNT_HINGE || m->jnt_type[j] == JNT_SLIDE)) {
    double value = d->qpos[m->jnt_qposadr[j]], margin = m->jnt_margin[j];
    for (int side = -1; side <= 1; side += 2) {
      double dist = side * (m->jnt_range[2 * j + (side + 1) / 2] - value);
      if (dist < margin) {
        int r = add_row(m, d, O_CNSTR_LIMIT_JOINT, j, dist, margin, 0);
        d->efc_J[r * nv + m->jnt_dofadr[j]] = -side; d->efc_diagApprox[r] = m->dof_invweight0[m->jnt_dofadr[j]];
      }
    }
  }
  d->nl = d->nefc - d->ne - d->nf;
  /* contacts (elliptic cones, condim 3) */
  for (int c = 0; c < d->ncon; c++) {
    OContact* con = d->contact + c;
    int b1 = m->geom_bodyid[con->geom1], b2 = m->geom_bodyid[con->geom2];
    o_jac(m, d, jp1, NULL, con->pos, b1); o_jac(m, d, jp2, NULL, con->pos, b2);
    con->efc_address = d->nefc;
    double tran = m->body_invweight0[2 * b1] + m->body_invweight0[2 * b2];
    for (int r = 0; r < con->dim; r++) {
      int i = add_row(m, d, O_CNSTR_CONTACT_ELLIPTIC, c, r == 0 ? con->dist : 0, r == 0 ? con->includemargin : 0, 0);
      if (i < 0) { con->efc_address = -1; break; }
      for (int k = 0; k < nv; k++) {
        double v = 0; for (int a = 0; a < 3; a++) v += con->frame[3 * r + a] * (jp2[a * nv + k] - jp1[a * nv + k]);
        d->efc_J[i * nv + k] = v;
      }
      d->efc_diagApprox[i] = tran;
    }
  }
  free(jp1); free(jp2);
  /* impedance, K, B, R, D (mj_makeImpedance) */
  for (int i = 0; i < d->nefc; i++) {
    const double *solref, *solimp; int id = d->efc_id[i]; int fric_row = 0;
    switch (d->efc_type[i]) {
      case O_CNSTR_EQUALITY: solref = m->eq_solref + 2 * id; solimp = m->eq_solimp + 5 * id; break;
      case O_CNSTR_FRICTION_DOF: solref = m->dof_solref + 2 * id; solimp = m->dof_solimp + 5 * id; fric_row = 1; break;
      case O_CNSTR_LIMIT_JOINT: solref = m->jnt_solref + 2 * id; solimp = m->jnt_solimp + 5 * id; break;
      default: solref = d->contact[id].solref; solimp = d->contact[id].solimp; fric_row = (i != d->contact[id].efc_address); break;
    }
    double imp = impedance(solimp, d->efc_pos[i], d->efc_margin[i]);
    double dmax = solimp[1]; if (dmax < MINIMP) dmax = MINIMP; if (dmax > MAXIMP) dmax = MAXIMP;
    double K, B;
    if (solref[0] > 0) {
      double tc = solref[0] < 2 * m->timestep ? 2 * m->timestep : solref[0], dr = solref[1];   /* refsafe */
      K = 1 / fmax(MINVAL, dmax * dmax * tc * tc * dr * dr); B = 2 / fmax(MINVAL, dmax * tc);
    } else { K = -solref[0] / fmax(MINVAL, dmax * dmax); B = -solref[1] / fmax(MINVAL, dmax); }
    if (fric_row) K = 0;
    d->efc_KBIP[4 * i] = K; d->efc_KBIP[4 * i + 1] = B; d->efc_KBIP[4 * i + 2] = imp; d->efc_KBIP[4 * i + 3] = 0;
    d->efc_R[i] = fmax(MINVAL, (1 - imp) * d->efc_diagApprox[i] / imp);
  }
  for (int c = 0; c < d->ncon; c++) {
    OContact* con = d->contact + c; int i = con->efc_address; if (i < 0) continue;
    d->efc_R[i + 1] = d->efc_R[i] / fmax(MINVAL, m->impratio);
    con->mu = con->friction[0] * sqrt(d->efc_R[i + 1] / d->efc_R[i]);
    for (int j = 1; j < con->dim - 1; j++) d->efc_R[i + j + 1] = d->efc_R[i + 1] * con->friction[0] * con->friction[0] / (con->friction[j] * con->friction[j]);
  }
  for (int i = 0; i < d->nefc; i++) d->efc_D[i] = 1 / d->efc_R[i];
}

static void transmission(const OModel* m, OData* d) {
  int nv = m->nv;
  for (int a = 0; a < m->nu; a++) {
    memset(d->actuator_moment + a * nv, 0, sizeof(double) * nv);
    double gear = m->actuator_gear[a];
    if (m->actuator_trntype[a] == TRN_JOINT) {
      int j = m->actuator_trnid[a];
      d->actuator_length[a] = d->qpos[m->jnt_qposadr[j]] * gear; d->actuator_moment[a * nv + m->jnt_dofadr[j]] = gear;
    } else {
      int t = m->actuator_trnid[a];
      d->actuator_length[a] = d->ten_length[t] * gear;
      for (int k = 0; k < nv; k++) d->actuator_moment[a * nv + k] = d->ten_J[t * nv + k] * gear;
    }
  }
}

static void fwd_position(const OModel* m, OData* d) {
  kinematics(m, d); com_pos(m, d); tendon(m, d); crb(m, d); chol_factor(d->qL, d->qM, m->nv);
  collision(m, d); make_constraint(m, d); transmission(m, d);
}

/* ------------------------------------------------------------------ velocity stage (SURVEY B.4) */
static void com_vel(const OModel* m, OData* d) {
  memset(d->cvel, 0, sizeof(double) * 6);
  for (int b = 1; b < m->nbody; b++) {
    double cvel[6]; memcpy(cvel, d->cvel + 6 * m->body_parentid[b], 48);
    int da = m->body_dofadr[b];
    for (int j = m->body_jntadr[b]; j < m->body_jntadr[b] + m->body_jntnum[b] && m->body_jntnum[b] > 0; j++) {
      if (m->jnt_type[j] == JNT_FREE) {
        memset(d->cdof_dot + 6 * da, 0, sizeof(double) * 18);
        for (int i = 0; i < 3; i++) for (int k = 0; k < 6; k++) cvel[k] += d->cdof[6 * (da + i) + k] * d->qvel[da + i];
        da += 3;
        for (int i = 0; i < 3; i++) cross_motion(d->cdof_dot + 6 * (da + i), cvel, d->cdof + 6 * (da + i));
        for (int i = 0; i < 3; i++) for (int k = 0; k < 6; k++) cvel[k] += d->cdof[6 * (da + i) + k] * d->qvel[da + i];
        da += 3;
      } else {
        cross_motion(d->cdof_dot + 6 * da, cvel, d->cdof + 6 * da);
        for (int k = 0; k < 6; k++) cvel[k] += d->cdof[6 * da + k] * d->qvel[da];
        da++;
      }
    }
    memcpy(d->cvel + 6 * b, cvel, 48);
  }
}

static void passive(const OModel* m, OData* d) {
  memset(d->qfrc_passive, 0, sizeof(double) * m->nv);
  for (int j = 0; j < m->njnt; j++) if (m->jnt_type[j] == JNT_HINGE || m->jnt_type[j] == JNT_SLIDE) {
    int qa = m->jnt_qposadr[j], da = m->jnt_dofadr[j];
    d->qfrc_passive[da] -= m->jnt_stiffness[j] * (d->qpos[qa] - m->qpos_spring[qa]);
  }
  for (int i = 0; i < m->nv; i++) d->qfrc_passive[i] -= m->dof_damping[i] * d->qvel[i];
}

static void rne(const OModel* m, OData* d, int flg_acc, double* result) {
  int nb = m->nbody;
  memset(d->cacc, 0, sizeof(double) * 6); for (int k = 0; k < 3; k++) d->cacc[3 + k] = -m->gravity[k];
  for (int b = 1; b < nb; b++) {
    double tmp[6] = {0, 0, 0, 0, 0, 0}; int da = m->body_dofadr[b];
    for (int i = 0; i < m->body_dofnum[b]; i++) for (int k = 0; k < 6; k++) tmp[k] += d->cdof_dot[6 * (da + i) + k] * d->qvel[da + i];
    if (flg_acc) for (int i = 0; i < m->body_dofnum[b]; i++) for (int k = 0; k < 6; k++) tmp[k] += d->cdof[6 * (da + i) + k] * d->qacc[da + i];
    for (int k = 0; k < 6; k++) d->cacc[6 * b + k] = d->cacc[6 * m->body_parentid[b] + k] + tmp[k];
    double t1[6], t2[6];
    mul_inert_vec(d->cfrc_body + 6 * b, d->cinert + 10 * b, d->cacc + 6 * b);
    mul_inert_vec(t1, d->cinert + 10 * b, d->cvel + 6 * b); cross_force(t2, d->cvel + 6 * b, t1);
    for (int k = 0; k < 6; k++) d->cfrc_body[6 * b + k] += t2[k];
  }
  memset(d->cfrc_body, 0, sizeof(double) * 6);
  for (int b = nb - 1; b > 0; b--) { int p = m->body_parentid[b]; if (p > 0) for (int k = 0; k < 6; k++) d->cfrc_body[6 * p + k] += d->cfrc_body[6 * b + k]; }
  for (int i = 0; i < m->nv; i++) { double v = 0; for (int k = 0; k < 6; k++) v += d->cdof[6 * i + k] * d->cfrc_body[6 * m->dof_bodyid[i] + k]; result[i] = v; }
}

static void reference_constraint(const OModel* m, OData* d) {
  int nv = m->nv;
  for (int i = 0; i < d->nefc; i++) {
    double v = 0; for (int k = 0; k < nv; k++) v += d->efc_J[i * nv + k] * d->qvel[k];
    d->efc_vel[i] = v;
    d->efc_aref[i] = -d->efc_KBIP[4 * i + 1] * v - d->efc_KBIP[4 * i] * d->efc_KBIP[4 * i + 2] * (d->efc_pos[i] - d->efc_margin[i]);
  }
}

static void fwd_velocity(const OModel* m, OData* d) {
  for (int t = 0; t < m->ntendon; t++) { double v = 0; for (int k = 0; k < m->nv; k++) v += d->ten_J[t * m->nv + k] * d->qvel[k]; d->ten_velocity[t] = v; }
  for (int a = 0; a < m->nu; a++) { double v = 0; for (int k = 0; k < m->nv; k++) v += d->actuator_moment[a * m->nv + k] * d->qvel[k]; d->actuator_velocity[a] = v; }
  com_vel(m, d); passive(m, d); reference_constraint(m, d); rne(m, d, 0, d->qfrc_bias);
}

static void fwd_actuation(const OModel* m, OData* d) {
  /* SURVEY B.5 */
  int nv = m->nv; memset(d->qfrc_actuator, 0, sizeof(double) * nv);
  for (int a = 0; a < m->nu; a++) {
    double c = d->ctrl[a];
    if (m->actuator_ctrllimited[a]) { if (c < m->actuator_ctrlrange[2 * a]) c = m->actuator_ctrlrange[2 * a]; if (c > m->actuator_ctrlrange[2 * a + 1]) c = m->actuator_ctrlrange[2 * a + 1]; }
    const double* bp = m->actuator_biasprm + 3 * a;
    double f = m->actuator_gainprm[a] * c + bp[0] + bp[1] * d->actuator_length[a] + bp[2] * d->actuator_velocity[a];
    if (m->actuator_forcelimited[a]) { if (f < m->actuator_forcerange[2 * a]) f = m->actuator_forcerange[2 * a]; if (f > m->actuator_forcerange[2 * a + 1]) f = m->actuator_forcerange[2 * a + 1]; }
    d->actuator_force[a] = f;
    for (int k = 0; k < nv; k++) d->qfrc_actuator[k] += d->actuator_moment[a * nv + k] * f;
  }
}

static void fwd_acceleration(const OModel* m, OData* d) {
  for (int i = 0; i < m->nv; i++) { d->qfrc_smooth[i] = d->qfrc_passive[i] - d->qfrc_bias[i] + d->qfrc_actuator[i]; d->qacc_smooth[i] = d->qfrc_smooth[i]; }
  chol_solve(d->qL, d->qacc_smooth, m->nv);
}

/* ------------------------------------------------------------------ primal Newton solver (SURVEY B.7) */
typedef struct { double quad[3]; } Quad;

/* per-row cost s(jar), force = -ds/djar, and for quadratic-state rows the active D; cone Hessians handled separately */
static double constraint_update(const OModel* m, OData* d, const double* jar, int flg_hess_cone, double* coneH /* per contact 9 */) {
  (void)m;
  double cost = 0; int nefc = d->nefc;
  for (int i = 0; i < nefc; i++) {
    double D = d->efc_D[i], R = d->efc_R[i], x = jar[i];
    int t = d->efc_type[i];
    if (t == O_CNSTR_EQUALITY) { d->efc_force[i] = -D * x; d->efc_state[i] = O_STATE_QUADRATIC; cost += 0.5 * D * x * x; }
    else if (t == O_CNSTR_FRICTION_DOF) {
      double f = d->efc_frictionloss[i], rf = R * f;
      if (x <= -rf) { d->efc_force[i] = f; d->efc_state[i] = O_STATE_LINEARNEG; cost += -0.5 * rf * f - f * x; }
      else if (x >= rf) { d->efc_force[i] = -f; d->efc_state[i] = O_STATE_LINEARPOS; cost += -0.5 * rf * f + f * x; }
      else { d->efc_force[i] = -D * x; d->efc_state[i] = O_STATE_QUADRATIC; cost += 0.5 * D * x * x; }
    } else if (t == O_CNSTR_LIMIT_JOINT) {
      if (x < 0) { d->efc_force[i] = -D * x; d->efc_state[i] = O_STATE_QUADRATIC; cost += 0.5 * D * x * x; }
      else { d->efc_force[i] = 0; d->efc_state[i] = O_STATE_SATISFIED; }
    } else { /* elliptic contact: handle the whole cone at its first row */
      OContact* con = d->contact + d->efc_id[i]; int dim = con->dim; double mu = con->mu;
      double U[6], N, T = 0;
      U[0] = jar[i] * mu; for (int j = 1; j < dim; j++) { U[j] = jar[i + j] * con->friction[j - 1]; T += U[j] * U[j]; }
      N = U[0]; T = sqrt(T);
      if (N >= mu * T || (T <= 0 && N >= 0)) {
        for (int j = 0; j < dim; j++) { d->efc_force[i + j] = 0; d->efc_state[i + j] = O_STATE_SATISFIED; }
      } else if (mu * N + T <= 0 || (T <= 0 && N < 0)) {
        for (int j = 0; j < dim; j++) { d->efc_force[i + j] = -d->efc_D[i + j] * jar[i + j]; d->efc_state[i + j] = O_STATE_QUADRATIC; cost += 0.5 * d->efc_D[i + j] * jar[i + j] * jar[i + j]; }
      } else {
        double Dm = d->efc_D[i] / (mu * mu * (1 + mu * mu)), NmT = N - mu * T;
        cost += 0.5 * Dm * NmT * NmT;
        d->efc_force[i] = -Dm * NmT * mu;
        for (int j = 1; j < dim; j++) d->efc_force[i + j] = -d->efc_force[i] / T * U[j] * con->friction[j - 1];
        for (int j = 0; j < dim; j++) d->efc_state[i + j] = O_STATE_CONE;
        if (flg_hess_cone && coneH && dim == 3) {
          /* Hessian of s wrt jar (3x3): diag(scale) * H_U * diag(scale) */
          double sc[3] = {mu, con->friction[0], con->friction[1]}, H[9];
          double u1 = U[1] / T, u2 = U[2] / T;
          H[0] = Dm; H[1] = H[3] = -Dm * mu * u1; H[2] = H[6] = -Dm * mu * u2;
          double a = Dm * mu * mu, b = -Dm * mu * NmT / T;
          H[4] = a * u1 * u1 + b * (1 - u1 * u1); H[8] = a * u2 * u2 + b * (1 - u2 * u2); H[5] = H[7] = a * u1 * u2 - b * u1 * u2;
          for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) coneH[9 * d->efc_id[i] + 3 * r + c] = H[3 * r + c] * sc[r] * sc[c];
        }
      }
      i += dim - 1;
    }
  }
  return cost;
}

static double total_cost(const OModel* m, OData* d, const double* qacc, double* Ma, double* jar) {
  int nv = m->nv;
  for (int i = 0; i < nv; i++) { double v = 0; for (int k = 0; k < nv; k++) v += d->qM[i * nv + k] * qacc[k]; Ma[i] = v; }
  for (int i = 0; i < d->nefc; i++) { double v = -d->efc_aref[i]; for (int k = 0; k < nv; k++) v += d->efc_J[i * nv + k] * qacc[k]; jar[i] = v; }
  double c = constraint_update(m, d, jar, 0, NULL);
  for (int i = 0; i < nv; i++) c += 0.5 * (Ma[i] - d->qfrc_smooth[i]) * (qacc[i] - d->qacc_smooth[i]);
  return c;
}

/* derivative and curvature of the line cost at alpha */
static void line_eval(const OModel* m, OData* d, const double* jar, const double* jv, double g1, double g2, double alpha, double* dphi, double* ddphi) {
  (void)m;
  double p1 = g1 + alpha * g2, p2 = g2;
  for (int i = 0; i < d->nefc; i++) {
    double D = d->efc_D[i], R = d->efc_R[i], x = jar[i] + alpha * jv[i], v = jv[i];
    int t = d->efc_type[i];
    if (t == O_CNSTR_EQUALITY) { p1 += D * x * v; p2 += D * v * v; }
    else if (t == O_CNSTR_FRICTION_DOF) {
      double f = d->efc_frictionloss[i], rf = R * f;
      if (x <= -rf) p1 += -f * v; else if (x >= rf) p1 += f * v; else { p1 += D * x * v; p2 += D * v * v; }
    } else if (t == O_CNSTR_LIMIT_JOINT) { if (x < 0) { p1 += D * x * v; p2 += D * v * v; } }
    else {
      OContact* con = d->contact + d->efc_id[i]; int dim = con->dim; double mu = con->mu;
      double U[6], V[6], T = 0;
      U[0] = x * mu; V[0] = v * mu;
      for (int j = 1; j < dim; j++) { U[j] = (jar[i + j] + alpha * jv[i + j]) * con->friction[j - 1]; V[j] = jv[i + j] * con->friction[j - 1]; T += U[j] * U[j]; }
      double N = U[0]; T = sqrt(T);
      if (N >= mu * T || (T <= 0 && N >= 0)) { }
      else if (mu * N + T <= 0 || (T <= 0 && N < 0)) {
        for (int j = 0; j < dim; j++) { double xx = jar[i + j] + alpha * jv[i + j]; p1 += d->efc_D[i + j] * xx * jv[i + j]; p2 += d->efc_D[i + j] * jv[i + j] * jv[i + j]; }
      } else {
        double Dm = d->efc_D[i] / (mu * mu * (1 + mu * mu)), NmT = N - mu * T;
        double UV = 0, VV = 0; for (int j = 1; j < dim; j++) { UV += U[j] * V[j]; VV += V[j] * V[j]; }
        double T1 = UV / T, T2 = VV / T - UV * UV / (T * T * T);
        double N1 = V[0];
        p1 += Dm * NmT * (N1 - mu * T1);
        p2 += Dm * ((N1 - mu * T1) * (N1 - mu * T1) - NmT * mu * T2);
      }
      i += dim - 1;
    }
  }
  *dphi = p1; *ddphi = p2;
}

static void solve_newton(const OModel* m, OData* d) {
  int nv = m->nv, nefc = d->nefc;
  d->solver_iter = 0;
  if (nefc == 0) { memcpy(d->qacc, d->qacc_smooth, sizeof(double) * nv); memset(d->qfrc_constraint, 0, sizeof(double) * nv); return; }
  double *Ma = (double*)malloc(sizeof(double) * nv), *jar = (double*)malloc(sizeof(double) * (nefc + 1)), *grad = (double*)malloc(sizeof(double) * nv),
         *search = (double*)malloc(sizeof(double) * nv), *Mv = (double*)malloc(sizeof(double) * nv), *jv = (double*)malloc(sizeof(double) * (nefc + 1)),
         *H = (double*)malloc(sizeof(double) * nv * nv), *L = (double*)malloc(sizeof(double) * nv * nv), *coneH = (double*)calloc(9 * (d->ncon + 1), sizeof(double)),
         *tmp = (double*)malloc(sizeof(double) * nv);
  /* warm start: keep qacc_warmstart unless qacc_smooth has lower cost (mj_fwdConstraint) */
  double cw = total_cost(m, d, d->qacc_warmstart, Ma, jar);
  double cs = total_cost(m, d, d->qacc_smooth, Ma, jar);
  memcpy(d->qacc, cw < cs ? d->qacc_warmstart : d->qacc_smooth, sizeof(double) * nv);
  double scale = 1.0 / (m->meaninertia * (nv > 1 ? nv : 1));
  double cost = 0;
  /* the oracle iterates to (near) machine precision rather than MuJoCo's tolerance 1e-8:
   * it represents the optimum that every conforming solver approaches */
  for (int iter = 0; iter < 200; iter++) {
    cost = total_cost(m, d, d->qacc, Ma, jar);
    constraint_update(m, d, jar, 1, coneH);
    for (int i = 0; i < nv; i++) { double v = Ma[i] - d->qfrc_smooth[i]; for (int r = 0; r < nefc; r++) v -= d->efc_J[r * nv + i] * d->efc_force[r]; grad[i] = v; }
    double gn = 0; for (int i = 0; i < nv; i++) gn += grad[i] * grad[i]; gn = sqrt(gn);
    d->solver_iter = iter;
    if (scale * gn < 1e-15) break;
    /* Hessian */
    memcpy(H, d->qM, sizeof(double) * nv * nv);
    for (int r = 0; r < nefc; r++) {
      if (d->efc_state[r] == O_STATE_QUADRATIC) {
        const double* J = d->efc_J + r * nv; double D = d->efc_D[r];
        for (int a = 0; a < nv; a++) if (J[a] != 0) for (int b = 0; b < nv; b++) H[a * nv + b] += D * J[a] * J[b];
      } else if (d->efc_state[r] == O_STATE_CONE) {
        int c = d->efc_id[r], dim = d->contact[c].dim; const double* Hc = coneH + 9 * c;
        for (int p = 0; p < dim; p++) for (int q = 0; q < dim; q++) {
          const double *Jp = d->efc_J + (r + p) * nv, *Jq = d->efc_J + (r + q) * nv; double h = Hc[3 * p + q];
          for (int a = 0; a < nv; a++) if (Jp[a] != 0) for (int b = 0; b < nv; b++) H[a * nv + b] += h * Jp[a] * Jq[b];
        }
        r += dim - 1;
      }
    }
    chol_factor(L, H, nv);
    for (int i = 0; i < nv; i++) search[i] = -grad[i];
    chol_solve(L, search, nv);
    for (int i = 0; i < nv; i++) { double v = 0; for (int k = 0; k < nv; k++) v += d->qM[i * nv + k] * search[k]; Mv[i] = v; }
    for (int r = 0; r < nefc; r++) { double v = 0; for (int k = 0; k < nv; k++) v += d->efc_J[r * nv + k] * search[k]; jv[r] = v; }
    double g1 = 0, g2 = 0; for (int i = 0; i < nv; i++) { g1 += search[i] * (Ma[i] - d->qfrc_smooth[i]); g2 += search[i] * Mv[i]; }
    /* exact line search: safeguarded Newton on phi'(alpha) */
    double lo = 0, hi = -1, alpha = 0, p1, p2;
    line_eval(m, d, jar, jv, g1, g2, 0, &p1, &p2);
    if (p1 >= 0) break;  /* not a descent direction: converged to roundoff */
    alpha = -p1 / p2;
    for (int ls = 0; ls < 100; ls++) {
      line_eval(m, d, jar, jv, g1, g2, alpha, &p1, &p2);
      if (fabs(p1) < 1e-16 * fabs(g1) + 1e-300) break;
      if (p1 < 0) lo = alpha; else hi = alpha;
      double na = alpha - p1 / p2;
      if (hi < 0) { if (na <= lo) na = 2 * alpha; }
      else if (na <= lo || na >= hi) na = 0.5 * (lo + hi);
      if (na == alpha) break;
      alpha = na;
    }
    for (int i = 0; i < nv; i++) d->qacc[i] += alpha * search[i];
    double nc = total_cost(m, d, d->qacc, Ma, jar);
    if (!(nc < cost) && iter > 0 && fabs(nc - cost) <= 1e-16 * fabs(cost)) { cost = nc; d->solver_iter = iter + 1; break; }
  }
  cost = total_cost(m, d, d->qacc, Ma, jar);
  d->solver_cost = cost;
  for (int i = 0; i < nv; i++) { double v = 0; for (int r = 0; r < nefc; r++) v += d->efc_J[r * nv + i] * d->efc_force[r]; d->qfrc_constraint[i] = v; }
  free(Ma); free(jar); free(grad); free(search); free(Mv); free(jv); free(H); free(L); free(coneH); free(tmp);
}

/* ------------------------------------------------------------------ pipeline */
void o_forward(const OModel* m, OData* d) {
  fwd_position(m, d); fwd_velocity(m, d); fwd_actuation(m, d); fwd_acceleration(m, d); solve_newton(m, d);
}

static int bad(double x) { return isnan(x) || x > 1e10 || x < -1e10; }

static void euler(const OModel* m, OData* d) {
  /* SURVEY B.8 (mj_Euler with implicit joint damping) */
  int nv = m->nv; int damp = 0;
  for (int i = 0; i < nv; i++) if (m->dof_damping[i] > 0) damp = 1;
  double* qacc = (double*)malloc(sizeof(double) * nv);
  if (!damp) memcpy(qacc, d->qacc, sizeof(double) * nv);
  else {
    memcpy(d->qH, d->qM, sizeof(double) * nv * nv);
    for (int i = 0; i < nv; i++) d->qH[i * nv + i] += m->timestep * m->dof_damping[i];
    double* L = (double*)malloc(sizeof(double) * nv * nv); chol_factor(L, d->qH, nv);
    for (int i = 0; i < nv; i++) qacc[i] = d->qfrc_smooth[i] + d->qfrc_constraint[i];
    chol_solve(L, qacc, nv); free(L);
  }
  double h = m->timestep;
  for (int i = 0; i < nv; i++) d->qvel[i] += h * qacc[i];
  for (int j = 0; j < m->njnt; j++) {
    int qa = m->jnt_qposadr[j], da = m->jnt_dofadr[j];
    if (m->jnt_type[j] == JNT_FREE) {
      for (int k = 0; k < 3; k++) d->qpos[qa + k] += h * d->qvel[da + k];
      double w[3] = {d->qvel[da + 3], d->qvel[da + 4], d->qvel[da + 5]}, qr[4];
      double n = norm3(w); if (n < MINVAL) { w[0] = 1; w[1] = w[2] = 0; n = 0; } else { w[0] /= n; w[1] /= n; w[2] /= n; }
      axis_angle2quat(qr, w, h * n);
      normalize4(d->qpos + qa + 3); mul_quat(d->qpos + qa + 3, d->qpos + qa + 3, qr);
    } else d->qpos[qa] += h * d->qvel[da];
  }
  d->time += h;
  free(qacc);
}

void o_step(const OModel* m, OData* d) {
  /* mj_step: checkPos, checkVel, forward, checkAcc, Euler (SURVEY 3.4, B.10) */
  int w = 0;
  for (int i = 0; i < m->nq; i++) if (bad(d->qpos[i])) w |= 1;
  for (int i = 0; i < m->nv; i++) if (bad(d->qvel[i])) w |= 2;
  if (w) { o_reset_data(m, d); d->warn_bad = w; }
  o_forward(m, d);
  for (int i = 0; i < m->nv; i++) if (bad(d->qacc[i])) w |= 4;
  if (w & 4) { o_reset_data(m, d); d->warn_bad = w; o_forward(m, d); }
  memcpy(d->qacc_warmstart, d->qacc, sizeof(double) * m->nv);
  euler(m, d);
}
void o_step_n(const OModel* m, OData* d, int n) { for (int i = 0; i < n; i++) o_step(m, d); }

/* ------------------------------------------------------------------ mj_setConst */
void o_set_const(OModel* m) {
  OData* d = o_data_new(m);
  int nv = m->nv;
  kinematics(m, d); com_pos(m, d);
  /* connect anchors on body2 at qpos0 */
  for (int e = 0; e < m->neq; e++) if (m->eq_type[e] == EQ_CONNECT) {
    int b1 = m->eq_obj1id[e], b2 = m->eq_obj2id[e]; double v[3], p[3];
    mat_vec3(v, d->xmat + 9 * b1, m->eq_data + 11 * e);
    for (int k = 0; k < 3; k++) p[k] = d->xpos[3 * b1 + k] + v[k] - d->xpos[3 * b2 + k];
    matT_vec3(m->eq_data + 11 * e + 3, d->xmat + 9 * b2, p);
  }
  tendon(m, d); crb(m, d); chol_factor(d->qL, d->qM, nv);
  double tr = 0; for (int i = 0; i < nv; i++) tr += d->qM[i * nv + i];
  m->meaninertia = nv > 0 ? tr / nv : 1;
  double* Minv = (double*)calloc(nv * nv + 1, sizeof(double));
  for (int c = 0; c < nv; c++) { double* col = (double*)calloc(nv, sizeof(double)); col[c] = 1; chol_solve(d->qL, col, nv); for (int r = 0; r < nv; r++) Minv[r * nv + c] = col[r]; free(col); }
  double* jp = (double*)malloc(sizeof(double) * 3 * nv + 8); double* jr = (double*)malloc(sizeof(double) * 3 * nv + 8);
  for (int b = 0; b < m->nbody; b++) {
    m->body_invweight0[2 * b] = m->body_invweight0[2 * b + 1] = 0;
    if (b == 0 || m->body_weldid[b] == 0) continue;
    o_jac(m, d, jp, jr, d->xipos + 3 * b, b);
    double tp = 0, trr = 0;
    for (int r = 0; r < 3; r++) for (int a = 0; a < nv; a++) for (int c = 0; c < nv; c++) {
      tp += jp[r * nv + a] * Minv[a * nv + c] * jp[r * nv + c]; trr += jr[r * nv + a] * Minv[a * nv + c] * jr[r * nv + c];
    }
    m->body_invweight0[2 * b] = tp / 3; m->body_invweight0[2 * b + 1] = trr / 3;
  }
  for (int j = 0; j < m->njnt; j++) {
    int da = m->jnt_dofadr[j];
    if (m->jnt_type[j] == JNT_FREE) {
      double a = 0, b = 0; for (int i = 0; i < 3; i++) { a += Minv[(da + i) * nv + da + i]; b += Minv[(da + 3 + i) * nv + da + 3 + i]; }
      for (int i = 0; i < 3; i++) { m->dof_invweight0[da + i] = a / 3; m->dof_invweight0[da + 3 + i] = b / 3; }
    } else m->dof_invweight0[da] = Minv[da * nv + da];
  }
  for (int t = 0; t < m->ntendon; t++) {
    double v = 0; for (int a = 0; a < nv; a++) for (int c = 0; c < nv; c++) v += d->ten_J[t * nv + a] * Minv[a * nv + c] * d->ten_J[t * nv + c];
    m->tendon_invweight0[t] = v;
  }
  free(Minv); free(jp); free(jr); o_data_free(d);
}

/* ------------------------------------------------------------------ controllers */
void o_rot_err(const double* xmat, const double* rv, double* err) {
  /* reference controller_func.py:30-48: rotvec of R_target * R_site^T (scipy conventions, SURVEY App. C) */
  double ang = norm3(rv), q[4];
  if (ang < 1e-300) { q[0] = 1; q[1] = q[2] = q[3] = 0; } else { double ax[3] = {rv[0] / ang, rv[1] / ang, rv[2] / ang}; axis_angle2quat(q, ax, ang); }
  double Rt[9]; quat2mat(Rt, q);
  double RsT[9] = {xmat[0], xmat[3], xmat[6], xmat[1], xmat[4], xmat[7], xmat[2], xmat[5], xmat[8]}, E[9];
  mat_mul3(E, Rt, RsT);
  /* matrix -> quaternion (Shepperd), canonical w >= 0, -> rotvec */
  double tr = E[0] + E[4] + E[8], w, x, y, z;
  if (tr > 0) { double s = sqrt(tr + 1.0) * 2; w = 0.25 * s; x = (E[7] - E[5]) / s; y = (E[2] - E[6]) / s; z = (E[3] - E[1]) / s; }
  else if (E[0] > E[4] && E[0] > E[8]) { double s = sqrt(1.0 + E[0] - E[4] - E[8]) * 2; w = (E[7] - E[5]) / s; x = 0.25 * s; y = (E[1] + E[3]) / s; z = (E[2] + E[6]) / s; }
  else if (E[4] > E[8]) { double s = sqrt(1.0 + E[4] - E[0] - E[8]) * 2; w = (E[2] - E[6]) / s; x = (E[1] + E[3]) / s; y = 0.25 * s; z = (E[5] + E[7]) / s; }
  else { double s = sqrt(1.0 + E[8] - E[0] - E[4]) * 2; w = (E[3] - E[1]) / s; x = (E[2] + E[6]) / s; y = (E[5] + E[7]) / s; z = 0.25 * s; }
  double nq = sqrt(w * w + x * x + y * y + z * z); w /= nq; x /= nq; y /= nq; z /= nq;
  if (w < 0) { w = -w; x = -x; y = -y; z = -z; }
  double sn = sqrt(x * x + y * y + z * z), a = 2 * atan2(sn, w);
  double k = sn < 1e-12 ? 2.0 : a / sn;
  err[0] = k * x; err[1] = k * y; err[2] = k * z;
}

void o_pid_task_ctrl(const OModel* m, const OData* d, int tcp, const double* traj, const double* g, double* u) {
  /* reference controller_func.py:68-117; gains12 = kp_pos[3], kd_pos[3], kp_rot[3], kd_rot[3] (diagonals) */
  int nv = m->nv; double ep[3], er[3];
  for (int k = 0; k < 3; k++) ep[k] = traj[k] - d->site_xpos[3 * tcp + k];
  o_rot_err(d->site_xmat + 9 * tcp, traj + 3, er);
  double* jp = (double*)malloc(sizeof(double) * 3 * nv); double* jr = (double*)malloc(sizeof(double) * 3 * nv);
  o_jac_site(m, d, jp, jr, tcp);
  double F[6];
  for (int r = 0; r < 3; r++) {
    double vp = 0, vr = 0; for (int k = 0; k < 6; k++) { vp += jp[r * nv + k] * d->qvel[k]; vr += jr[r * nv + k] * d->qvel[k]; }
    F[r] = g[r] * ep[r] - g[3 + r] * vp; F[3 + r] = g[6 + r] * er[r] - g[9 + r] * vr;
  }
  for (int k = 0; k < 6; k++) {
    double v = d->qfrc_bias[k];
    for (int r = 0; r < 3; r++) v += jp[r * nv + k] * F[r] + jr[r * nv + k] * F[3 + r];
    u[k] = v;
  }
  u[6] = traj[6] * m->actuator_ctrlrange[2 * (m->nu - 1) + 1];
  free(jp); free(jr);
}

void o_pd_joint_ctrl(const OModel* m, const OData* d, const double* target, const double* kp, const double* kd, double* u) {
  /* reference controller_func.py:128-167 with move_j.get_joint_delta (move_j.py:30-38): delta = target - q */
  for (int i = 0; i < 6; i++) {
    double q = d->qpos[i], t = q + (target[i] - q);
    if (t < m->jnt_range[2 * i]) t = m->jnt_range[2 * i]; if (t > m->jnt_range[2 * i + 1]) t = m->jnt_range[2 * i + 1];
    double v = kp[i] * (t - q) + kd[i] * -d->qvel[i];
    if (v < m->actuator_ctrlrange[2 * i]) v = m->actuator_ctrlrange[2 * i]; if (v > m->actuator_ctrlrange[2 * i + 1]) v = m->actuator_ctrlrange[2 * i + 1];
    u[i] = v;
  }
}
