/*
 * r2ik_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE (see r2ik_oracle.h).
 *
 * Literal CPU restatement of the reference algorithm: 4x4 homogeneous matrices,
 * scipy's quaternion-based Rotation algorithms, numpy's isclose/linspace/%
 * semantics.  Deliberately written in the reference's own "frame peeling" style
 * (NOT the restructured 3-vector form the CUDA kernels use) so that the two
 * implementations are independent.
 *
 * Citations: "sik" = src/reachy2_symbolic_ik/symbolic_ik.py,
 *            "utl" = src/reachy2_symbolic_ik/utils.py,
 *            "ctl" = src/reachy2_symbolic_ik/control_ik.py,
 *            "rxp" = scipy/spatial/transform/_rotation_xp.py (scipy 1.18.1).
 */
#include "r2ik_oracle.h"

#include <math.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#define ORC_PI M_PI

typedef struct {
  orc_arm_config cfg;
  /* derived constants (sik:64-83) */
  double gripper_size;
  double max_arm_length;
  double shoulder_wrist_min_distance;
  double elbow_singularity_position[3];
  double wrist_singularity_position[3];
  /* mutable solver state: self.goal_pose / self.wrist_position /
   * self.intersection_circle / self.elbow_position of the reference */
  double goal_position[3];
  double goal_orientation[3];
  double wrist_position[3];
  double circle_center[3];
  double circle_radius;
  double circle_normal[3];
  double elbow_position[3];
} orc_solver;

/* ------------------------------------------------------------------------- */
/* numpy / python scalar semantics                                            */
/* ------------------------------------------------------------------------- */

/* Python / NumPy float `%` (result takes the sign of the divisor). */
double orc_pymod(double a, double m) {
  double r = fmod(a, m);
  if (r != 0.0) {
    if ((m < 0.0) != (r < 0.0)) r += m;
  } else {
    r = copysign(0.0, m);
  }
  return r;
}

/* np.isclose(a, b) with default rtol=1e-5, atol=1e-8 (asymmetric in b). */
static int np_isclose(double a, double b) { return fabs(a - b) <= 1e-8 + 1e-5 * fabs(b); }

static double norm3(const double v[3]) { return sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }
static double dot3(const double a[3], const double b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static void cross3(const double a[3], const double b[3], double o[3]) {
  double x = a[1] * b[2] - a[2] * b[1];
  double y = a[2] * b[0] - a[0] * b[2];
  double z = a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z;
}

/* utl:486-490 angle_diff */
double orc_angle_diff(double a, double b) {
  double d = a - b;
  return orc_pymod(d + ORC_PI, 2 * ORC_PI) - ORC_PI;
}

/* ------------------------------------------------------------------------- */
/* 4x4 homogeneous helpers (utl:12-23 make_homogenous_matrix_from_rotation_matrix) */
/* ------------------------------------------------------------------------- */
typedef struct { double m[4][4]; } mat4;

static mat4 make_homogeneous(const double p[3], const double r[3][3]) {
  mat4 t;
  for (int i = 0; i < 3; i++) {
    for (int j = 0; j < 3; j++) t.m[i][j] = r[i][j];
    t.m[i][3] = p[i];
  }
  t.m[3][0] = 0.0; t.m[3][1] = 0.0; t.m[3][2] = 0.0; t.m[3][3] = 1.0;
  return t;
}
static mat4 mat4_mul(const mat4 *a, const mat4 *b) {
  mat4 c;
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) {
      double s = 0.0;
      for (int k = 0; k < 4; k++) s += a->m[i][k] * b->m[k][j];
      c.m[i][j] = s;
    }
  return c;
}
static void mat4_apply(const mat4 *t, const double p4[4], double o4[4]) {
  for (int i = 0; i < 4; i++) {
    double s = 0.0;
    for (int k = 0; k < 4; k++) s += t->m[i][k] * p4[k];
    o4[i] = s;
  }
}
static void transpose3(const double a[3][3], double o[3][3]) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) o[i][j] = a[j][i];
}
static void matvec3(const double a[3][3], const double v[3], double o[3]) {
  for (int i = 0; i < 3; i++) o[i] = a[i][0] * v[0] + a[i][1] * v[1] + a[i][2] * v[2];
}

/* ------------------------------------------------------------------------- */
/* scipy Rotation restated (quaternion is x,y,z,w)                            */
/* ------------------------------------------------------------------------- */

/* rxp:1035-1049 _make_elementary_quat */
static void quat_elementary(int axis, double angle, double q[4]) {
  q[0] = 0.0; q[1] = 0.0; q[2] = 0.0;
  q[3] = cos(angle / 2.0);
  q[axis] = sin(angle / 2.0);
}
/* rxp:1114-1127 compose_quat */
static void quat_compose(const double p[4], const double q[4], double o[4]) {
  double c[3];
  cross3(p, q, c);
  double qx = p[3] * q[0] + q[3] * p[0] + c[0];
  double qy = p[3] * q[1] + q[3] * p[1] + c[1];
  double qz = p[3] * q[2] + q[3] * p[2] + c[2];
  double qw = p[3] * q[3] - p[0] * q[0] - p[1] * q[1] - p[2] * q[2];
  o[0] = qx; o[1] = qy; o[2] = qz; o[3] = qw;
}
/* rxp:1024-1033 _elementary_quat_compose / rxp:192-224 from_euler */
static void quat_from_euler(const int axes[3], int intrinsic, const double ang[3], double q[4]) {
  double t[4], e[4];
  quat_elementary(axes[0], ang[0], q);
  for (int i = 1; i < 3; i++) {
    quat_elementary(axes[i], ang[i], e);
    if (intrinsic) quat_compose(q, e, t); else quat_compose(e, q, t);
    memcpy(q, t, sizeof t);
  }
}
/* rxp:302-333 as_matrix */
static void quat_as_matrix(const double q[4], double m[3][3]) {
  double x = q[0], y = q[1], z = q[2], w = q[3];
  double x2 = x * x, y2 = y * y, z2 = z * z, w2 = w * w;
  double xy = x * y, zw = z * w, xz = x * z, yw = y * w, yz = y * z, xw = x * w;
  m[0][0] = x2 - y2 - z2 + w2; m[0][1] = 2 * (xy - zw);       m[0][2] = 2 * (xz + yw);
  m[1][0] = 2 * (xy + zw);     m[1][1] = -x2 + y2 - z2 + w2;  m[1][2] = 2 * (yz - xw);
  m[2][0] = 2 * (xz - yw);     m[2][1] = 2 * (yz + xw);       m[2][2] = -x2 - y2 + z2 + w2;
}

static double det3(const double m[3][3]) {
  return m[0][0] * (m[1][1] * m[2][2] - m[1][2] * m[2][1]) -
         m[0][1] * (m[1][0] * m[2][2] - m[1][2] * m[2][0]) +
         m[0][2] * (m[1][0] * m[2][1] - m[1][1] * m[2][0]);
}
static void inv3_transpose(const double a[3][3], double o[3][3]) {
  /* o = inverse(a)^T = cofactor(a) / det(a) */
  double d = det3(a);
  o[0][0] = (a[1][1] * a[2][2] - a[1][2] * a[2][1]) / d;
  o[0][1] = (a[1][2] * a[2][0] - a[1][0] * a[2][2]) / d;
  o[0][2] = (a[1][0] * a[2][1] - a[1][1] * a[2][0]) / d;
  o[1][0] = (a[0][2] * a[2][1] - a[0][1] * a[2][2]) / d;
  o[1][1] = (a[0][0] * a[2][2] - a[0][2] * a[2][0]) / d;
  o[1][2] = (a[0][1] * a[2][0] - a[0][0] * a[2][1]) / d;
  o[2][0] = (a[0][1] * a[1][2] - a[0][2] * a[1][1]) / d;
  o[2][1] = (a[0][2] * a[1][0] - a[0][0] * a[1][2]) / d;
  o[2][2] = (a[0][0] * a[1][1] - a[0][1] * a[1][0]) / d;
}

/* rxp:51-152 from_matrix.  det <= 0 -> error (ValueError in scipy).  A matrix whose
 * Gramian differs from I (isclose, rtol 1e-5 / atol 1e-12) is replaced by U @ Vt of its
 * SVD, i.e. by its orthogonal polar factor; here that factor is computed with the
 * Newton iteration X <- (X + X^-T)/2, which converges to the same (unique) matrix. */
static int quat_from_matrix(const double min[3][3], double q[4]) {
  double m[3][3];
  memcpy(m, min, sizeof m);
  if (!(det3(m) > 0.0)) return -1;
  int orthogonal = 1;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double g = m[i][0] * m[j][0] + m[i][1] * m[j][1] + m[i][2] * m[j][2];
      double e = (i == j) ? 1.0 : 0.0;
      if (!(fabs(g - e) <= 1e-12 + 1e-5 * fabs(e))) orthogonal = 0;
    }
  if (!orthogonal) {
    /* U @ Vt does not depend on the scale of the block, while the iteration only halves a scale error per step:
     * a block whose largest entry lies outside [2^-4, 2^4] is first scaled to unit size by an exact power of two. */
    double mx = 0.0;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) mx = fmax(mx, fabs(m[i][j]));
    if (mx < 0.0625 || (mx > 16.0 && mx < INFINITY)) {
      int e = ilogb(mx);
      for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) m[i][j] = ldexp(m[i][j], -e);
    }
    for (int it = 0; it < 60; it++) {
      double y[3][3], delta = 0.0;
      inv3_transpose(m, y);
      for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
          double nx = 0.5 * (m[i][j] + y[i][j]);
          delta = fmax(delta, fabs(nx - m[i][j]));
          m[i][j] = nx;
        }
      if (delta < 1e-16) break;
    }
  }
  /* rxp:100-156 _from_matrix_orthogonal (Shepperd / Markley) */
  double tr = m[0][0] + m[1][1] + m[2][2];
  double dec[4] = {m[0][0], m[1][1], m[2][2], tr};
  int choice = 0;
  for (int i = 1; i < 4; i++)
    if (dec[i] > dec[choice]) choice = i; /* argmax: first maximum wins */
  if (choice == 0) {
    q[0] = 1 - tr + 2 * m[0][0]; q[1] = m[1][0] + m[0][1];
    q[2] = m[2][0] + m[0][2];    q[3] = m[2][1] - m[1][2];
  } else if (choice == 1) {
    q[0] = m[1][0] + m[0][1];    q[1] = 1 - tr + 2 * m[1][1];
    q[2] = m[2][1] + m[1][2];    q[3] = m[0][2] - m[2][0];
  } else if (choice == 2) {
    q[0] = m[2][0] + m[0][2];    q[1] = m[2][1] + m[1][2];
    q[2] = 1 - tr + 2 * m[2][2]; q[3] = m[1][0] - m[0][1];
  } else {
    q[0] = m[2][1] - m[1][2];    q[1] = m[0][2] - m[2][0];
    q[2] = m[1][0] - m[0][1];    q[3] = 1 + tr;
  }
  double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int i = 0; i < 4; i++) q[i] /= n;
  return 0;
}

/* rxp:365-404 as_euler + rxp:1052-1111 _get_angles.  seq_axes as written ("ZYZ" -> 2,1,2). */
static void quat_as_euler(const double q[4], const int seq_axes[3], int extrinsic, double out[3]) {
  int i, j, k;
  if (extrinsic) { i = seq_axes[0]; j = seq_axes[1]; k = seq_axes[2]; }
  else           { i = seq_axes[2]; j = seq_axes[1]; k = seq_axes[0]; }
  int symmetric = (i == k);
  if (symmetric) k = 3 - i - j;
  int prod = (i - j) * (j - k) * (k - i);
  double sign = (double)(prod / 2); /* exact: prod is +-2 */
  double a, b, c, d;
  if (symmetric) { a = q[3]; b = q[i]; c = q[j]; d = q[k] * sign; }
  else { a = q[3] - q[j]; b = q[i] + q[k] * sign; c = q[j] + q[3]; d = q[k] * sign - q[i]; }
  const double eps = 1e-7, lamb = ORC_PI / 2;
  double half_sum = atan2(b, a);
  double half_diff = atan2(d, c);
  double ang[3] = {0.0, 0.0, 0.0};
  ang[1] = 2 * atan2(hypot(c, d), hypot(a, b));
  int first = extrinsic ? 0 : 2, third = extrinsic ? 2 : 0;
  int case1 = fabs(ang[1]) <= eps;
  int case2 = fabs(ang[1] - ORC_PI) <= eps;
  int case0 = !(case1 || case2);
  ang[0] = case1 ? 2 * half_sum : 2 * half_diff * (extrinsic ? -1.0 : 1.0);
  ang[first] = case0 ? half_sum - half_diff : ang[first];
  double a3 = case0 ? half_sum + half_diff : ang[third];
  if (!symmetric) {
    a3 = a3 * sign;
    ang[1] = ang[1] - lamb;
  }
  ang[third] = a3;
  for (int t = 0; t < 3; t++) out[t] = orc_pymod(ang[t] + ORC_PI, 2 * ORC_PI) - ORC_PI;
}

static const int AX_XYZ[3] = {0, 1, 2};
static const int AX_ZYZ[3] = {2, 1, 2};

/* R.from_euler("xyz", e).as_matrix() */
static void rot_from_euler_xyz(const double e[3], double m[3][3]) {
  double q[4];
  quat_from_euler(AX_XYZ, 0, e, q);
  quat_as_matrix(q, m);
}
void orc_matrix_from_euler_xyz(const double euler[3], double m9[9]) {
  double m[3][3];
  rot_from_euler_xyz(euler, m);
  memcpy(m9, m, sizeof m);
}
/* utl:84-90 get_euler_from_homogeneous_matrix: R.from_matrix(M[:3,:3]).as_euler("xyz") */
void orc_euler_xyz_from_matrix(const double m9[9], double euler[3], int *status) {
  double m[3][3], q[4];
  memcpy(m, m9, sizeof m);
  int rc = quat_from_matrix(m, q);
  if (status) *status = rc;
  if (rc) { euler[0] = euler[1] = euler[2] = NAN; return; }
  quat_as_euler(q, AX_XYZ, 1, euler);
}

/* utl:508-519 limit_orbita3d_joints */
void orc_limit_orbita3d_joints(const double in3[3], double max_angle, double out3[3]) {
  double q[4], zyz[3];
  quat_from_euler(AX_XYZ, 1, in3, q);          /* from_euler("XYZ") */
  quat_as_euler(q, AX_ZYZ, 0, zyz);            /* as_euler("ZYZ")   */
  zyz[1] = fmin(max_angle, fmax(-max_angle, zyz[1]));
  quat_from_euler(AX_ZYZ, 1, zyz, q);          /* from_euler("ZYZ") */
  quat_as_euler(q, AX_XYZ, 0, out3);           /* as_euler("XYZ")   */
}

/* ------------------------------------------------------------------------- */
/* utils.py geometry helpers                                                  */
/* ------------------------------------------------------------------------- */

/* utl:59-81 rotation_matrix_from_vector */
static void rotation_matrix_from_vector(const double vect[3], double r[3][3]) {
  double n = norm3(vect);
  double u[3] = {vect[0] / n, vect[1] / n, vect[2] / n};
  static const double ex[3] = {1.0, 0.0, 0.0};
  memset(r, 0, 9 * sizeof(double));
  if (np_isclose(ex[0], u[0]) && np_isclose(ex[1], u[1]) && np_isclose(ex[2], u[2])) {
    r[0][0] = 1; r[1][1] = 1; r[2][2] = 1;
    return;
  }
  if (np_isclose(ex[0], -u[0]) && np_isclose(ex[1], -u[1]) && np_isclose(ex[2], -u[2])) {
    r[0][0] = -1; r[1][1] = 1; r[2][2] = -1;
    return;
  }
  double v[3];
  cross3(ex, u, v);
  double c = dot3(ex, u);
  double s = norm3(v);
  double k[3][3] = {{0, -v[2], v[1]}, {v[2], 0, -v[0]}, {-v[1], v[0], 0}};
  double f = (1 - c) / (s * s);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double kk = k[i][0] * k[0][j] + k[i][1] * k[1][j] + k[i][2] * k[2][j];
      r[i][j] = (i == j ? 1.0 : 0.0) + k[i][j] + kk * f;
    }
}
void orc_rotation_matrix_from_vector(const double v[3], double m9[9]) {
  double r[3][3];
  rotation_matrix_from_vector(v, r);
  memcpy(m9, r, sizeof r);
}

/* utl:477-483 make_projection_on_plane */
static void make_projection_on_plane(const double p_plane[3], const double nrm[3], const double pt[3], double o[3]) {
  double v[3] = {pt[0] - p_plane[0], pt[1] - p_plane[1], pt[2] - p_plane[2]};
  double dist = dot3(v, nrm);
  for (int i = 0; i < 3; i++) o[i] = pt[i] - dist * nrm[i];
}

/* utl:468-474 is_valid_angle */
static int is_valid_angle(double angle, const double interval[2]) {
  if (orc_pymod(interval[0], 2 * ORC_PI) == orc_pymod(interval[1], 2 * ORC_PI)) return 1;
  if (interval[0] < interval[1]) return (interval[0] <= angle) && (angle <= interval[1]);
  return (interval[0] <= angle) || (angle <= interval[1]);
}

/* utl:93-112 limit_theta_to_interval */
void orc_limit_theta_to_interval(double theta, double previous_theta, const double interval[2], double *out) {
  theta = orc_pymod(theta, 2 * ORC_PI);
  if (theta > ORC_PI) theta -= 2 * ORC_PI;
  previous_theta = orc_pymod(previous_theta, 2 * ORC_PI);
  if (previous_theta > ORC_PI) previous_theta -= 2 * ORC_PI;
  (void)previous_theta;
  if (is_valid_angle(theta, interval)) { *out = theta; return; }
  double pos_diff = orc_angle_diff(theta, interval[1]);
  double neg_diff = orc_angle_diff(theta, interval[0]);
  if (fabs(pos_diff) < fabs(neg_diff)) { *out = interval[1]; return; }
  *out = interval[0];
}

/* utl:443-465 is_elbow_ok (the first test, utl:452-455, is dead: overwritten at :457) */
static int is_elbow_ok(const double e[3], int side, double sing_offset, double sing_coeff, const double esp[3]) {
  int ok = (e[1] * side < -0.2);
  ok = ok && (e[2] < (e[0] - esp[0]) * sing_coeff + esp[2] - sing_offset);
  return ok;
}

/* ------------------------------------------------------------------------- */
/* SymbolicIK                                                                 */
/* ------------------------------------------------------------------------- */

/* utl:26-43 get_singularity_position */
static void get_singularity_position(const orc_arm_config *c, double elbow[3], double wrist[3]) {
  double q[4], r[3][3], e[3];
  /* from_euler("xyz", offset, degrees=True): deg2rad then compose */
  for (int i = 0; i < 3; i++) e[i] = c->shoulder_orientation_deg[i] * (ORC_PI / 180.0);
  quat_from_euler(AX_XYZ, 0, e, q);
  quat_as_matrix(q, r);
  mat4 t = make_homogeneous(c->shoulder_position, r);
  double pe[4] = {0.0, -c->upper_arm_size * c->side, 0.0, 1.0}, o[4];
  mat4_apply(&t, pe, o);
  memcpy(elbow, o, 3 * sizeof(double));
  double pw[4] = {0.0, -(c->upper_arm_size + c->forearm_size) * c->side, 0.0, 1.0};
  mat4_apply(&t, pw, o);
  memcpy(wrist, o, 3 * sizeof(double));
}

/* sik:26-83 SymbolicIK.__init__ */
static void solver_init(orc_solver *s, const orc_arm_config *cfg) {
  memset(s, 0, sizeof *s);
  s->cfg = *cfg;
  s->gripper_size = norm3(cfg->tip_position);
  s->max_arm_length = cfg->upper_arm_size + cfg->forearm_size + s->gripper_size;
  double L1 = cfg->upper_arm_size, L2 = cfg->forearm_size;
  s->shoulder_wrist_min_distance =
      sqrt(L1 * L1 + L2 * L2 - 2 * L1 * L2 * cos((180 - cfg->elbow_limit_deg) * (ORC_PI / 180.0)));
  get_singularity_position(cfg, s->elbow_singularity_position, s->wrist_singularity_position);
}

/* sik:284-307 is_pose_in_robot_reach */
static int is_pose_in_robot_reach(const orc_solver *s, const double pos_in[3], double pos[3], int *state) {
  const double *sh = s->cfg.shoulder_position;
  memcpy(pos, pos_in, 3 * sizeof(double));
  double dv[3] = {pos[0] - sh[0], pos[1] - sh[1], pos[2] - sh[2]};
  double d = norm3(dv);
  int ok = 1;
  *state = -1;
  if (d > s->max_arm_length) {
    ok = 0;
    double nd = norm3(dv) + s->cfg.projection_margin;
    for (int i = 0; i < 3; i++) pos[i] = sh[i] + (dv[i] / nd) * s->max_arm_length;
    *state = ORC_STATE_POSE_OUT_OF_REACH;
  }
  if (pos[0] < s->cfg.backward_limit) {
    ok = 0;
    pos[0] = s->cfg.backward_limit;
    *state = ORC_STATE_BACKWARD_POSE;
  }
  return ok;
}

/* sik:418-425 get_wrist_position */
static void get_wrist_position(const orc_solver *s, const double pos[3], const double eul[3], double w[3]) {
  double r[3][3];
  rot_from_euler_xyz(eul, r);
  mat4 t = make_homogeneous(pos, r);
  const double *tip = s->cfg.tip_position;
  double p[4] = {-tip[0], tip[1], tip[2], 1.0}, o[4];
  mat4_apply(&t, p, o);
  memcpy(w, o, 3 * sizeof(double));
}

/* sik:337-349 reduce_goal_pose_no_limits (mutates s->wrist_position) */
static void reduce_goal_pose_no_limits(orc_solver *s, double pos[3], double d_sw, double d_max) {
  const double *sh = s->cfg.shoulder_position;
  double den = fabs(d_sw) + s->cfg.projection_margin;
  double nw[3], diff[3];
  for (int i = 0; i < 3; i++) {
    double dir = (s->wrist_position[i] - sh[i]) / den;
    nw[i] = sh[i] + dir * d_max;
    diff[i] = nw[i] - s->wrist_position[i];
  }
  for (int i = 0; i < 3; i++) {
    pos[i] = pos[i] + diff[i];
    s->wrist_position[i] = nw[i];
  }
}

/* sik:366-399 get_intersection_circle; returns 0 if the spheres do not intersect */
static int get_intersection_circle(orc_solver *s) {
  const double *sh = s->cfg.shoulder_position;
  double L1 = s->cfg.upper_arm_size, L2 = s->cfg.forearm_size;
  double P[3] = {s->wrist_position[0] - sh[0], s->wrist_position[1] - sh[1], s->wrist_position[2] - sh[2]};
  double d = sqrt(P[0] * P[0] + P[1] * P[1] + P[2] * P[2]);
  if (d > L1 + L2) return 0;
  double e[3] = {0.0, -asin(P[2] / d), atan2(P[1], P[0])};
  double r[3][3];
  rot_from_euler_xyz(e, r);
  double d2 = d * d, L1s = L1 * L1, L2s = L2 * L2;
  double k = d2 - L2s + L1s;
  double radius = 1 / (2 * d) * sqrt(4 * d2 * L1s - k * k);
  double pc[3] = {k / (2 * d), 0.0, 0.0}, psc[3];
  matvec3(r, pc, psc);
  for (int i = 0; i < 3; i++) s->circle_center[i] = psc[i] + sh[i];
  s->circle_radius = radius;
  double ex[3] = {1.0, 0.0, 0.0};
  matvec3(r, ex, s->circle_normal);
  return 1;
}

/* sik:401-416 get_limitation_wrist_circle */
static void get_limitation_wrist_circle(const orc_solver *s, const double pos[3], double center[3], double *radius, double normal[3]) {
  double L2 = s->cfg.forearm_size;
  for (int i = 0; i < 3; i++) normal[i] = s->wrist_position[i] - pos[i];
  *radius = sin(s->cfg.wrist_limit_deg * (ORC_PI / 180.0)) * L2;
  double n = norm3(normal);
  double h = sqrt(L2 * L2 - (*radius) * (*radius));
  for (int i = 0; i < 3; i++) center[i] = s->wrist_position[i] + normal[i] / n * h;
}

/* sik:570-586 intersection_point: least-squares solution of [v1 -v2](t,u)^T = p02-p01
 * (np.linalg.lstsq -> LAPACK gelsd in the reference; a Householder-free 3x2 QR here --
 * the system is consistent and full rank, so both yield the unique solution). */
static int intersection_point(const double v1[3], const double p01[3], const double v2[3], const double p02[3], double q[3]) {
  double a0[3] = {v1[0], v1[1], v1[2]};
  double a1[3] = {-v2[0], -v2[1], -v2[2]};
  double b[3] = {p02[0] - p01[0], p02[1] - p01[1], p02[2] - p01[2]};
  /* modified Gram-Schmidt QR */
  double r00 = norm3(a0);
  double q0[3] = {a0[0] / r00, a0[1] / r00, a0[2] / r00};
  double r01 = dot3(q0, a1);
  double w[3] = {a1[0] - r01 * q0[0], a1[1] - r01 * q0[1], a1[2] - r01 * q0[2]};
  double r11 = norm3(w);
  double q1[3] = {w[0] / r11, w[1] / r11, w[2] / r11};
  double c0 = dot3(q0, b), c1 = dot3(q1, b);
  double u = c1 / r11;
  double t = (c0 - r01 * u) / r00;
  /* np.all(np.isclose(params, params[0])) */
  if (np_isclose(t, t) && np_isclose(u, t)) return 0;
  for (int i = 0; i < 3; i++) q[i] = v1[i] * t + p01[i];
  return 1;
}

/* sik:588-606 points_of_nearest_approach */
static int points_of_nearest_approach(const double p1[3], const double n1[3], const double p2[3], const double n2[3], double q[3], double v[3]) {
  cross3(n1, n2, v);
  double nv = norm3(v);
  for (int i = 0; i < 3; i++) v[i] /= nv;
  double vect1[3], vect2[3];
  cross3(v, n1, vect1);
  cross3(v, n2, vect2);
  return intersection_point(vect1, p1, vect2, p2, q);
}

/* sik:608-645 intersection_circle_line_3d_vd; returns number of points (0 = None) */
static int intersection_circle_line(const double center[3], double radius, const double dir[3], const double pl[3], double pts[2][3]) {
  double w[3] = {pl[0] - center[0], pl[1] - center[1], pl[2] - center[2]};
  double a = dot3(dir, dir);
  double b = 2 * dot3(dir, w);
  double c = dot3(w, w) - radius * radius;
  double disc = b * b - 4 * a * c;
  if (disc < 0) return 0;
  if (disc == 0) {
    double t = -b / (2 * a);
    for (int i = 0; i < 3; i++) pts[0][i] = pl[i] + t * dir[i];
    return 1;
  }
  double t1 = (-b + sqrt(disc)) / (2 * a);
  double t2 = (-b - sqrt(disc)) / (2 * a);
  for (int i = 0; i < 3; i++) {
    pts[0][i] = pl[i] + t1 * dir[i];
    pts[1][i] = pl[i] + t2 * dir[i];
  }
  return 2;
}

/* sik:511-568 get_interval_from_intersection */
static void get_interval_from_intersection(int npts, double pts[2][3], const mat4 *T_it, const mat4 *T_ti, const mat4 *T_lt, double radius2, double interval[2]) {
  double p4[4], o[4];
  if (npts == 1) {
    p4[0] = pts[0][0]; p4[1] = pts[0][1]; p4[2] = pts[0][2]; p4[3] = 1;
    mat4_apply(T_it, p4, o);
    double angle = atan2(o[2], o[1]);
    interval[0] = angle; interval[1] = angle;
    return;
  }
  p4[0] = pts[0][0]; p4[1] = pts[0][1]; p4[2] = pts[0][2]; p4[3] = 1;
  mat4_apply(T_it, p4, o);
  double angle1 = atan2(o[2], o[1]);
  p4[0] = pts[1][0]; p4[1] = pts[1][1]; p4[2] = pts[1][2]; p4[3] = 1;
  mat4_apply(T_it, p4, o);
  double angle2 = atan2(o[2], o[1]);
  if (angle2 < angle1) { double t = angle1; angle1 = angle2; angle2 = t; } /* sorted() */
  double angle_test = (angle1 + angle2) / 2;
  double tp[4] = {0, cos(angle_test) * radius2, sin(angle_test) * radius2, 1}, tt[4], tl[4];
  mat4_apply(T_ti, tp, tt);
  mat4_apply(T_lt, tt, tl);
  if (tl[0] > 0) { interval[0] = angle1; interval[1] = angle2; }
  else { interval[0] = angle2; interval[1] = angle1; }
}

/* sik:427-509 are_circles_linked; returns 1 with interval set, 0 for the empty interval */
static int are_circles_linked(const orc_solver *s, const double lc[3], double lr, const double ln[3], double interval[2]) {
  double radius1 = lr, radius2 = s->circle_radius;
  double p1[3], p2[3];
  for (int i = 0; i < 3; i++) {
    p1[i] = lc[i] - s->wrist_position[i];
    p2[i] = s->circle_center[i] - s->wrist_position[i];
  }
  double n1[3] = {ln[0], ln[1], ln[2]};
  double n2[3] = {s->circle_normal[0], s->circle_normal[1], s->circle_normal[2]};

  double R_ti[3][3], R_it[3][3], P_it[3];
  rotation_matrix_from_vector(n2, R_ti);
  mat4 T_ti = make_homogeneous(p2, R_ti);
  transpose3(R_ti, R_it);
  double nR[3][3];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) nR[i][j] = -R_it[i][j];
  matvec3(nR, p2, P_it);
  mat4 T_it = make_homogeneous(P_it, R_it);

  double R_tl[3][3], R_lt[3][3], P_lt[3];
  rotation_matrix_from_vector(n1, R_tl);
  transpose3(R_tl, R_lt);
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) nR[i][j] = -R_lt[i][j];
  matvec3(nR, p1, P_lt);
  mat4 T_lt = make_homogeneous(P_lt, R_lt);

  double c2[4] = {p2[0], p2[1], p2[2], 1}, plc[4];
  mat4_apply(&T_lt, c2, plc);

  if (n1[0] != 0 || n1[1] != 0 || n1[2] != 0) { double n = norm3(n1); for (int i = 0; i < 3; i++) n1[i] /= n; }
  if (n2[0] != 0 || n2[1] != 0 || n2[2] != 0) { double n = norm3(n2); for (int i = 0; i < 3; i++) n2[i] /= n; }

  double mg = s->cfg.normal_vector_margin;
  int par_a = 1, par_b = 1;
  for (int i = 0; i < 3; i++) {
    if (!(fabs(n2[i] - n1[i]) < mg)) par_a = 0;
    if (!(fabs(n2[i] + n1[i]) < mg)) par_b = 0;
  }
  if (par_a || par_b) {
    if (plc[0] > 0) { interval[0] = -ORC_PI; interval[1] = ORC_PI; return 1; }
    return 0;
  }
  double q[3], v[3];
  if (!points_of_nearest_approach(p1, n1, p2, n2, q, v)) {
    if (plc[0] > 0) { interval[0] = -ORC_PI; interval[1] = ORC_PI; return 1; }
    return 0;
  }
  double pts[2][3];
  int np_ = intersection_circle_line(p1, radius1, v, q, pts);
  if (np_ == 0) {
    if (plc[0] > 0) { interval[0] = -ORC_PI; interval[1] = ORC_PI; return 1; }
    return 0;
  }
  get_interval_from_intersection(np_, pts, &T_it, &T_ti, &T_lt, radius2, interval);
  return 1;
}

/* sik:121-282 is_reachable */
static int solver_is_reachable(orc_solver *s, const double pos_in[3], const double eul[3], double interval[2], int *state) {
  double pos[3];
  int rs;
  int ok = is_pose_in_robot_reach(s, pos_in, pos, &rs);
  interval[0] = NAN; interval[1] = NAN;
  if (!ok) { *state = rs; return 0; }
  memcpy(s->goal_position, pos, sizeof pos);
  memcpy(s->goal_orientation, eul, 3 * sizeof(double));
  get_wrist_position(s, pos, eul, s->wrist_position);
  if (s->wrist_position[0] < s->cfg.backward_limit) {
    double diff = s->cfg.backward_limit - s->wrist_position[0];
    pos[0] = pos[0] + diff;
    s->wrist_position[0] = s->wrist_position[0] + diff;
    memcpy(s->goal_position, pos, sizeof pos);
  }
  const double *sh = s->cfg.shoulder_position;
  double dv[3] = {s->wrist_position[0] - sh[0], s->wrist_position[1] - sh[1], s->wrist_position[2] - sh[2]};
  double d = norm3(dv);
  if (d > s->cfg.upper_arm_size + s->cfg.forearm_size) { *state = ORC_STATE_WRIST_OUT_OF_RANGE; return 0; }
  if (d < s->shoulder_wrist_min_distance) {
    reduce_goal_pose_no_limits(s, pos, d, s->shoulder_wrist_min_distance);
    get_wrist_position(s, pos, eul, s->wrist_position);
    memcpy(s->goal_position, pos, sizeof pos);
  }
  int has_circle = get_intersection_circle(s);
  double lc[3], lr, ln[3];
  get_limitation_wrist_circle(s, pos, lc, &lr, ln);
  if (has_circle) {
    if (are_circles_linked(s, lc, lr, ln, interval)) { *state = ORC_STATE_REACHABLE; return 1; }
    interval[0] = NAN; interval[1] = NAN;
    *state = ORC_STATE_LIMITED_BY_WRIST;
    return 0;
  }
  *state = ORC_STATE_SHOULD_NOT_HAPPEN;
  return 0;
}

/* sik:85-119 is_reachable_no_limits */
static int solver_is_reachable_no_limits(orc_solver *s, const double pos_in[3], const double eul[3]) {
  double pos[3];
  int rs;
  is_pose_in_robot_reach(s, pos_in, pos, &rs);
  memcpy(s->goal_position, pos, sizeof pos);
  memcpy(s->goal_orientation, eul, 3 * sizeof(double));
  get_wrist_position(s, pos, eul, s->wrist_position);
  if (s->wrist_position[0] < s->cfg.backward_limit) {
    double diff = s->cfg.backward_limit - s->wrist_position[0];
    pos[0] = pos[0] + diff;
    get_wrist_position(s, pos, eul, s->wrist_position);
    memcpy(s->goal_position, pos, sizeof pos);
  }
  const double *sh = s->cfg.shoulder_position;
  double dv[3] = {s->wrist_position[0] - sh[0], s->wrist_position[1] - sh[1], s->wrist_position[2] - sh[2]};
  double d = norm3(dv);
  double L12 = s->cfg.upper_arm_size + s->cfg.forearm_size;
  if (d > L12) {
    /* sik:102-105: self.goal_pose = reduce(...); the LOCAL goal_pose is left untouched */
    double gp[3] = {pos[0], pos[1], pos[2]};
    reduce_goal_pose_no_limits(s, gp, d, L12);
    memcpy(s->goal_position, gp, sizeof gp);
  }
  if (d < s->shoulder_wrist_min_distance) {
    reduce_goal_pose_no_limits(s, pos, d, s->shoulder_wrist_min_distance);
    get_wrist_position(s, pos, eul, s->wrist_position);
    memcpy(s->goal_position, pos, sizeof pos);
  }
  return get_intersection_circle(s);
}

/* sik:684-695 get_elbow_position */
static void get_elbow_position(const orc_solver *s, double theta, double e[3]) {
  double r[3][3];
  rotation_matrix_from_vector(s->circle_normal, r);
  mat4 t = make_homogeneous(s->circle_center, r);
  double p[4] = {0, s->circle_radius * cos(theta), s->circle_radius * sin(theta), 1}, o[4];
  mat4_apply(&t, p, o);
  memcpy(e, o, 3 * sizeof(double));
}

/* sik:647-682 make_elbow_projection */
static void make_elbow_projection(const orc_solver *s, const double goal[3], const double elbow[3], double new_goal[3], double new_elbow[3]) {
  double coeff = s->cfg.singularity_limit_coeff;
  double alpha = atan2(-coeff, 1);
  double e[3] = {0, alpha, 0}, M[3][3];
  rot_from_euler_xyz(e, M);
  mat4 T = make_homogeneous(s->elbow_singularity_position, M);
  double p0[4] = {0, 0, -s->cfg.singularity_offset, 1}, P[4];
  mat4_apply(&T, p0, P);
  T = make_homogeneous(P, M);
  double n1[4] = {1, 0, 0, 1}, n2[4] = {0, 1, 0, 1}, o1[4], o2[4];
  mat4_apply(&T, n1, o1);
  mat4_apply(&T, n2, o2);
  double v1[3] = {o1[0] - P[0], o1[1] - P[1], o1[2] - P[2]};
  double v2[3] = {o2[0] - P[0], o2[1] - P[1], o2[2] - P[2]};
  double v3[3];
  cross3(v1, v2, v3);
  double n = norm3(v3);
  for (int i = 0; i < 3; i++) v3[i] /= n;
  const double *sh = s->cfg.shoulder_position;
  double pc[3];
  make_projection_on_plane(P, v3, sh, pc);
  double dsc[3] = {sh[0] - pc[0], sh[1] - pc[1], sh[2] - pc[2]};
  double nd = norm3(dsc);
  double radius = sqrt(s->cfg.upper_arm_size * s->cfg.upper_arm_size - nd * nd);
  double pe[3];
  make_projection_on_plane(P, v3, elbow, pe);
  double vc[3] = {pe[0] - pc[0], pe[1] - pc[1], pe[2] - pc[2]};
  double nvc = norm3(vc);
  for (int i = 0; i < 3; i++) new_elbow[i] = pc[i] + radius * (vc[i] / nvc);
  for (int i = 0; i < 3; i++) new_goal[i] = goal[i] + (new_elbow[i] - elbow[i]);
}

static mat4 elementary_T(int axis, double angle) {
  double e[3] = {0, 0, 0}, r[3][3], z[3] = {0, 0, 0};
  e[axis] = angle;
  rot_from_euler_xyz(e, r);
  return make_homogeneous(z, r);
}

/* sik:697-863 get_joints (mutates the solver exactly like the reference when the
 * elbow projection fires: goal_pose, elbow_position, wrist_position) */
static void solver_get_joints(orc_solver *s, double theta, const double previous_joints[7], double joints[7], double elbow_out[3]) {
  const orc_arm_config *c = &s->cfg;
  get_elbow_position(s, theta, s->elbow_position);
  if (s->elbow_position[2] >
      (s->elbow_position[0] - s->elbow_singularity_position[0]) * c->singularity_limit_coeff +
          s->elbow_singularity_position[2] - c->singularity_offset) {
    double ng[3], ne[3];
    make_elbow_projection(s, s->goal_position, s->elbow_position, ng, ne);
    memcpy(s->goal_position, ng, sizeof ng);
    memcpy(s->elbow_position, ne, sizeof ne);
    get_wrist_position(s, s->goal_position, s->goal_orientation, s->wrist_position);
  }
  const double *go = s->goal_orientation;
  double P_t_sh[4] = {c->shoulder_position[0], c->shoulder_position[1], c->shoulder_position[2], 1};
  double P_t_el[4] = {s->elbow_position[0], s->elbow_position[1], s->elbow_position[2], 1};
  double P_t_wr[4] = {s->wrist_position[0], s->wrist_position[1], s->wrist_position[2], 1};
  double P_t_goal[4] = {s->goal_position[0], s->goal_position[1], s->goal_position[2], 1};

  /* sik:728-733 M_torso_shoulder = R(xyz, rad(offset)) * R(xyz,[0,pi/2,0]) */
  double q1[4], q2[4], q12[4], eo[3], e90[3] = {0.0, ORC_PI / 2, 0.0};
  for (int i = 0; i < 3; i++) eo[i] = c->shoulder_orientation_deg[i] * (ORC_PI / 180.0);
  quat_from_euler(AX_XYZ, 0, eo, q1);
  quat_from_euler(AX_XYZ, 0, e90, q2);
  quat_compose(q1, q2, q12);
  { /* Rotation.__mul__ re-normalises the product (scipy _rotation.py:1802-1805) */
    double qn = sqrt(q12[0] * q12[0] + q12[1] * q12[1] + q12[2] * q12[2] + q12[3] * q12[3]);
    for (int i = 0; i < 4; i++) q12[i] /= qn;
  }
  double M_ts[3][3], M_st[3][3], nM[3][3], P_sh_t[3];
  quat_as_matrix(q12, M_ts);
  transpose3(M_ts, M_st);
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) nM[i][j] = -M_st[i][j];
  matvec3(nM, P_t_sh, P_sh_t);
  mat4 T_sh_t = make_homogeneous(P_sh_t, M_st);

  double P[4];
  mat4_apply(&T_sh_t, P_t_el, P);
  double shoulder_pitch;
  if (P[0] == 0 && P[2] == 0) shoulder_pitch = previous_joints[0];
  else shoulder_pitch = -atan2(P[2], P[0]);

  mat4 T1 = elementary_T(1, -shoulder_pitch);
  mat4 T_sp_t = mat4_mul(&T1, &T_sh_t);
  mat4_apply(&T_sp_t, P_t_el, P);
  double shoulder_roll = atan2(P[1], P[0]);

  mat4 T2 = elementary_T(2, -shoulder_roll);
  mat4 T_el_t = mat4_mul(&T2, &T_sp_t);
  T_el_t.m[0][3] -= c->upper_arm_size;

  mat4_apply(&T_el_t, P_t_wr, P);
  double elbow_yaw;
  if (P[1] == 0 && P[2] == 0) elbow_yaw = previous_joints[2];
  else elbow_yaw = -ORC_PI / 2 + atan2(P[2], -P[1]);

  mat4 T3 = elementary_T(0, elbow_yaw);
  mat4 T_ey_t = mat4_mul(&T3, &T_el_t);
  mat4_apply(&T_ey_t, P_t_wr, P);
  double elbow_pitch = -atan2(P[2], P[0]);

  mat4 T4 = elementary_T(1, -elbow_pitch);
  mat4 T_wr_t = mat4_mul(&T4, &T_ey_t);
  T_wr_t.m[0][3] -= c->forearm_size;

  double Rg[3][3];
  rot_from_euler_xyz(go, Rg);
  mat4 T_t_goal = make_homogeneous(P_t_goal, Rg);
  double P_g_tip[4] = {-c->tip_position[0], c->tip_position[1], 0, 1.0}, P_t_tip[4];
  mat4_apply(&T_t_goal, P_g_tip, P_t_tip);

  mat4_apply(&T_wr_t, P_t_tip, P);
  double wrist_roll = ORC_PI - atan2(P[1], -P[0]);
  if (wrist_roll > ORC_PI) wrist_roll = wrist_roll - 2 * ORC_PI;

  mat4 T5 = elementary_T(2, -wrist_roll);
  mat4 T_wrr_t = mat4_mul(&T5, &T_wr_t);
  mat4_apply(&T_wrr_t, P_t_tip, P);
  double wrist_pitch = atan2(P[2], P[0]);

  mat4 T6 = elementary_T(1, wrist_pitch);
  mat4 T_tip_t = mat4_mul(&T6, &T_wrr_t);
  T_tip_t.m[0][3] -= c->tip_position[2];

  double P_goal_point[4] = {0.1, 0.0, 0.0, 1.0}, P_t_point[4];
  mat4 T_t_g2 = make_homogeneous(P_t_tip, Rg);
  mat4_apply(&T_t_g2, P_goal_point, P_t_point);
  mat4_apply(&T_tip_t, P_t_point, P);
  double wrist_yaw = -atan2(P[1], P[2]);

  joints[0] = shoulder_pitch; joints[1] = shoulder_roll; joints[2] = elbow_yaw; joints[3] = elbow_pitch;
  joints[4] = wrist_roll; joints[5] = -wrist_pitch; joints[6] = -wrist_yaw;
  double el = c->elbow_limit_deg * (ORC_PI / 180.0);
  if (joints[3] > el) joints[3] = el;
  if (joints[3] < -el) joints[3] = -el;
  if (elbow_out) memcpy(elbow_out, s->elbow_position, 3 * sizeof(double));
}

/* ------------------------------------------------------------------------- */
/* theta policies (utils.py)                                                  */
/* ------------------------------------------------------------------------- */

/* np.linspace(start, stop, num)[i] (endpoint=True) */
static double np_linspace_at(double start, double stop, int num, int i) {
  int div = num - 1;
  double delta = stop - start;
  if (div <= 0) return start;
  if (i == num - 1) return stop;
  double step = delta / div;
  if (step == 0.0) return ((double)i / div) * delta + start;
  return (double)i * step + start;
}

/* utl:334-396 get_best_discrete_theta; returns found flag, theta in *out */
static int get_best_discrete_theta(const orc_solver *s, double previous_theta, const double interval[2], int nb, double preferred_theta, double *out) {
  const orc_arm_config *c = &s->cfg;
  double e[3];
  if (is_valid_angle(preferred_theta, interval)) {
    get_elbow_position(s, preferred_theta, e);
    if (is_elbow_ok(e, c->side, c->singularity_offset, c->singularity_limit_coeff, s->elbow_singularity_position)) {
      *out = preferred_theta;
      return 1;
    }
  }
  double start, stop;
  if (fabs(fabs(interval[0]) + fabs(interval[1]) - 2 * ORC_PI) < 0.00001) {
    start = ORC_PI / 2; stop = ORC_PI / 2 + 2 * ORC_PI;
  } else if (interval[0] < interval[1]) {
    start = interval[0]; stop = interval[1];
  } else {
    start = interval[0]; stop = interval[1] + 2 * ORC_PI;
  }
  int found = 0;
  double best_theta = 0, best_distance = INFINITY;
  for (int i = 0; i < nb; i++) {
    double theta = np_linspace_at(start, stop, nb, i);
    get_elbow_position(s, theta, e);
    if (is_elbow_ok(e, c->side, c->singularity_offset, c->singularity_limit_coeff, s->elbow_singularity_position)) {
      double distance = fabs(orc_angle_diff(theta, preferred_theta));
      if (distance < best_distance) { best_theta = theta; best_distance = distance; found = 1; }
    }
  }
  if (found) { *out = best_theta; return 1; }
  *out = previous_theta;
  return 0;
}

/* utl:220-264 get_best_continuous_theta2 */
static int get_best_continuous_theta2(const orc_solver *s, double previous_theta, const double interval[2], int nb, double d_theta_max, double preferred_theta, double *out) {
  double theta_goal;
  if (!get_best_discrete_theta(s, previous_theta, interval, nb, preferred_theta, &theta_goal)) {
    *out = previous_theta;
    return 0;
  }
  if (fabs(orc_angle_diff(theta_goal, previous_theta)) < d_theta_max) { *out = theta_goal; return 1; }
  double ad = orc_angle_diff(theta_goal, previous_theta);
  double sign = ad / fabs(ad);
  *out = previous_theta + sign * d_theta_max;
  return 1;
}

/* utl:115-127 tend_to_preferred_theta */
static double tend_to_preferred_theta(double previous_theta, double d_theta_max, double goal_theta) {
  if (fabs(orc_angle_diff(goal_theta, previous_theta)) < d_theta_max) return goal_theta;
  double ad = orc_angle_diff(goal_theta, previous_theta);
  double sign = ad / fabs(ad);
  return previous_theta + sign * d_theta_max;
}

static double joints_angle_dist(const double a[7], const double b[7]) {
  double s = 0;
  for (int i = 0; i < 7; i++) { double d = orc_angle_diff(a[i], b[i]); s += d * d; }
  return sqrt(s);
}

/* utl:267-331 get_best_theta_to_current_joints (get_joints mutates the solver, as in
 * the reference: the state leak is part of the result when the projection fires) */
static double get_best_theta_to_current_joints(orc_solver *s, const double current_joints[7], double preferred_theta) {
  static const double zero7[7] = {0, 0, 0, 0, 0, 0, 0};
  double low = -ORC_PI, high = ORC_PI;
  if (s->cfg.side < 0) { low = 0; high = 2 * ORC_PI; }
  const double tolerance = 0.01;
  double j[7], j2[7];
  solver_get_joints(s, preferred_theta, zero7, j, 0);
  if (joints_angle_dist(j, current_joints) < tolerance) return preferred_theta;
  while ((high - low) > tolerance) {
    double mid1 = low + (high - low) / 3;
    double mid2 = high - (high - low) / 3;
    solver_get_joints(s, mid1, zero7, j, 0);
    solver_get_joints(s, mid2, zero7, j2, 0);
    double f1 = joints_angle_dist(j, current_joints);
    double f2 = joints_angle_dist(j2, current_joints);
    if (f1 < f2) high = mid2; else low = mid1;
  }
  double best = (low + high) / 2;
  solver_get_joints(s, best, zero7, j, 0); /* reference calls it once more (state leak) */
  return best;
}

/* ctl:464-497 safety_checks = limit_orbita3d_joints_wrist -> allow_multiturn -> multiturn_safety_check */
static int safety_checks(double joints[7], const double previous_sol[7], double orbita_max) {
  double w[3] = {joints[4], joints[5], joints[6]}, o[3];
  orc_limit_orbita3d_joints(w, orbita_max, o); /* utl:522-532 */
  joints[4] = o[0]; joints[5] = o[1]; joints[6] = o[2];
  for (int i = 0; i < 7; i++) { /* utl:493-505 allow_multiturn */
    double diff = orc_angle_diff(joints[i], previous_sol[i]);
    joints[i] = previous_sol[i] + diff;
  }
  int bits = 0; /* utl:535-568 multiturn_safety_check */
  const double lim = 6 * ORC_PI;
  if (joints[0] > lim) { joints[0] = lim; bits |= ORC_EMG_SHOULDER_PITCH; }
  if (joints[0] < -lim) { joints[0] = -lim; bits |= ORC_EMG_SHOULDER_PITCH; }
  if (joints[2] > lim) { joints[2] = lim; bits |= ORC_EMG_ELBOW_YAW; }
  if (joints[2] < -lim) { joints[2] = -lim; bits |= ORC_EMG_ELBOW_YAW; }
  if (joints[6] > lim) { joints[6] = lim; bits |= ORC_EMG_WRIST_YAW; }
  if (joints[6] < -lim) { joints[6] = -lim; bits |= ORC_EMG_WRIST_YAW; }
  return bits;
}

/* ctl:212-217: M -> (position, euler) with the identity snap (np.allclose(M[:3,:3], eye)) */
static int pose_from_matrix(const double *M, double pos[3], double eul[3]) {
  pos[0] = M[3]; pos[1] = M[7]; pos[2] = M[11];
  int close = 1;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double e = (i == j) ? 1.0 : 0.0;
      if (!(fabs(M[4 * i + j] - e) <= 1e-8 + 1e-5 * fabs(e))) close = 0;
    }
  if (close) { eul[0] = eul[1] = eul[2] = 0.0; return 0; }
  double m9[9] = {M[0], M[1], M[2], M[4], M[5], M[6], M[8], M[9], M[10]};
  int st;
  orc_euler_xyz_from_matrix(m9, eul, &st);
  return st;
}

/* plain conversion (no snap) used by the SymbolicIK (N,4,4) entry point */
static int pose_from_matrix_nosnap(const double *M, double pos[3], double eul[3]) {
  pos[0] = M[3]; pos[1] = M[7]; pos[2] = M[11];
  double m9[9] = {M[0], M[1], M[2], M[4], M[5], M[6], M[8], M[9], M[10]};
  int st;
  orc_euler_xyz_from_matrix(m9, eul, &st);
  return st;
}

/* ctl:225-252 interval_limit with l_arm mirroring */
void orc_interval_limit(int side, int low_elbow, double out[2]) {
  double il[2];
  if (!low_elbow) { il[0] = 3 * ORC_PI / 4; il[1] = -2 * ORC_PI / 6; }
  else { il[0] = -4 * ORC_PI / 5; il[1] = 0; }
  if (side < 0) {
    double a = -ORC_PI - il[1], b = -ORC_PI - il[0];
    il[0] = a; il[1] = b;
    if (il[0] < -ORC_PI) il[0] = orc_pymod(il[0], 2 * ORC_PI);
    if (il[1] < -ORC_PI) il[1] = orc_pymod(il[1], 2 * ORC_PI);
    if (il[0] > ORC_PI) il[0] = orc_pymod(il[0], -2 * ORC_PI);
    if (il[1] > ORC_PI) il[1] = orc_pymod(il[1], -2 * ORC_PI);
  }
  out[0] = il[0]; out[1] = il[1];
}

/* ------------------------------------------------------------------------- */
/* public entry points                                                        */
/* ------------------------------------------------------------------------- */

static void fill_nan(double *p, int n) { for (int i = 0; i < n; i++) p[i] = NAN; }

static int load_pose(int kind, const double *pose, double pos[3], double eul[3]) {
  if (kind == ORC_POSE_EULER6) {
    memcpy(pos, pose, 3 * sizeof(double));
    memcpy(eul, pose + 3, 3 * sizeof(double));
    return 0;
  }
  return pose_from_matrix_nosnap(pose, pos, eul);
}

int orc_symik_solve(const orc_arm_config *cfg, int pose_kind, const double *pose, const double *theta,
                    const double prev_joints[7], uint8_t *reachable, uint8_t *state, double interval[2],
                    double joints[7], double elbow[3]) {
  static const double zero7[7] = {0, 0, 0, 0, 0, 0, 0};
  orc_solver s;
  solver_init(&s, cfg);
  double pos[3], eul[3];
  fill_nan(joints, 7); fill_nan(elbow, 3); fill_nan(interval, 2);
  if (load_pose(pose_kind, pose, pos, eul)) { *reachable = 0; *state = ORC_STATE_INVALID_ROTATION; return 0; }
  int st;
  int ok = solver_is_reachable(&s, pos, eul, interval, &st);
  *reachable = (uint8_t)ok;
  *state = (uint8_t)st;
  if (ok) {
    double th = theta ? *theta : interval[0];
    solver_get_joints(&s, th, prev_joints ? prev_joints : zero7, joints, elbow);
  }
  return 0;
}

void orc_symik_batch(const orc_arm_config *cfg, int pose_kind, const double *poses, const double *theta, int64_t n,
                     uint8_t *reachable, uint8_t *state, double *interval, double *joints, double *elbow) {
  int stride = pose_kind == ORC_POSE_EULER6 ? 6 : 16;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; i++)
    orc_symik_solve(cfg, pose_kind, poses + i * stride, theta ? theta + i : 0, 0, reachable + i, state + i,
                    interval + 2 * i, joints + 7 * i, elbow + 3 * i);
}

/* sik:697-718: does get_joints(theta) take the make_elbow_projection branch on the solved pose?  (The reference then
 * returns the elbow as a 3-vector instead of get_elbow_position's homogeneous [x, y, z, 1], sik:714 / :863.) */
static int elbow_projection_fires(const orc_solver *s, double theta) {
  double e[3];
  get_elbow_position(s, theta, e);
  return e[2] > (e[0] - s->elbow_singularity_position[0]) * s->cfg.singularity_limit_coeff +
                    s->elbow_singularity_position[2] - s->cfg.singularity_offset;
}

void orc_symik_no_limits_batch(const orc_arm_config *cfg, int pose_kind, const double *poses, const double *theta,
                               const double *prev_joints, int64_t n, double *joints, double *elbow, uint8_t *projected) {
  static const double zero7[7] = {0, 0, 0, 0, 0, 0, 0};
  int stride = pose_kind == ORC_POSE_EULER6 ? 6 : 16;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; i++) {
    orc_solver s;
    solver_init(&s, cfg);
    double pos[3], eul[3];
    if (projected) projected[i] = 0;
    if (load_pose(pose_kind, poses + i * stride, pos, eul) || !solver_is_reachable_no_limits(&s, pos, eul)) {
      fill_nan(joints + 7 * i, 7); fill_nan(elbow + 3 * i, 3);
      continue;
    }
    if (projected) projected[i] = (uint8_t)elbow_projection_fires(&s, theta[i]);
    solver_get_joints(&s, theta[i], prev_joints ? prev_joints + 7 * i : zero7, joints + 7 * i, elbow + 3 * i);
  }
}

void orc_elbow_positions_batch(const orc_arm_config *cfg, int pose_kind, const double *poses, const double *thetas,
                               int K, int64_t n, int no_limits, double *elbows, uint8_t *projected) {
  int stride = pose_kind == ORC_POSE_EULER6 ? 6 : 16;
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; i++) {
    orc_solver s;
    solver_init(&s, cfg);
    double pos[3], eul[3], itv[2];
    int st;
    int bad = load_pose(pose_kind, poses + i * stride, pos, eul);
    /* the intersection circle is stored as soon as it exists (sik:197), also when the wrist limit then rejects the pose */
    if (!bad) bad = no_limits ? !solver_is_reachable_no_limits(&s, pos, eul)
                              : !(solver_is_reachable(&s, pos, eul, itv, &st) || st == ORC_STATE_LIMITED_BY_WRIST);
    if (bad) {
      fill_nan(elbows + (size_t)i * K * 3, K * 3);
      if (projected) memset(projected + (size_t)i * K, 0, (size_t)K);
      continue;
    }
    for (int k = 0; k < K; k++) {
      get_elbow_position(&s, thetas[(size_t)i * K + k], elbows + ((size_t)i * K + k) * 3);
      if (projected) projected[(size_t)i * K + k] = (uint8_t)elbow_projection_fires(&s, thetas[(size_t)i * K + k]);
    }
  }
}

/* One scalar call sequence of the reference's SymbolicIK on goal_pose6 = (x, y, z, roll, pitch, yaw):
 *   is_reachable (no_limits = 0, sik:121-282) or is_reachable_no_limits (1, sik:85-119), then -- when the call
 *   succeeded -- get_elbow_position(theta) (sik:684-695) and get_joints(theta, previous_joints) (sik:697-863) with
 *   theta = *theta_opt or theta_interval[0].  The record also holds the solver attributes the two calls leave behind. */
void orc_symik_scalar(const orc_arm_config *cfg, const double *goal_pose6, int no_limits, const double *theta_opt,
                      const double *prev_joints, orc_scalar_result *out) {
  static const double zero7[7] = {0, 0, 0, 0, 0, 0, 0};
  orc_solver s;
  solver_init(&s, cfg);
  memset(out, 0, sizeof *out);
  fill_nan(out->interval, 2); fill_nan(out->joints, 7); fill_nan(out->elbow, 3); fill_nan(out->elbow_on_circle, 3);
  fill_nan(out->goal_position_solved, 3); fill_nan(out->wrist_position_solved, 3);
  fill_nan(out->goal_position, 3); fill_nan(out->wrist_position, 3);
  int st = ORC_STATE_REACHABLE, ok;
  if (no_limits) {
    ok = solver_is_reachable_no_limits(&s, goal_pose6, goal_pose6 + 3);
    if (ok) { out->interval[0] = -ORC_PI; out->interval[1] = ORC_PI; } else st = ORC_STATE_SHOULD_NOT_HAPPEN;
  } else {
    ok = solver_is_reachable(&s, goal_pose6, goal_pose6 + 3, out->interval, &st);
  }
  out->reachable = ok;
  out->state = st;
  /* attributes exist once the pre-checks passed (sik:143-144); the circle once it was found (sik:197) */
  int attrs = no_limits || st == ORC_STATE_REACHABLE || st == ORC_STATE_LIMITED_BY_WRIST || st == ORC_STATE_WRIST_OUT_OF_RANGE ||
              st == ORC_STATE_SHOULD_NOT_HAPPEN;
  if (attrs) {
    memcpy(out->goal_position_solved, s.goal_position, 3 * sizeof(double));
    memcpy(out->wrist_position_solved, s.wrist_position, 3 * sizeof(double));
  }
  int circle = ok || st == ORC_STATE_LIMITED_BY_WRIST;
  if (circle && (theta_opt || ok)) {
    double th = theta_opt ? *theta_opt : out->interval[0];
    get_elbow_position(&s, th, out->elbow_on_circle);
    if (ok) {
      out->projected = elbow_projection_fires(&s, th);
      solver_get_joints(&s, th, prev_joints ? prev_joints : zero7, out->joints, out->elbow);
      memcpy(out->goal_position, s.goal_position, 3 * sizeof(double));
      memcpy(out->wrist_position, s.wrist_position, 3 * sizeof(double));
    }
  }
}

/* ctl:409-462 symbolic_inverse_kinematics_discrete (+ front end ctl:212-217) */
static void ctl_discrete_one(const orc_arm_config *cfg, const orc_ctl_params *par, const double *M,
                             const double prev_joints[7], const double current_joints[7], double joints[7],
                             uint8_t *reachable, uint8_t *state, uint8_t *emergency) {
  orc_solver s;
  solver_init(&s, cfg);
  double pos[3], eul[3], itv[2];
  if (pose_from_matrix(M, pos, eul)) {
    fill_nan(joints, 7);
    *reachable = 0; *state = ORC_STATE_INVALID_ROTATION; *emergency = 0;
    return;
  }
  int st;
  int ok = solver_is_reachable(&s, pos, eul, itv, &st);
  double theta = 0;
  if (ok) {
    ok = get_best_discrete_theta(&s, 0.0, itv, par->nb_search_points, par->preferred_theta, &theta);
    if (!ok) st = ORC_STATE_LIMITED_BY_SHOULDER;
  }
  if (ok) {
    orc_limit_theta_to_interval(theta, 0.0, par->interval_limit, &theta);
    solver_get_joints(&s, theta, prev_joints, joints, 0);
  } else {
    memcpy(joints, current_joints, 7 * sizeof(double));
  }
  int bits = safety_checks(joints, prev_joints, par->orbita3d_max_angle);
  *reachable = (uint8_t)ok;
  *state = (uint8_t)st;
  *emergency = (uint8_t)bits;
}

void orc_ctl_discrete_batch(const orc_arm_config *cfg, const orc_ctl_params *par, const double *M, int64_t n,
                            const double prev_joints[7], const double current_joints[7], double *joints,
                            uint8_t *reachable, uint8_t *state, uint8_t *emergency) {
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < n; i++)
    ctl_discrete_one(cfg, par, M + 16 * i, prev_joints, current_joints, joints + 7 * i, reachable + i, state + i,
                     emergency + i);
}

/* ctl:276-407 symbolic_inverse_kinematics_continuous, one waypoint */
static void ctl_continuous_step(const orc_arm_config *cfg, const orc_ctl_params *par, const double *M,
                                const double current_joints[7], const double *current_pose, orc_ctl_state *cs,
                                double joints[7], uint8_t *reachable, uint8_t *state) {
  /* ctl:205-210 emergency latch */
  if (cs->emergency_stop) {
    memcpy(joints, cs->previous_sol, 7 * sizeof(double));
    *reachable = 0; *state = ORC_STATE_EMERGENCY;
    return;
  }
  orc_solver s;
  solver_init(&s, cfg);
  double pos[3], eul[3];
  if (pose_from_matrix(M, pos, eul)) {
    fill_nan(joints, 7);
    *reachable = 0; *state = ORC_STATE_INVALID_ROTATION;
    return;
  }
  int st_out = ORC_STATE_EMPTY;
  if (!cs->has_previous_sol) { /* ctl:306-325 */
    memcpy(cs->previous_sol, current_joints, 7 * sizeof(double));
    cs->has_previous_sol = 1;
    cs->init = 1;
    double cpos[3], ceul[3];
    pose_from_matrix(current_pose, cpos, ceul);
    solver_is_reachable_no_limits(&s, cpos, ceul);
    cs->previous_theta = get_best_theta_to_current_joints(&s, current_joints, par->preferred_theta);
  }
  double itv[2], theta;
  int rs;
  int ok = solver_is_reachable(&s, pos, eul, itv, &rs);
  if (ok) { /* ctl:338-366 */
    ok = get_best_continuous_theta2(&s, cs->previous_theta, itv, par->nb_search_points_continuous, par->d_theta_max,
                                    par->preferred_theta_ctor, &theta);
    if (!ok) st_out = ORC_STATE_LIMITED_BY_SHOULDER;
    orc_limit_theta_to_interval(theta, cs->previous_theta, par->interval_limit, &theta);
    cs->previous_theta = theta;
    solver_get_joints(&s, theta, cs->previous_sol, joints, 0);
  } else { /* ctl:368-388 */
    solver_is_reachable_no_limits(&s, pos, eul);
    theta = tend_to_preferred_theta(cs->previous_theta, par->d_theta_max, par->preferred_theta);
    orc_limit_theta_to_interval(theta, cs->previous_theta, par->interval_limit, &theta);
    cs->previous_theta = theta;
    solver_get_joints(&s, theta, cs->previous_sol, joints, 0);
    st_out = rs;
  }
  int bits = safety_checks(joints, cs->previous_sol, par->orbita3d_max_angle); /* ctl:393 */
  if (bits) { cs->emergency_stop = 1; cs->emergency_bits |= bits; }
  if (!cs->init) { /* ctl:395-400 + utl:571-589 continuity_check */
    static const double max_step[7] = {0.5, 0.5, 0.5, 0.5, 1.0, 1.0, 1.0};
    int disc = 0;
    for (int i = 0; i < 7; i++)
      if (fabs(orc_angle_diff(joints[i], cs->previous_sol[i])) > max_step[i]) disc = 1;
    if (disc) {
      memcpy(joints, cs->previous_sol, 7 * sizeof(double));
      cs->emergency_stop = 1;
      cs->emergency_bits |= ORC_EMG_DISCONTINUITY;
    }
  }
  cs->init = 0;
  if (!cs->emergency_stop) memcpy(cs->previous_sol, joints, 7 * sizeof(double));
  *reachable = (uint8_t)ok;
  *state = (uint8_t)st_out;
}

void orc_ctl_continuous_batch(const orc_arm_config *cfg, const orc_ctl_params *par, const double *M, int64_t T,
                              int32_t W, const double *current_joints, const double *current_pose, orc_ctl_state *st,
                              double *joints, uint8_t *reachable, uint8_t *state) {
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t t = 0; t < T; t++)
    for (int32_t w = 0; w < W; w++) {
      size_t k = (size_t)t * W + w;
      ctl_continuous_step(cfg, par, M + 16 * k, current_joints + 7 * t, current_pose + 16 * t, st + t, joints + 7 * k,
                          reachable + k, state + k);
    }
}

void orc_reach_map(const orc_arm_config *cfg, const double origin[3], const double step[3], const int32_t dims[3],
                   const double *orientations_euler, int32_t ori_begin, int32_t ori_end, uint32_t *counts) {
  int64_t nv = (int64_t)dims[0] * dims[1] * dims[2];
#pragma omp parallel for schedule(dynamic, 64)
  for (int64_t v = 0; v < nv; v++) {
    int iz = (int)(v % dims[2]);
    int iy = (int)((v / dims[2]) % dims[1]);
    int ix = (int)(v / ((int64_t)dims[2] * dims[1]));
    double pos[3] = {origin[0] + ix * step[0], origin[1] + iy * step[1], origin[2] + iz * step[2]};
    orc_solver s;
    solver_init(&s, cfg);
    uint32_t c = 0;
    for (int o = ori_begin; o < ori_end; o++) {
      double itv[2];
      int st;
      c += (uint32_t)solver_is_reachable(&s, pos, orientations_euler + 3 * o, itv, &st);
    }
    counts[v] = c;
  }
}

int orc_max_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

/* torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arms of bench.py ask for the host's threads explicitly */
void orc_set_threads(int n) {
#ifdef _OPENMP
  if (n > 0) omp_set_num_threads(n);
#else
  (void)n;
#endif
}
