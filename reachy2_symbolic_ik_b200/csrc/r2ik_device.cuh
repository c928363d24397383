// r2ik_device.cuh -- per-pose solver math of the Reachy2 symbolic IK, FP64, sm_100a.
//
// One thread owns one pose (or one trajectory): everything below is straight-line scalar
// FP64 code on 3-vectors held in registers.  The reference's 4x4 "frame peeling" is
// restructured into progressive 2-D rotations of the few points that are still needed, its
// np.linalg.lstsq into the closed form of the consistent 3x2 system, and its asin/atan2/
// from_euler construction of the elbow-circle normal into n = P/d (SURVEY.md A.7); all
// thresholds, branch orders and Python/NumPy semantics (%, isclose, linspace, strict-<
// arg-min) are kept exactly.  Citations: "sik" = src/reachy2_symbolic_ik/symbolic_ik.py,
// "utl" = .../utils.py, "ctl" = .../control_ik.py, "rxp" = scipy _rotation_xp.py (1.18.1).
//
// The functions are __host__ __device__ so that tests/hostsim can run this exact source on
// the CPU for debugging; libr2ik.so exports no host implementation of any entry point.
#pragma once

#include <math.h>
#include <stdint.h>

#include "../../include/r2ik.h"
#include "r2ik_math.cuh"

namespace r2ik {

constexpr double kPi = 3.14159265358979323846;
constexpr double kTwoPi = 2.0 * kPi;
constexpr double kHalfPi = kPi / 2;

// Per-arm constants derived once on the host (r2ik_create) and passed to every kernel as a
// __grid_constant__ parameter (constant bank, broadcast to all threads).
struct ArmConst {
  double s[3];                // shoulder position
  double L1, L2, L12;         // upper arm, forearm, L1 + L2
  double L1sq, L2sq;
  double wo[3];               // wrist in the goal frame: (-tip.x, tip.y, tip.z)     sik:422
  double to[3];               // tip point in the goal frame: (-tip.x, tip.y, 0)     sik:810
  double tip_z;               //                                                     sik:837
  double max_arm_length;      // L1 + L2 + |tip|                                     sik:65
  double d_min;               // shoulder_wrist_min_distance                         sik:73-77
  double proj_margin;         // 1e-8
  double backward_limit;      // 0.02
  double nvm;                 // normal_vector_margin 1e-7
  double rL, rLsq, hL;        // wrist-limit circle radius, its square, centre offset sik:413-414
  double Mst[9];              // M_shoulder_torso = (R(offset) * Ry(pi/2))^T, row-major sik:728-736
  double Pst[3];              // -Mst * s                                            sik:737
  double es[3];               // elbow_singularity_position                          utl:26-43
  double sing_coeff, sing_offset;
  double plP[3], plV[3];      // singularity-limit plane: point, unit normal         sik:653-669
  double plC[3], plRho;       // shoulder projected on the plane, circle radius      sik:671-672
  double elbow_limit;         // radians(elbow_limit)                                sik:853
  double side;                // +1 r_arm, -1 l_arm
};

// ---------------------------------------------------------------------------------------
// Python / NumPy scalar semantics
// ---------------------------------------------------------------------------------------

// Fast / literal duality.  The hot kernels run the solver with LIT = false: every elementary
// function is straight-line code that is only valid for "ordinary" magnitudes, and each use
// ORs its validity test into a `degenerate` flag instead of branching.  A pose that raised the
// flag (exact zeros, under/overflowing magnitudes -- never on physical data) is solved again
// by the out-of-line LIT = true instantiation, which calls the math library exactly where the
// reference calls numpy / scipy.  The hot instruction stream thus contains no library slow
// path and no branch around one.

// (c, s) = (cos a, sin a) for a = atan2(y, x), without evaluating the angle: the reference builds
// its elementary frame rotations as from_euler(atan2(...)) (sik:758-829); x/h, y/h equal
// cos/sin of that angle to ~1 ulp.
template <bool LIT>
R2IK_HD void cs_of_atan2(double y, double x, double &c, double &s, bool &degenerate) {
  if (LIT) {
    sincos(atan2(y, x), &s, &c);
  } else {
    double h2 = x * x + y * y;
    // 1e-280 < h2 < 1e280, tested on the exponent field (integer pipe)
    degenerate = degenerate || !((unsigned)(hi_word(h2) - 0x05e00000) < (unsigned)(0x7a000000 - 0x05e00000));
    double ih = rsqrt_pos(h2);
    c = x * ih; s = y * ih;
  }
}

// (c, s) as above AND the angle a = atan2(y, x) itself: the fast route reads the angle off the unit
// vector (angle_of_unit, no division).
template <bool LIT>
R2IK_HD double cs_and_angle(double y, double x, double &c, double &s, bool &degenerate) {
  cs_of_atan2<LIT>(y, x, c, s, degenerate);
  if (LIT) return atan2(y, x);
  return angle_of_unit(c, s);
}

// atan2 as a leaf value.
template <bool LIT>
R2IK_HD double atan2_leaf(double y, double x, bool &degenerate) {
  if (LIT) return atan2(y, x);
  degenerate = degenerate || !atan2_core_ok(y, x);
  return atan2_core(y, x);
}

// sin / cos of an arbitrary angle: the straight-line kernel for moderate arguments, the library (out of
// line on the device) beyond.
#if defined(__CUDACC__)
__device__ __noinline__ double2 sincos_library_dev(double a) {
  double s, c;
  sincos(a, &s, &c);
  return make_double2(s, c);
}
#endif
R2IK_HD void sincos_any(double a, double &s, double &c) {
  if (sincos_small_ok(a)) { sincos_small(a, s, c); return; }
#if defined(__CUDA_ARCH__)
  double2 r = sincos_library_dev(a);
  s = r.x; c = r.y;
#else
  sincos(a, &s, &c);
#endif
}

// Python float `%`: fmod is exact; the result takes the sign of the divisor.
R2IK_HD double pymod(double a, double m) {
  double r = fmod(a, m);
  if (r != 0.0) {
    if ((m < 0.0) != (r < 0.0)) r += m;
  } else {
    r = copysign(0.0, m);
  }
  return r;
}

// pymod(x, 2 pi) for the arguments the controller produces.  Python's float % is fmod (exact) plus at
// most one rounded `+ m`.  For 0 <= x < 8 pi the exact remainder is reached by subtracting 4 pi /
// 2 pi when x is at least that: 2 pi and 4 pi are exact multiples of the same double and every
// difference below is exactly representable (both operands are multiples of the ulp of the result
// range), so each step is error-free and the value is bit-identical to fmod's.  Negative x in
// [-2 pi, 0) is Python's `fmod(x) + m`, one rounded add and nothing more: for -x below half an ulp of
// 2 pi that sum rounds to 2 pi itself, which Python returns as it is.  Anything else takes pymod().
// For x = -0 this returns -0 where Python gives +0: pymod_2pi below adds the fix, angle_diff (whose
// argument is never -0) does without it.
R2IK_HD double pymod_2pi_not_minus_zero(double x) {
  const double two_pi = R2IK_WRAP(1), four_pi = R2IK_WRAP(2);
  if (!(x >= -two_pi && x < R2IK_WRAP(3))) return pymod(x, kTwoPi);
  double r = x >= four_pi ? x - four_pi : x;
  r = r >= two_pi ? r - two_pi : r;
  return x < 0.0 ? x + two_pi : r;
}
// A zero remainder is +0: `+ 0.0` turns -0 into +0 and leaves every other value as it is.
R2IK_HD double pymod_2pi(double x) { return pymod_2pi_not_minus_zero(x) + 0.0; }

// utl:486-490.  (a - b) + pi is never -0 (a sum is -0 only when both terms are).
R2IK_HD double angle_diff(double a, double b) { return pymod_2pi_not_minus_zero((a - b) + R2IK_WRAP(0)) - R2IK_WRAP(0); }

// np.isclose(a, b), rtol 1e-5, atol 1e-8 (asymmetric in b)
R2IK_HD bool np_isclose(double a, double b) { return fabs(a - b) <= 1e-8 + 1e-5 * fabs(b); }

// utl:468-474
R2IK_HD bool is_valid_angle(double angle, double i0, double i1) {
  if (pymod_2pi(i0) == pymod_2pi(i1)) return true;
  if (i0 < i1) return (i0 <= angle) && (angle <= i1);
  return (i0 <= angle) || (angle <= i1);
}

// utl:93-112 (previous_theta is normalised but never used by the reference)
R2IK_HD double limit_theta_to_interval(double theta, double i0, double i1) {
  theta = pymod_2pi(theta);
  if (theta > kPi) theta -= kTwoPi;
  if (is_valid_angle(theta, i0, i1)) return theta;
  double pos_diff = angle_diff(theta, i1);
  double neg_diff = angle_diff(theta, i0);
  if (fabs(pos_diff) < fabs(neg_diff)) return i1;
  return i0;
}

// a * b + c with two roundings (numpy evaluates linspace as arange * step + start, unfused)
R2IK_HD double mul_add_unfused(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(__dmul_rn(a, b), c);
#else
  return a * b + c;
#endif
}

// np.linspace(start, stop, num) with the per-array quantities hoisted out of the sample loop
struct Linspace {
  double start, stop, delta, step;
  int div;
};
R2IK_HD Linspace make_linspace(double start, double stop, int num) {
  Linspace L;
  L.start = start; L.stop = stop; L.div = num - 1; L.delta = stop - start;
  L.step = L.div > 0 ? L.delta / (double)L.div : 0.0;
  return L;
}
R2IK_HD double linspace_value(const Linspace &L, int i) {
  if (L.div <= 0) return L.start;
  if (i == L.div) return L.stop;
  if (L.step == 0.0) return mul_add_unfused((double)i / (double)L.div, L.delta, L.start);
  return mul_add_unfused((double)i, L.step, L.start);
}

// Sampling range of get_best_discrete_theta (utl:366-375): full circle uses a vertical
// symmetry [pi/2, 5pi/2]; a wrapped interval is unrolled past pi.
R2IK_HD void search_range(double i0, double i1, double &start, double &stop) {
  if (fabs(fabs(i0) + fabs(i1) - kTwoPi) < 0.00001) { start = kHalfPi; stop = kHalfPi + kTwoPi; }
  else if (i0 < i1) { start = i0; stop = i1; }
  else { start = i0; stop = i1 + kTwoPi; }
}

// ---------------------------------------------------------------------------------------
// scipy Rotation, quaternion (x, y, z, w)
// ---------------------------------------------------------------------------------------
struct Quat { double x, y, z, w; };

// rxp:1114-1127 compose_quat
R2IK_HD Quat quat_mul(const Quat &p, const Quat &q) {
  Quat o;
  o.x = p.w * q.x + q.w * p.x + (p.y * q.z - p.z * q.y);
  o.y = p.w * q.y + q.w * p.y + (p.z * q.x - p.x * q.z);
  o.z = p.w * q.z + q.w * p.z + (p.x * q.y - p.y * q.x);
  o.w = p.w * q.w - p.x * q.x - p.y * q.y - p.z * q.z;
  return o;
}

R2IK_HD Quat quat_axis(int axis, double angle) {
  double s, c;
  sincos(angle / 2.0, &s, &c);
  Quat q = {0.0, 0.0, 0.0, c};
  if (axis == 0) q.x = s; else if (axis == 1) q.y = s; else q.z = s;
  return q;
}

// rxp:192-224 from_euler: extrinsic composes q <- q_axis o q, intrinsic q <- q o q_axis
R2IK_HD Quat quat_from_euler(int a0, int a1, int a2, bool intrinsic, double e0, double e1, double e2) {
  Quat q = quat_axis(a0, e0);
  Quat q1 = quat_axis(a1, e1);
  q = intrinsic ? quat_mul(q, q1) : quat_mul(q1, q);
  Quat q2 = quat_axis(a2, e2);
  q = intrinsic ? quat_mul(q, q2) : quat_mul(q2, q);
  return q;
}

// rxp:302-333 as_matrix (row-major 3x3)
R2IK_HD void quat_to_matrix(const Quat &q, double m[9]) {
  double x2 = q.x * q.x, y2 = q.y * q.y, z2 = q.z * q.z, w2 = q.w * q.w;
  double xy = q.x * q.y, zw = q.z * q.w, xz = q.x * q.z, yw = q.y * q.w, yz = q.y * q.z, xw = q.x * q.w;
  m[0] = x2 - y2 - z2 + w2; m[1] = 2 * (xy - zw);       m[2] = 2 * (xz + yw);
  m[3] = 2 * (xy + zw);     m[4] = -x2 + y2 - z2 + w2;  m[5] = 2 * (yz - xw);
  m[6] = 2 * (xz - yw);     m[7] = 2 * (yz + xw);       m[8] = -x2 - y2 + z2 + w2;
}

// R.from_euler("xyz", e).as_matrix(), specialised: q = qz o (qy o qx)
R2IK_HD void rot_from_euler_xyz(double e0, double e1, double e2, double m[9]) {
  double sx, cx, sy, cy, sz, cz;
  sincos_any(e0 / 2.0, sx, cx);
  sincos_any(e1 / 2.0, sy, cy);
  sincos_any(e2 / 2.0, sz, cz);
  // qy o qx with p = (0,sy,0,cy), q = (sx,0,0,cx)
  Quat a = {cy * sx, cx * sy, -(sy * sx), cy * cx};
  // qz o a with p = (0,0,sz,cz)
  Quat q;
  q.x = cz * a.x - sz * a.y;
  q.y = cz * a.y + sz * a.x;
  q.z = cz * a.z + a.w * sz;
  q.w = cz * a.w - sz * a.z;
  quat_to_matrix(q, m);
}

R2IK_HD double det3(const double m[9]) {
  return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
}

// Orthogonal polar factor of a nonsingular 3x3 (what scipy's SVD projection U @ Vt computes,
// rxp:78-95), by the Newton iteration X <- (X + X^-T) / 2.  The iteration converges quadratically: once
// two iterates agree to 1e-8 the next one is the fixed point to rounding, so one more step is taken and
// the loop ends (waiting for the step itself to fall below one ulp, as an earlier version did, never
// happens when the last bits keep flipping -- 60 iterations for every nearly-orthonormal input).
// The plain iteration only halves a scale error per step (a block scaled by 10^k needs ~3.3 |k| steps, far more than
// the 60 allowed), so a block whose largest entry lies outside [2^-4, 2^4] is first brought to unit size by an exact
// power-of-two scaling -- the polar factor does not depend on the scale.  Ordinary blocks are iterated as they are.
R2IK_HD void polar_orthogonalize(double m[9]) {
  double mx = 0.0;
  for (int k = 0; k < 9; ++k) mx = fmax(mx, fabs(m[k]));
  if (mx < 0.0625 || (mx > 16.0 && mx < INFINITY)) {
    const int e = ilogb(mx);
    for (int k = 0; k < 9; ++k) m[k] = ldexp(m[k], -e);
  }
  bool last = false;
  for (int it = 0; it < 60; ++it) {
    double id = 1.0 / det3(m);
    double c[9];
    c[0] = (m[4] * m[8] - m[5] * m[7]) * id; c[1] = (m[5] * m[6] - m[3] * m[8]) * id; c[2] = (m[3] * m[7] - m[4] * m[6]) * id;
    c[3] = (m[2] * m[7] - m[1] * m[8]) * id; c[4] = (m[0] * m[8] - m[2] * m[6]) * id; c[5] = (m[1] * m[6] - m[0] * m[7]) * id;
    c[6] = (m[1] * m[5] - m[2] * m[4]) * id; c[7] = (m[2] * m[3] - m[0] * m[5]) * id; c[8] = (m[0] * m[4] - m[1] * m[3]) * id;
    double delta = 0.0;
    for (int k = 0; k < 9; ++k) {
      double nx = 0.5 * (m[k] + c[k]);
      delta = fmax(delta, fabs(nx - m[k]));
      m[k] = nx;
    }
    if (last) break;
    if (delta < 1e-8) last = true;
  }
}

// rxp:51-156 from_matrix.  Returns false when det <= 0 (scipy raises ValueError).
R2IK_HD bool quat_from_matrix(const double min[9], Quat &q) {
  double m[9];
  for (int k = 0; k < 9; ++k) m[k] = min[k];
  if (!(det3(m) > 0.0)) return false;
  bool orthogonal = true;
  for (int i = 0; i < 3; ++i)
    for (int j = i; j < 3; ++j) {
      double g = m[3 * i] * m[3 * j] + m[3 * i + 1] * m[3 * j + 1] + m[3 * i + 2] * m[3 * j + 2];
      double e = (i == j) ? 1.0 : 0.0;
      if (!(fabs(g - e) <= 1e-12 + 1e-5 * e)) orthogonal = false;
    }
  if (!orthogonal) polar_orthogonalize(m);
  double tr = m[0] + m[4] + m[8];
  // argmax over (m00, m11, m22, trace): the first maximum wins
  int choice = 0;
  double best = m[0];
  if (m[4] > best) { best = m[4]; choice = 1; }
  if (m[8] > best) { best = m[8]; choice = 2; }
  if (tr > best) { choice = 3; }
  if (choice == 0) {
    q.x = 1 - tr + 2 * m[0]; q.y = m[3] + m[1]; q.z = m[6] + m[2]; q.w = m[7] - m[5];
  } else if (choice == 1) {
    q.x = m[3] + m[1]; q.y = 1 - tr + 2 * m[4]; q.z = m[7] + m[5]; q.w = m[2] - m[6];
  } else if (choice == 2) {
    q.x = m[6] + m[2]; q.y = m[7] + m[5]; q.z = 1 - tr + 2 * m[8]; q.w = m[3] - m[1];
  } else {
    q.x = m[7] - m[5]; q.y = m[2] - m[6]; q.z = m[3] - m[1]; q.w = 1 + tr;
  }
  double n = sqrt(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
  q.x /= n; q.y /= n; q.z /= n; q.w /= n;
  return true;
}

// rxp:1052-1111 _get_angles
R2IK_HD void get_angles(bool extrinsic, bool symmetric, double sign, double a, double b, double c, double d, double out[3]) {
  const double eps = 1e-7;
  double half_sum = atan2(b, a);
  double half_diff = atan2(d, c);
  double ang0 = 0.0, ang2 = 0.0;
  double ang1 = 2 * atan2(hypot(c, d), hypot(a, b));
  bool case1 = fabs(ang1) <= eps;
  bool case2 = fabs(ang1 - kPi) <= eps;
  bool case0 = !(case1 || case2);
  ang0 = case1 ? 2 * half_sum : 2 * half_diff * (extrinsic ? -1.0 : 1.0);
  double first, third;
  if (extrinsic) {  // angle_first = 0, angle_third = 2
    first = case0 ? half_sum - half_diff : ang0;
    third = case0 ? half_sum + half_diff : ang2;
  } else {          // angle_first = 2, angle_third = 0
    first = case0 ? half_sum - half_diff : ang2;
    third = case0 ? half_sum + half_diff : ang0;
  }
  if (!symmetric) {
    third = third * sign;
    ang1 = ang1 - kHalfPi;
  }
  if (extrinsic) { ang0 = first; ang2 = third; } else { ang2 = first; ang0 = third; }
  out[0] = pymod_2pi(ang0 + kPi) - kPi;
  out[1] = pymod_2pi(ang1 + kPi) - kPi;
  out[2] = pymod_2pi(ang2 + kPi) - kPi;
}

// rxp:365-404 as_euler for the three sequences the reference uses
R2IK_HD void quat_as_euler_xyz_extrinsic(const Quat &q, double out[3]) {  // "xyz": i,j,k = 0,1,2; sign = +1
  get_angles(true, false, 1.0, q.w - q.y, q.x + q.z, q.y + q.w, q.z - q.x, out);
}
R2IK_HD void quat_as_euler_XYZ_intrinsic(const Quat &q, double out[3]) {  // "XYZ": i,j,k = 2,1,0; sign = -1
  get_angles(false, false, -1.0, q.w - q.y, q.z - q.x, q.y + q.w, -q.x - q.z, out);
}
R2IK_HD void quat_as_euler_ZYZ_intrinsic(const Quat &q, double out[3]) {  // "ZYZ": i,j,k = 2,1,0(sym); sign = -1
  get_angles(false, true, -1.0, q.w, q.z, q.y, q.x * -1.0, out);
}

// utl:84-90 get_euler_from_homogeneous_matrix on the rotation block of a row-major 4x4
R2IK_HD bool euler_xyz_from_mat4(const double *M, double e[3]) {
  double m9[9] = {M[0], M[1], M[2], M[4], M[5], M[6], M[8], M[9], M[10]};
  Quat q;
  if (!quat_from_matrix(m9, q)) return false;
  quat_as_euler_xyz_extrinsic(q, e);
  return true;
}

// ctl:212 np.allclose(M[:3,:3], np.eye(3))
R2IK_HD bool rotation_is_identity(const double *M) {
  bool close = true;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double e = (i == j) ? 1.0 : 0.0;
      if (!(fabs(M[4 * i + j] - e) <= 1e-8 + 1e-5 * e)) close = false;
    }
  return close;
}

// utl:508-519 limit_orbita3d_joints on joints[4:7]
R2IK_HD void limit_orbita3d_wrist(double j[7], double max_angle) {
  // Algebraic route.  For R = Rx(a) Ry(b) Rz(c) = Rz(alpha) Ry(beta) Rz(gamma):
  //   cos(beta) = R22 = cos a cos b,   (cos alpha, sin alpha) sin(beta) = (R02, R12) = (sin b, -sin a cos b),
  //   (-cos gamma, sin gamma) sin(beta) = (R20, R21).
  // Inside the cone (beta <= max) with (a, b, c) in as_euler's canonical ranges the four conversions
  // are the identity (to rounding).  Outside, the clamped rotation Rz(alpha) Ry(max) Rz(gamma) is built
  // from those unit vectors and read back as XYZ angles (a' = atan2(-R12, R22), b' = asin(R02),
  // c' = atan2(-R01, R00)): three small sincos, one rsqrt, three atan2, all straight-line.  Inputs in
  // a gimbal band of either sequence (where scipy zeroes an angle) or outside the canonical ranges take
  // the literal conversions below.
  {
    const double a = j[4], b = j[5], c = j[6];
    if (fabs(a) <= kPi && fabs(c) <= kPi && fabs(b) < kHalfPi - 1e-3 && sincos_small_ok(max_angle)) {
      // Exactly zero roll and pitch (the wrist of ControlIK's default previous solution, which every unreachable
      // pose returns): R = Rz(c), beta = 0 sits in scipy's ZYZ gimbal band where the conversions give
      // alpha = c, gamma = 0 and back (0, 0, c) -- the input, to one rounding of c / 2.
      if (a == 0.0 && b == 0.0) return;
      double sa, ca, sb, cb, sm, cm;
      sincos_small(a, sa, ca);
      sincos_small(b, sb, cb);
      sincos_small(max_angle, sm, cm);
      const double cbeta = ca * cb;
      if (cbeta < 1.0 - 1e-12) {          // beta > ~1.4e-6: outside scipy's ZYZ gimbal band (1e-7)
        if (cbeta >= cm) return;          // inside the cone
        double sc, cc;
        sincos_small(c, sc, cc);
        const double r02 = sb, r12 = -sa * cb;
        const double r20 = sa * sc - ca * sb * cc, r21 = sa * cc + ca * sb * sc;
        const double isb = rsqrt_pos(r02 * r02 + r12 * r12);
        const double cal = r02 * isb, sal = r12 * isb, cga = -r20 * isb, sga = r21 * isb;
        const double q02 = cal * sm, q12 = sal * sm, q22 = cm;
        const double q00 = cal * cm * cga - sal * sga, q01 = -(cal * cm) * sga - sal * cga;
        j[4] = atan2_core(-q12, q22);
        j[5] = atan2_core(q02, sqrt_nonneg(q12 * q12 + q22 * q22));
        j[6] = atan2_core(-q01, q00);
        return;
      }
    }
  }
  Quat q = quat_from_euler(0, 1, 2, true, j[4], j[5], j[6]);   // from_euler("XYZ")
  double zyz[3];
  quat_as_euler_ZYZ_intrinsic(q, zyz);
  zyz[1] = fmin(max_angle, fmax(-max_angle, zyz[1]));
  Quat q2 = quat_from_euler(2, 1, 2, true, zyz[0], zyz[1], zyz[2]);  // from_euler("ZYZ")
  double rpy[3];
  quat_as_euler_XYZ_intrinsic(q2, rpy);
  j[4] = rpy[0]; j[5] = rpy[1]; j[6] = rpy[2];
}

// ---------------------------------------------------------------------------------------
// SymbolicIK solve state (the reference's self.goal_pose / wrist_position / intersection_circle)
// ---------------------------------------------------------------------------------------
struct Solve {
  double p[3];   // goal position (after the reference's shifts / projections)
  double R[9];   // goal rotation, R.from_euler("xyz", goal_orientation).as_matrix()
  double w[3];   // wrist position
  double c[3];   // elbow circle centre
  double r;      // elbow circle radius
  double a1[3];  // columns 1, 2 of rotation_matrix_from_vector(circle normal):
  double a2[3];  //   elbow(theta) = c + a1 * r cos(theta) + a2 * r sin(theta)       sik:684-695
};

// utl:59-81 rotation_matrix_from_vector, columns of R for an (un-normalised) vector v.
R2IK_HD void rmfv_columns(double vx, double vy, double vz, bool normalise, double c0[3], double a1[3], double a2[3]) {
  double ux = vx, uy = vy, uz = vz;
  if (normalise) {
    double in = rsqrt_pos(vx * vx + vy * vy + vz * vz);
    ux = vx * in; uy = vy * in; uz = vz * in;
  }
  if (np_isclose(1.0, ux) && np_isclose(0.0, uy) && np_isclose(0.0, uz)) {
    c0[0] = 1; c0[1] = 0; c0[2] = 0;
    a1[0] = 0; a1[1] = 1; a1[2] = 0;
    a2[0] = 0; a2[1] = 0; a2[2] = 1;
    return;
  }
  if (np_isclose(1.0, -ux) && np_isclose(0.0, -uy) && np_isclose(0.0, -uz)) {
    c0[0] = -1; c0[1] = 0; c0[2] = 0;
    a1[0] = 0; a1[1] = 1; a1[2] = 0;
    a2[0] = 0; a2[1] = 0; a2[2] = -1;
    return;
  }
  // R = I + K + K^2 (1 - c) / s^2 with k = e_x x u = (0, -uz, uy)
  // (1 - c) / s^2 with s = |k|: s^2 is taken as uy^2 + uz^2 directly (the reference squares the norm)
  double f = div_fast(1.0 - ux, uy * uy + uz * uz);
  c0[0] = 1.0 + (-(uy * uy) - (uz * uz)) * f; c0[1] = uy; c0[2] = uz;
  a1[0] = -uy; a1[1] = 1.0 + (-(uy * uy)) * f; a1[2] = (-(uy * uz)) * f;
  a2[0] = -uz; a2[1] = (-(uy * uz)) * f;       a2[2] = 1.0 + (-(uz * uz)) * f;
}

// sik:418-425 get_wrist_position: w = p + R * wo
R2IK_HD void wrist_from_goal(const ArmConst &A, const double p[3], const double R[9], double w[3]) {
  w[0] = R[0] * A.wo[0] + R[1] * A.wo[1] + R[2] * A.wo[2] + p[0];
  w[1] = R[3] * A.wo[0] + R[4] * A.wo[1] + R[5] * A.wo[2] + p[1];
  w[2] = R[6] * A.wo[0] + R[7] * A.wo[1] + R[8] * A.wo[2] + p[2];
}

// sik:337-349 reduce_goal_pose_no_limits: wrist pulled radially to distance d_target;
// the same displacement is applied to the goal.
R2IK_HD void reduce_goal(const ArmConst &A, double p[3], double w[3], double d, double d_target) {
  double sc = div_fast(d_target, fabs(d) + A.proj_margin);
  for (int k = 0; k < 3; ++k) {
    double nw = A.s[k] + (w[k] - A.s[k]) * sc;
    p[k] = p[k] + (nw - w[k]);
    w[k] = nw;
  }
}

// sik:366-399 get_intersection_circle (n = P/d form, SURVEY.md A.7).  false <=> None.
// (d, invd) = |w - s| and its reciprocal, computed by the caller from the current S.w.
// r2 = radius^2 (negative when the radicand is: the reference's radius is then nan); WANT_R = false skips the root.
template <bool WANT_R>
R2IK_HD bool elbow_circle(const ArmConst &A, Solve &S, double d, double invd, double n[3], double &r2) {
  double Px = S.w[0] - A.s[0], Py = S.w[1] - A.s[1], Pz = S.w[2] - A.s[2];
  if (d > A.L12) return false;
  double d2 = d * d;
  double k = d2 - A.L2sq + A.L1sq;
  double inv2d = 0.5 * invd;
  double rad = 4.0 * d2 * A.L1sq - k * k;          // < 0 by rounding at d ~ L1 + L2: np.sqrt gives nan
  r2 = rad * (inv2d * inv2d);
  if (WANT_R) S.r = hi_word(rad) < 0 ? NAN : inv2d * sqrt_nonneg(rad);
  double cd = k * inv2d;
  n[0] = Px * invd; n[1] = Py * invd; n[2] = Pz * invd;
  S.c[0] = n[0] * cd + A.s[0];
  S.c[1] = n[1] * cd + A.s[1];
  S.c[2] = n[2] * cd + A.s[2];
  return true;
}

// Result of the pose-level solve.
struct Reach {
  int state;        // R2IK_STATE_*
  double i0, i1;    // theta interval (i0 > i1 means wrapped); NaN when unreachable
  double c0, s0;    // cos(i0), sin(i0): lets get_joints(theta_interval[0]) skip a sincos
  bool degenerate;  // LIT = false only: the result is not valid, solve again with LIT = true
  bool literal;     // set by solve_core: the literal instantiation produced this result (and S)
};

constexpr double kSinMinusPi = -1.2246467991473532e-16;  // np.sin(-np.pi)

// sik:284-307 is_pose_in_robot_reach: out-of-reach projection and backward clamp of the goal
// position.  Returns -1 when the pose passes, else the reference's state code.
R2IK_HD int reach_prechecks(const ArmConst &A, double &px, double &py, double &pz) {
  int pre_state = -1;
  double dx = px - A.s[0], dy = py - A.s[1], dz = pz - A.s[2];
  // dg > max_arm_length decided on the squares; only a pose within 1e-12 of the sphere takes the root
  const double dg2 = dx * dx + dy * dy + dz * dz, L2 = A.max_arm_length * A.max_arm_length;
  bool outside = dg2 > L2;
  if (fabs(dg2 - L2) <= 1e-12) outside = sqrt(dg2) > A.max_arm_length;
  if (outside) {
    // a goal beyond ~1.3e154 m overflows dg2: the reference's norm is then inf and the goal lands on the shoulder
    // (dx / inf = 0), where sqrt_nonneg(inf) would be NaN
    double sc = dg2 < INFINITY ? div_fast(A.max_arm_length, sqrt_nonneg(dg2) + A.proj_margin) : 0.0;
    px = A.s[0] + dx * sc;
    py = A.s[1] + dy * sc;
    pz = A.s[2] + dz * sc;
    pre_state = R2IK_STATE_POSE_OUT_OF_REACH;
  }
  if (px < A.backward_limit) {
    px = A.backward_limit;
    pre_state = R2IK_STATE_BACKWARD_POSE;
  }
  return pre_state;
}

// Body of sik:121-282 is_reachable (NO_LIMITS = false) / sik:85-119 is_reachable_no_limits
// (true) after the pre-checks: S.p (pre-checked goal position) and S.R (goal rotation) are
// set by the caller.  FLAG_ONLY skips the interval angles (reach-map kernel): state is exact,
// i0/i1 are not computed.
// CIRCLE_ONLY: stop once the elbow circle and its frame are in S (a pose already known to be reachable whose
// interval is not needed again: the joints pass of the continuous mode).
template <bool NO_LIMITS, bool FLAG_ONLY, bool LIT, bool CIRCLE_ONLY = false>
R2IK_HD Reach solve_core_impl(const ArmConst &A, Solve &S) {
  Reach out;
  out.i0 = NAN; out.i1 = NAN; out.c0 = NAN; out.s0 = NAN; out.degenerate = false; out.literal = false;
  wrist_from_goal(A, S.p, S.R, S.w);
  // --- sik:146-153 / sik:94-98 keep the wrist in front of the torso plane
  if (S.w[0] < A.backward_limit) {
    double diff = A.backward_limit - S.w[0];
    S.p[0] = S.p[0] + diff;
    if (NO_LIMITS) wrist_from_goal(A, S.p, S.R, S.w);
    else S.w[0] = S.w[0] + diff;
  }
  double d, invd;
  {
    double dx = S.w[0] - A.s[0], dy = S.w[1] - A.s[1], dz = S.w[2] - A.s[2];
    d = sqrt_rsqrt_nonneg(dx * dx + dy * dy + dz * dz, invd);
  }
  bool moved = false;
  if (d > A.L12) {
    if (!NO_LIMITS) { out.state = R2IK_STATE_WRIST_OUT_OF_RANGE; return out; }
    reduce_goal(A, S.p, S.w, d, A.L12);                       // sik:102-105
    moved = true;
  }
  if (d < A.d_min) {                                          // sik:166-171 / sik:107-112
    reduce_goal(A, S.p, S.w, d, A.d_min);
    wrist_from_goal(A, S.p, S.R, S.w);
    moved = true;
  }
  if (moved) {   // rare: the wrist was pulled in / pushed out, its distance is recomputed (sik:376)
    double dx = S.w[0] - A.s[0], dy = S.w[1] - A.s[1], dz = S.w[2] - A.s[2];
    d = sqrt_rsqrt_nonneg(dx * dx + dy * dy + dz * dz, invd);
  }
  double n[3], r2;
  if (!elbow_circle<!FLAG_ONLY || LIT>(A, S, d, invd, n, r2)) { out.state = R2IK_STATE_SHOULD_NOT_HAPPEN; return out; }
  if (!FLAG_ONLY) {
    double c0[3];
    rmfv_columns(n[0], n[1], n[2], false, c0, S.a1, S.a2);    // sik:454, sik:686
  }
  if (NO_LIMITS) {
    out.state = R2IK_STATE_REACHABLE; out.i0 = -kPi; out.i1 = kPi; out.c0 = -1.0; out.s0 = kSinMinusPi;
    return out;
  }
  if (CIRCLE_ONLY) { out.state = R2IK_STATE_REACHABLE; return out; }

  // --- sik:401-416 wrist-limit circle, relative to the wrist: centre p1 = n1 * hL
  double nLx = S.w[0] - S.p[0], nLy = S.w[1] - S.p[1], nLz = S.w[2] - S.p[2];
  double inLn = rsqrt_pos(nLx * nLx + nLy * nLy + nLz * nLz);
  double n1[3] = {nLx * inLn, nLy * inLn, nLz * inLn};
  double p1[3] = {n1[0] * A.hL, n1[1] * A.hL, n1[2] * A.hL};
  double p2[3] = {S.c[0] - S.w[0], S.c[1] - S.w[1], S.c[2] - S.w[2]};
  const double *n2 = n;
  if (!LIT) {
    // Fast route: circle linking in the plane of the elbow circle.  Both circles lie on the forearm sphere
    // (centre w, radius L2), so the points where the reference's plane-plane line meets the limit circle
    // (sik:588-645) are the points of the ELBOW circle that lie in the limit plane n1 . (X - p1) = 0.  With
    // X(theta) = p2 + r (a1 cos theta + a2 sin theta), the signed x of X in the limitation frame -- the
    // quantity of the reference's mid-arc test, sik:541-558 -- is
    //     xl(theta) = Xc + r (A cos theta + B sin theta) = Xc + r rho cos(theta - phi),
    //     A = n1 . a1,  B = n1 . a2,  rho = |n1 x n2|,  Xc = n1 . (p2 - p1)   (sik:466-467),
    // hence: the discriminant of sik:608-645 has the sign of r^2 rho^2 - Xc^2; the intersection angles are
    // phi -+ alpha with cos(alpha) = kappa = -Xc / (r rho); and the reference's sort + mid-arc test keeps
    // the arc on which xl > 0, i.e. the interval runs counter-clockwise from phi - alpha to phi + alpha.
    // No line, no 3-D points, no sort: ~120 fewer FP64 operations per pose than the literal construction,
    // and theta is read off O(1) quantities instead of point coordinates at radius r.  Everything the
    // reference decides by a special case goes to the literal instantiation: rmfv(n1) near +-e_x, (nearly)
    // parallel planes, np.isclose line parameters, a radicand or discriminant within rounding of zero.
    const double b0 = p2[0] - p1[0], b1 = p2[1] - p1[1], b2 = p2[2] - p1[2];
    const double Xc = n1[0] * b0 + n1[1] * b1 + n1[2] * b2;
    const double nb = n2[0] * b0 + n2[1] * b1 + n2[2] * b2;
    double Aa = 0.0, Ba = 0.0, rho2;
    if (FLAG_ONLY) {
      const double Ca = n1[0] * n2[0] + n1[1] * n2[1] + n1[2] * n2[2];
      rho2 = fma(-Ca, Ca, 1.0);
    } else {
      Aa = n1[0] * S.a1[0] + n1[1] * S.a1[1] + n1[2] * S.a1[2];
      Ba = n1[0] * S.a2[0] + n1[1] * S.a2[1] + n1[2] * S.a2[2];
      rho2 = Aa * Aa + Ba * Ba;
    }
    const double rr = r2 * rho2;
    const double dl = rr - Xc * Xc;                       // sign of the reference's discriminant
    bool deg = fabs(n1[1]) < 1e-7 && fabs(n1[2]) < 1e-7;  // utl:66-70 special cases of rmfv(nL)
    // ... and of rmfv(n2): within its isclose band a1, a2 are e_y, +-e_z, up to 1e-8 rad off the plane normal to n2, so
    // X(theta) leaves the forearm sphere and the angles where it crosses the limit plane are not the reference's, which
    // converts the true intersection points with that frame.  (The flag pass needs no frame: rho2 = 1 - Ca^2 is exact.)
    // Tested on the high words, off the FP64 pipe: both |n2[1]|, |n2[2]| < 2^-24 (6e-8), a superset of the band.
    if (!FLAG_ONLY) deg = deg || ((hi_word(n2[1]) & 0x7fffffff) < 0x3e700000 && (hi_word(n2[2]) & 0x7fffffff) < 0x3e700000);
    deg = deg || !(rho2 > 1e-12);                         // sik:475-483 (|n2 -+ n1| < 1e-7 componentwise => rho2 < 3e-14)
    deg = deg || fabs(Xc - nb) <= 1e-8 + 1e-5 * fabs(nb); // superset of np.isclose(u, t), sik:581: u - t = (Xc - nb) / rho
    deg = deg || !(r2 > 0.0) || fabs(dl) <= 1e-12 * (rr + Xc * Xc);
    out.degenerate = out.degenerate || deg;
    if (dl < 0.0) {
      if (Xc > 0) { out.state = R2IK_STATE_REACHABLE; out.i0 = -kPi; out.i1 = kPi; out.c0 = -1.0; out.s0 = kSinMinusPi; }
      else out.state = R2IK_STATE_LIMITED_BY_WRIST;
      return out;
    }
    out.state = R2IK_STATE_REACHABLE;
    if (FLAG_ONLY) return out;
    const double irr = rsqrt_pos(rr);
    const double kappa = -Xc * irr, sp = sqrt_nonneg(dl) * irr;
    const double irho = rsqrt_pos(rho2);
    const double cph = Aa * irho, sph = Ba * irho;
    const double c_lo = cph * kappa + sph * sp, s_lo = sph * kappa - cph * sp;   // phi - alpha
    const double c_hi = cph * kappa - sph * sp, s_hi = sph * kappa + cph * sp;   // phi + alpha
    out.i0 = angle_of_unit(c_lo, s_lo);
    out.i1 = angle_of_unit(c_hi, s_hi);
    out.c0 = c_lo; out.s0 = s_lo;
    return out;
  }
  // Literal route: the reference's own construction.
  // column 0 of rotation_matrix_from_vector(nL): only the x row of T_limitation_torso is used
  double l0[3], t1[3], t2[3];
  rmfv_columns(n1[0], n1[1], n1[2], false, l0, t1, t2);
  // sik:466-467 P_limitation_intersectionCenter[0]
  double Xc = l0[0] * (p2[0] - p1[0]) + l0[1] * (p2[1] - p1[1]) + l0[2] * (p2[2] - p1[2]);

  bool linked_full = false, decided = false;
  // sik:475-483 parallel planes
  {
    bool pa = (fabs(n2[0] - n1[0]) < A.nvm) && (fabs(n2[1] - n1[1]) < A.nvm) && (fabs(n2[2] - n1[2]) < A.nvm);
    bool pb = (fabs(n2[0] + n1[0]) < A.nvm) && (fabs(n2[1] + n1[1]) < A.nvm) && (fabs(n2[2] + n1[2]) < A.nvm);
    if (pa || pb) { decided = true; linked_full = Xc > 0; }
  }
  double q[3], v[3];
  if (!decided) {
    // sik:588-606 line of intersection of the two planes; sik:570-586 closed form of lstsq
    v[0] = n1[1] * n2[2] - n1[2] * n2[1];
    v[1] = n1[2] * n2[0] - n1[0] * n2[2];
    v[2] = n1[0] * n2[1] - n1[1] * n2[0];
    double inv = rsqrt_pos(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    v[0] *= inv; v[1] *= inv; v[2] *= inv;
    double e1[3] = {v[1] * n1[2] - v[2] * n1[1], v[2] * n1[0] - v[0] * n1[2], v[0] * n1[1] - v[1] * n1[0]};
    double b[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
    // Line parameters of the consistent 3x2 system [e1 -e2](t, u)^T = b with e_i = v x n_i:
    //   t = (n2 . b) / (n2 . e1),  u = -(n1 . b) / (n1 . e2),  and  n2 . e1 = -(n1 . e2) = v . (n1 x n2)
    //   = |n1 x n2| = 1 / inv: both share the reciprocal that normalised v.
    double t = (n2[0] * b[0] + n2[1] * b[1] + n2[2] * b[2]) * inv;
    double u = (n1[0] * b[0] + n1[1] * b[1] + n1[2] * b[2]) * inv;
    if (np_isclose(u, t)) { decided = true; linked_full = Xc > 0; }
    q[0] = e1[0] * t + p1[0]; q[1] = e1[1] * t + p1[1]; q[2] = e1[2] * t + p1[2];
  }
  if (!decided) {
    // sik:608-645 limit circle (centre p1, radius rL) with the line q + t v
    double wv[3] = {q[0] - p1[0], q[1] - p1[1], q[2] - p1[2]};
    double qa = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    double qb = 2.0 * (v[0] * wv[0] + v[1] * wv[1] + v[2] * wv[2]);
    double qc = (wv[0] * wv[0] + wv[1] * wv[1] + wv[2] * wv[2]) - A.rLsq;
    double disc = qb * qb - 4.0 * qa * qc;
    if (disc < 0) {
      decided = true; linked_full = Xc > 0;
    } else if (FLAG_ONLY) {
      out.state = R2IK_STATE_REACHABLE;   // one or two intersection points: an interval exists
      return out;
    } else {
      // sik:511-568 angles of the intersection points in the elbow-circle frame
      double sq = sqrt_nonneg(disc);
      double inv2a = rcp_fast(2.0 * qa);
      double ta = (disc == 0) ? (-qb * inv2a) : ((-qb + sq) * inv2a);
      double Pa[3] = {q[0] + ta * v[0] - p2[0], q[1] + ta * v[1] - p2[1], q[2] + ta * v[2] - p2[2]};
      double ya = S.a2[0] * Pa[0] + S.a2[1] * Pa[1] + S.a2[2] * Pa[2];
      double xa = S.a1[0] * Pa[0] + S.a1[1] * Pa[1] + S.a1[2] * Pa[2];
      double ca, sa;                      // cos / sin of ang1 (unit vector of the point in the circle plane)
      double ang1 = cs_and_angle<LIT>(ya, xa, ca, sa, out.degenerate);
      if (disc == 0) {
        out.state = R2IK_STATE_REACHABLE; out.i0 = ang1; out.i1 = ang1;
        out.c0 = ca; out.s0 = sa;
        return out;
      }
      double tb = (-qb - sq) * inv2a;
      double Pb[3] = {q[0] + tb * v[0] - p2[0], q[1] + tb * v[1] - p2[1], q[2] + tb * v[2] - p2[2]};
      double yb = S.a2[0] * Pb[0] + S.a2[1] * Pb[1] + S.a2[2] * Pb[2];
      double xb = S.a1[0] * Pb[0] + S.a1[1] * Pb[1] + S.a1[2] * Pb[2];
      double cb, sb;
      double ang2 = cs_and_angle<LIT>(yb, xb, cb, sb, out.degenerate);
      if (ang2 < ang1) {
        double tmp = ang1; ang1 = ang2; ang2 = tmp;
        tmp = ca; ca = cb; cb = tmp;
        tmp = sa; sa = sb; sb = tmp;
      }
      // cos / sin of the mid-arc angle (ang1 + ang2) / 2 (sik:541-547): the bisector of the two unit
      // vectors, reversed when the arc from ang1 to ang2 is longer than pi.  Exactly opposite points
      // (|bisector| ~ 0) are flagged degenerate and take the literal sincos.
      double sm, cm;
      if (LIT) {
        sincos((ang1 + ang2) / 2.0, &sm, &cm);
      } else {
        double bx = ca + cb, by = sa + sb;
        double b2 = bx * bx + by * by;
        out.degenerate = out.degenerate || !(b2 > 1e-12);
        double ib = rsqrt_pos(b2);
        if (ang2 - ang1 > kPi) ib = -ib;
        cm = bx * ib; sm = by * ib;
      }
      double yc = cm * S.r, zc = sm * S.r;
      // test point in the torso(wrist-relative) frame, then its x in the limitation frame
      double Tm[3] = {S.a1[0] * yc + S.a2[0] * zc + p2[0] - p1[0], S.a1[1] * yc + S.a2[1] * zc + p2[1] - p1[1],
                      S.a1[2] * yc + S.a2[2] * zc + p2[2] - p1[2]};
      double xl = l0[0] * Tm[0] + l0[1] * Tm[1] + l0[2] * Tm[2];
      out.state = R2IK_STATE_REACHABLE;
      if (xl > 0) { out.i0 = ang1; out.i1 = ang2; out.c0 = ca; out.s0 = sa; }
      else { out.i0 = ang2; out.i1 = ang1; out.c0 = cb; out.s0 = sb; }
      return out;
    }
  }
  if (linked_full) { out.state = R2IK_STATE_REACHABLE; out.i0 = -kPi; out.i1 = kPi; out.c0 = -1.0; out.s0 = kSinMinusPi; }
  else out.state = R2IK_STATE_LIMITED_BY_WRIST;
  return out;
}

// sik:121-282 is_reachable / sik:85-119 is_reachable_no_limits for a goal position and a goal
// rotation matrix already stored in S.R.  Fills S for get_joints / elbow_position.
// Out-of-line literal instantiation (see "Fast / literal duality"): S travels through a local
// copy so that the caller's S stays in registers on the hot path.
template <bool NO_LIMITS, bool FLAG_ONLY>
#if defined(__CUDACC__)
__host__ __device__ __noinline__
#else
inline
#endif
void solve_core_literal(const ArmConst &A, Solve *S, Reach *out) {
  *out = solve_core_impl<NO_LIMITS, FLAG_ONLY, true>(A, *S);
}

// S.p (pre-checked goal position) and S.R (goal rotation) set by the caller.
template <bool NO_LIMITS, bool FLAG_ONLY>
R2IK_HD Reach solve_core(const ArmConst &A, Solve &S) {
  const double p0 = S.p[0], p1 = S.p[1], p2 = S.p[2];
  Reach out = solve_core_impl<NO_LIMITS, FLAG_ONLY, false>(A, S);
  if (out.degenerate) {
    Solve T;
    T.p[0] = p0; T.p[1] = p1; T.p[2] = p2;
    for (int k = 0; k < 9; ++k) T.R[k] = S.R[k];
    Reach lit;
    solve_core_literal<NO_LIMITS, FLAG_ONLY>(A, &T, &lit);
    S = T;
    out = lit;
    out.literal = true;
  }
  return out;
}

// Elbow circle of a pose that is_reachable has already accepted (pre-checks passed, wrist in range): the state
// is_reachable leaves in S, without the circle linking.
R2IK_HD void circle_of_reachable(const ArmConst &A, const double pos[3], Solve &S) {
  S.p[0] = pos[0]; S.p[1] = pos[1]; S.p[2] = pos[2];
  solve_core_impl<false, false, false, true>(A, S);
}

template <bool NO_LIMITS>
R2IK_HD Reach is_reachable_R(const ArmConst &A, const double pos[3], Solve &S) {
  double px = pos[0], py = pos[1], pz = pos[2];
  int pre_state = reach_prechecks(A, px, py, pz);
  if (!NO_LIMITS && pre_state >= 0) {
    Reach out;
    out.state = pre_state; out.i0 = NAN; out.i1 = NAN; out.c0 = NAN; out.s0 = NAN; out.degenerate = false; out.literal = false;
    return out;
  }
  S.p[0] = px; S.p[1] = py; S.p[2] = pz;
  return solve_core<NO_LIMITS, false>(A, S);
}

// The same from the reference's goal_pose (position, xyz euler).
template <bool NO_LIMITS>
R2IK_HD Reach is_reachable(const ArmConst &A, const double pos[3], const double eul[3], Solve &S) {
  rot_from_euler_xyz(eul[0], eul[1], eul[2], S.R);
  return is_reachable_R<NO_LIMITS>(A, pos, S);
}

// sik:684-695 get_elbow_position, from (cos theta, sin theta)
R2IK_HD void elbow_position_cs(const Solve &S, double ct, double st, double E[3]) {
  double y = S.r * ct, z = S.r * st;
  E[0] = S.a1[0] * y + S.a2[0] * z + S.c[0];
  E[1] = S.a1[1] * y + S.a2[1] * z + S.c[1];
  E[2] = S.a1[2] * y + S.a2[2] * z + S.c[2];
}

R2IK_HD void elbow_position(const Solve &S, double theta, double E[3]) {
  double st, ct;
  sincos_any(theta, st, ct);
  double y = S.r * ct, z = S.r * st;
  E[0] = S.a1[0] * y + S.a2[0] * z + S.c[0];
  E[1] = S.a1[1] * y + S.a2[1] * z + S.c[1];
  E[2] = S.a1[2] * y + S.a2[2] * z + S.c[2];
}

// utl:443-465 is_elbow_ok (effective predicate; the first test is dead code, utl:452-457)
R2IK_HD bool is_elbow_ok(const ArmConst &A, const double E[3]) {
  bool ok = (E[1] * A.side < -0.2);
  ok = ok && (E[2] < (E[0] - A.es[0]) * A.sing_coeff + A.es[2] - A.sing_offset);
  return ok;
}

// sik:697-718: get_joints takes the make_elbow_projection branch for this elbow position.  (The reference then returns
// the elbow as a 3-vector instead of get_elbow_position's homogeneous [x, y, z, 1], sik:714, :863.)
R2IK_HD bool elbow_projection_fires(const ArmConst &A, const double E[3]) {
  return E[2] > (E[0] - A.es[0]) * A.sing_coeff + A.es[2] - A.sing_offset;
}

// 2-D rotation helpers: the reference's elementary frame changes (sik:758-837)
struct P3 { double x, y, z; };
R2IK_HD void rot_y(P3 &p, double c, double s) {  // R_y(a) with c = cos a, s = sin a
  double x = c * p.x + s * p.z, z = -s * p.x + c * p.z;
  p.x = x; p.z = z;
}
R2IK_HD void rot_z(P3 &p, double c, double s) {  // R_z(a)
  double x = c * p.x - s * p.y, y = s * p.x + c * p.y;
  p.x = x; p.y = y;
}
R2IK_HD void rot_x(P3 &p, double c, double s) {  // R_x(a)
  double y = c * p.y - s * p.z, z = s * p.y + c * p.z;
  p.y = y; p.z = z;
}
R2IK_HD P3 to_shoulder(const ArmConst &A, const double X[3]) {
  P3 o;
  o.x = A.Mst[0] * X[0] + A.Mst[1] * X[1] + A.Mst[2] * X[2] + A.Pst[0];
  o.y = A.Mst[3] * X[0] + A.Mst[4] * X[1] + A.Mst[5] * X[2] + A.Pst[1];
  o.z = A.Mst[6] * X[0] + A.Mst[7] * X[1] + A.Mst[8] * X[2] + A.Pst[2];
  return o;
}

// sik:697-863 get_joints.  Mutates S like the reference when the elbow projection fires
// (sik:708-718: goal_pose, elbow_position, wrist_position).  prev0 / prev2 are
// previous_joints[0] / [2], used only at the exact-zero singularities (sik:751, 782).
// (ct, st) = (cos theta, sin theta).  The reference's frame rotations R(+-joint angle) are
// applied from the (cos, sin) of the atan2 that defines the joint (cs_of_atan2): the seven
// atan2 that produce the outputs are then off the dependent chain.
// Returns false (LIT = false only) when a degenerate input needs the literal instantiation; S.p /
// S.w may then have been modified and must be restored by the caller.
template <bool LIT>
R2IK_HD bool get_joints_impl(const ArmConst &A, Solve &S, double ct, double st, double prev0, double prev2, double joints[7],
                             double E[3]) {
  bool degenerate = false;
  elbow_position_cs(S, ct, st, E);
  if (elbow_projection_fires(A, E)) {
    // sik:647-682 make_elbow_projection with the plane constants hoisted to the host
    double dist = (E[0] - A.plP[0]) * A.plV[0] + (E[1] - A.plP[1]) * A.plV[1] + (E[2] - A.plP[2]) * A.plV[2];
    double vc[3] = {E[0] - dist * A.plV[0] - A.plC[0], E[1] - dist * A.plV[1] - A.plC[1], E[2] - dist * A.plV[2] - A.plC[2]};
    double sc = A.plRho * rsqrt_pos(vc[0] * vc[0] + vc[1] * vc[1] + vc[2] * vc[2]);
    for (int k = 0; k < 3; ++k) {
      double ne = A.plC[k] + vc[k] * sc;
      S.p[k] = S.p[k] + (ne - E[k]);
      E[k] = ne;
    }
    wrist_from_goal(A, S.p, S.R, S.w);
  }
  // points carried through the frames: elbow, wrist, tip point, a point 0.1 along the goal x axis
  double tipw[3] = {S.R[0] * A.to[0] + S.R[1] * A.to[1] + S.R[2] * A.to[2] + S.p[0],
                    S.R[3] * A.to[0] + S.R[4] * A.to[1] + S.R[5] * A.to[2] + S.p[1],
                    S.R[6] * A.to[0] + S.R[7] * A.to[1] + S.R[8] * A.to[2] + S.p[2]};
  double ptw[3] = {S.R[0] * 0.1 + tipw[0], S.R[3] * 0.1 + tipw[1], S.R[6] * 0.1 + tipw[2]};
  P3 el = to_shoulder(A, E), wr = to_shoulder(A, S.w), tp = to_shoulder(A, tipw), pt = to_shoulder(A, ptw);
  double s, c;

  // Six of the seven joint angles are atan2 of a pair whose (cos, sin) also drives the next frame
  // rotation: cs_and_angle normalises once and reads the angle off the unit vector.  The angles are
  // leaves of the dependency graph (nothing downstream consumes them), so their polynomial
  // evaluations interleave with the frame chain on the FP64 pipe.
  double at[7];
  // sik:751-755 shoulder pitch; sik:758 R_y(-shoulder_pitch)
  const bool sing0 = is_zero(el.x) && is_zero(el.z);
  if (LIT && sing0) { at[0] = 0.0; sincos(-prev0, &s, &c); }
  else at[0] = cs_and_angle<LIT>(el.z, el.x, c, s, degenerate);
  rot_y(el, c, s); rot_y(wr, c, s); rot_y(tp, c, s); rot_y(pt, c, s);
  // sik:766 shoulder roll = atan2(el.y, el.x); sik:769 R_z(-shoulder_roll)
  at[1] = -cs_and_angle<LIT>(-el.y, el.x, c, s, degenerate);
  rot_z(wr, c, s); rot_z(tp, c, s); rot_z(pt, c, s);
  wr.x -= A.L1; tp.x -= A.L1; pt.x -= A.L1;        // sik:776-777 elbow frame
  // sik:782-786 elbow yaw (not wrapped: range (-3pi/2, pi/2]); sik:789 R_x(elbow_yaw):
  // cos(-pi/2 + a) = sin a, sin(-pi/2 + a) = -cos a with a = atan2(wr.z, -wr.y)
  const bool sing2 = is_zero(wr.y) && is_zero(wr.z);
  if (LIT && sing2) { at[2] = 0.0; sincos(prev2, &s, &c); }
  else {
    double ca, sa;
    at[2] = cs_and_angle<LIT>(wr.z, -wr.y, ca, sa, degenerate);
    c = sa; s = -ca;
  }
  rot_x(wr, c, s); rot_x(tp, c, s); rot_x(pt, c, s);
  // sik:797 elbow pitch; sik:800 R_y(-elbow_pitch)
  at[3] = cs_and_angle<LIT>(wr.z, wr.x, c, s, degenerate);
  rot_y(tp, c, s); rot_y(pt, c, s);
  tp.x -= A.L2; pt.x -= A.L2;                      // sik:805-806 wrist frame
  // sik:815-817 wrist roll = pi - atan2(tp.y, -tp.x); sik:820 R_z(-wrist_roll):
  // cos(-(pi - a)) = -cos a, sin(-(pi - a)) = -sin a
  {
    double ca, sa;
    at[4] = cs_and_angle<LIT>(tp.y, -tp.x, ca, sa, degenerate);
    c = -ca; s = -sa;
  }
  rot_z(tp, c, s); rot_z(pt, c, s);
  // sik:826 wrist pitch; sik:829 R_y(wrist_pitch)
  at[5] = cs_and_angle<LIT>(tp.z, tp.x, c, s, degenerate);
  rot_y(pt, c, s);
  // (the x -= tip_z of sik:836-837 does not touch y, z); sik:848 wrist yaw
  at[6] = atan2_leaf<LIT>(pt.y, pt.z, degenerate);
  // exact-zero singularities (sik:751, 782) make cs_of_atan2 flag the pose: literal route
  double shoulder_pitch = sing0 ? prev0 : -at[0];
  double shoulder_roll = at[1];
  double elbow_yaw = sing2 ? prev2 : -kHalfPi + at[2];
  double elbow_pitch = -at[3];
  double wrist_roll = kPi - at[4];
  if (wrist_roll > kPi) wrist_roll = wrist_roll - kTwoPi;
  double wrist_pitch = at[5];
  double wrist_yaw = -at[6];

  joints[0] = shoulder_pitch; joints[1] = shoulder_roll; joints[2] = elbow_yaw; joints[3] = elbow_pitch;
  joints[4] = wrist_roll; joints[5] = -wrist_pitch; joints[6] = -wrist_yaw;
  if (joints[3] > A.elbow_limit) joints[3] = A.elbow_limit;     // sik:853-861
  if (joints[3] < -A.elbow_limit) joints[3] = -A.elbow_limit;
  return !degenerate;
}

#if defined(__CUDACC__)
__host__ __device__ __noinline__
#else
inline
#endif
void get_joints_literal(const ArmConst &A, Solve *S, double ct, double st, double prev0, double prev2, double *joints,
                        double *E) {
  get_joints_impl<true>(A, *S, ct, st, prev0, prev2, joints, E);
}

R2IK_HD void get_joints_cs(const ArmConst &A, Solve &S, double ct, double st, double prev0, double prev2, double joints[7],
                           double E[3]) {
  const double p0 = S.p[0], p1 = S.p[1], p2 = S.p[2], w0 = S.w[0], w1 = S.w[1], w2 = S.w[2];
  if (!get_joints_impl<false>(A, S, ct, st, prev0, prev2, joints, E)) {
    Solve T = S;   // local copy: only this rare path touches memory
    T.p[0] = p0; T.p[1] = p1; T.p[2] = p2; T.w[0] = w0; T.w[1] = w1; T.w[2] = w2;
    double jj[7], EE[3];
    get_joints_literal(A, &T, ct, st, prev0, prev2, jj, EE);
    S = T;
    for (int k = 0; k < 7; ++k) joints[k] = jj[k];
    for (int k = 0; k < 3; ++k) E[k] = EE[k];
  }
}

R2IK_HD void get_joints(const ArmConst &A, Solve &S, double theta, double prev0, double prev2, double joints[7], double E[3]) {
  double st, ct;
  sincos_any(theta, st, ct);
  get_joints_cs(A, S, ct, st, prev0, prev2, joints, E);
}

// ---------------------------------------------------------------------------------------
// Pose loading (the reference's goal_pose is (position, xyz euler))
// ---------------------------------------------------------------------------------------
// MAT4 layout, SymbolicIK batch: euler = R.from_matrix(M[:3,:3]).as_euler("xyz") (utl:84-90);
// snap = ControlIK front end (ctl:212-217) which replaces near-identity rotations by zeros.
R2IK_HD bool pose_from_mat4(const double *M, bool snap, double pos[3], double eul[3]) {
  pos[0] = M[3]; pos[1] = M[7]; pos[2] = M[11];
  if (snap && rotation_is_identity(M)) { eul[0] = 0.0; eul[1] = 0.0; eul[2] = 0.0; return true; }
  return euler_xyz_from_mat4(M, eul);
}

// Goal rotation the solver sees for a 4x4 input.  The reference converts M to xyz Euler angles
// (from_matrix -> as_euler, utl:84-90) and every later use rebuilds the matrix from them
// (from_euler, sik:420): for a rotation matrix that round trip is the identity up to rounding,
// so an orthonormal (Gramian within 1e-13 of I), right-handed M outside scipy's gimbal-lock
// band is used as it is.  Anything else -- scaled / skewed input that scipy projects or
// normalises, |cos(pitch)| < 1e-5 where as_euler zeroes the third angle (rxp:1085-1099),
// det <= 0 -- takes the literal route.  false <=> scipy raises (det <= 0).
// Literal route of rotation_from_mat4: from_matrix -> as_euler("xyz") -> from_euler (utl:84-90,
// sik:420).  Out of line on the device: it is the rare path (non-orthonormal or gimbal-band
// input) and it is large (SVD-equivalent projection, three atan2, three sincos).
#if defined(__CUDACC__)
__host__ __device__ __noinline__
#else
inline
#endif
bool rotation_from_mat3_literal(const double m[9], double R[9]) {
  if (!(det3(m) > 0.0)) return false;
  // A block that fails scipy's orthogonality test (rxp:78-95) is replaced there by its polar factor; outside the
  // gimbal band of as_euler the from_matrix -> as_euler -> from_euler round trip of that factor is the identity
  // up to rounding, so the factor is the goal rotation (saves the quaternion / three atan2 / three sincos detour
  // for every non-orthonormal input, e.g. all float32-rounded rotations re-solved by the FP32 path).
  {
    bool orthogonal = true;
    for (int i = 0; i < 3; ++i)
      for (int j = i; j < 3; ++j) {
        double g = m[3 * i] * m[3 * j] + m[3 * i + 1] * m[3 * j + 1] + m[3 * i + 2] * m[3 * j + 2];
        double e = (i == j) ? 1.0 : 0.0;
        if (!(fabs(g - e) <= 1e-12 + 1e-5 * e)) orthogonal = false;
      }
    if (!orthogonal) {
      double p[9];
      for (int k = 0; k < 9; ++k) p[k] = m[k];
      polar_orthogonalize(p);
      if (p[0] * p[0] + p[3] * p[3] > 1e-10) {
        for (int k = 0; k < 9; ++k) R[k] = p[k];
        return true;
      }
    }
  }
  double e[3];
  Quat q;
  if (!quat_from_matrix(m, q)) return false;
  quat_as_euler_xyz_extrinsic(q, e);
  rot_from_euler_xyz(e[0], e[1], e[2], R);
  return true;
}

R2IK_HD bool rotation_from_mat4(const double *M, bool snap, double R[9]) {
  if (snap && rotation_is_identity(M)) {
    R[0] = 1; R[1] = 0; R[2] = 0; R[3] = 0; R[4] = 1; R[5] = 0; R[6] = 0; R[7] = 0; R[8] = 1;
    return true;
  }
  const double m[9] = {M[0], M[1], M[2], M[4], M[5], M[6], M[8], M[9], M[10]};
  bool direct = true;
  for (int i = 0; i < 3; ++i)
    for (int j = i; j < 3; ++j) {
      double g = m[3 * i] * m[3 * j] + m[3 * i + 1] * m[3 * j + 1] + m[3 * i + 2] * m[3 * j + 2];
      double e = (i == j) ? 1.0 : 0.0;
      if (!(fabs(g - e) <= 1e-13)) direct = false;
    }
  if (!(m[0] * m[0] + m[3] * m[3] > 1e-10)) direct = false;   // cos^2(pitch)
  if (!(det3(m) > 0.0)) direct = false;
  if (direct) {
    for (int k = 0; k < 9; ++k) R[k] = m[k];
    return true;
  }
  // address-taken copies live in local memory only on this rare path; m / R stay in registers
  double mm[9], RR[9];
  for (int k = 0; k < 9; ++k) mm[k] = m[k];
  bool ok = rotation_from_mat3_literal(mm, RR);
  for (int k = 0; k < 9; ++k) R[k] = RR[k];
  return ok;
}

// Doubles per row of a pose buffer
R2IK_HD constexpr int pose_stride(int kind) { return kind == R2IK_POSE_EULER6 ? 6 : kind == R2IK_POSE_MAT34 ? 12 : 16; }

// Two doubles at a 16-byte aligned address (pose buffers: checked by the C entry points): one 128-bit read-only load on
// the device
R2IK_HD void load2(const double *p, double &a, double &b) {
#if defined(__CUDA_ARCH__)
  const double2 v = __ldg(reinterpret_cast<const double2 *>(p));
  a = v.x; b = v.y;
#else
  a = p[0]; b = p[1];
#endif
}

// 3x4 top of a row-major 4x4 (the last row is never read): 6 x 128-bit loads
R2IK_HD void load_mat4(const double *M, double m[16]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    load2(M + 4 * r, m[4 * r], m[4 * r + 1]);
    load2(M + 4 * r + 2, m[4 * r + 2], m[4 * r + 3]);
  }
  m[12] = 0.0; m[13] = 0.0; m[14] = 0.0; m[15] = 1.0;
}

// Goal position + goal rotation matrix of one pose row.  false <=> invalid rotation (det <= 0).  MAT34 rows are the
// 3x4 top of the matrix, 12 doubles per pose: every byte that crosses HBM (and PCIe) is used.
template <int KIND>
R2IK_HD bool load_pose(const double *row, bool snap, double pos[3], double R[9]) {
  if (KIND == R2IK_POSE_EULER6) {
    double e[3];
    load2(row, pos[0], pos[1]);
    load2(row + 2, pos[2], e[0]);
    load2(row + 4, e[1], e[2]);
    rot_from_euler_xyz(e[0], e[1], e[2], R);
    return true;
  }
  double m[16];
  load_mat4(row, m);
  pos[0] = m[3]; pos[1] = m[7]; pos[2] = m[11];
  return rotation_from_mat4(m, snap, R);
}

// ---------------------------------------------------------------------------------------
// Per-pose bodies of the SymbolicIK kernels (r2ik_kernels.cu; tests/hostsim loops over the same functions)
// ---------------------------------------------------------------------------------------
// K1, solve: is_reachable (NO_LIMITS: is_reachable_no_limits) on a pose row (INVALID_ROTATION with a NaN interval for
// det <= 0).
template <int KIND, bool NO_LIMITS = false>
R2IK_HD Reach symik_reach(const ArmConst &A, const double *row, Solve &S) {
  double pos[3];
  Reach rc;
  rc.state = R2IK_STATE_INVALID_ROTATION; rc.i0 = NAN; rc.i1 = NAN;
  if (load_pose<KIND>(row, false, pos, S.R)) rc = is_reachable_R<NO_LIMITS>(A, pos, S);
  return rc;
}

// K1, joints: get_joints at *theta, or without theta at theta_interval[0] (its cos / sin come with the interval); NaN
// for a pose that is not reachable.
R2IK_HD void symik_joints(const ArmConst &A, Solve &S, const Reach &rc, const double *theta, double prev0, double prev2,
                          double j[7], double E[3]) {
  if (rc.state == R2IK_STATE_REACHABLE) {
    double ct = rc.c0, st = rc.s0;
    if (theta) sincos_any(*theta, st, ct);
    get_joints_cs(A, S, ct, st, prev0, prev2, j, E);
  } else {
#pragma unroll
    for (int k = 0; k < 7; ++k) j[k] = NAN;
    E[0] = NAN; E[1] = NAN; E[2] = NAN;
  }
}

// K1b: is_reachable_no_limits + get_joints(*theta, prev[0], prev[2]) (prev may be null: zeros; they only matter at the
// exact singularities, sik:751, 782).  NaN without an elbow circle or for an invalid rotation.  Returns whether the
// elbow projection fires at theta.
template <int KIND>
R2IK_HD bool symik_no_limits(const ArmConst &A, const double *row, const double *theta, const double *prev, double j[7],
                             double E[3]) {
  double pos[3];
  Solve S;
  bool ok = load_pose<KIND>(row, false, pos, S.R);
  if (ok) ok = is_reachable_R<true>(A, pos, S).state == R2IK_STATE_REACHABLE;
  bool proj = false;
  if (ok) {
    double prev0 = 0.0, prev2 = 0.0;
    if (prev) { prev0 = prev[0]; prev2 = prev[2]; }
    double st, ct, Ep[3];
    sincos_any(*theta, st, ct);
    elbow_position_cs(S, ct, st, Ep);
    proj = elbow_projection_fires(A, Ep);
    get_joints_cs(A, S, ct, st, prev0, prev2, j, E);
  } else {
    for (int k = 0; k < 7; ++k) j[k] = NAN;
    E[0] = NAN; E[1] = NAN; E[2] = NAN;
  }
  return proj;
}

// K1b: the elbow circle is_reachable (NO_LIMITS = false) or is_reachable_no_limits (true) stores for a pose row.  The
// reference stores the circle as soon as it exists (sik:197), i.e. also when the wrist limit then rejects the pose.
// false: no circle.
template <int KIND, bool NO_LIMITS>
R2IK_HD bool pose_elbow_circle(const ArmConst &A, const double *row, Solve &S) {
  double pos[3];
  bool ok = load_pose<KIND>(row, false, pos, S.R);
  if (ok) {
    const int st = is_reachable_R<NO_LIMITS>(A, pos, S).state;
    ok = st == R2IK_STATE_REACHABLE || (!NO_LIMITS && st == R2IK_STATE_LIMITED_BY_WRIST);
  }
  return ok;
}

// Elbow-angle sweep (k_symik_sweep): angle k of K for a pose solved by symik_reach.  row: the pose's K given angles, or
// null for K samples placed on theta_interval as get_best_discrete_theta places them (utl:366-375).  NaN for a pose
// that is not reachable.
R2IK_HD double sweep_theta(const Reach &rc, const double *row, int K, int k) {
  if (rc.state != R2IK_STATE_REACHABLE) return NAN;
  if (row) return row[k];
  double start, stop;
  search_range(rc.i0, rc.i1, start, stop);
  return linspace_value(make_linspace(start, stop, K), k);
}

// One sample of the sweep: get_joints(theta) as the first call on the pose's solve S0 -- the value K1 (K1b) returns for
// the same pose and theta.  get_joints moves S.p / S.w when the elbow projection fires, so every sample starts from its
// own copy of S0.  NaN for a pose that is not reachable.  Returns whether the elbow projection fires at theta.
R2IK_HD bool sweep_sample(const ArmConst &A, const Solve &S0, const Reach &rc, double theta, double prev0, double prev2,
                          double j[7], double E[3]) {
  if (rc.state != R2IK_STATE_REACHABLE) {
    for (int k = 0; k < 7; ++k) j[k] = NAN;
    E[0] = NAN; E[1] = NAN; E[2] = NAN;
    return false;
  }
  Solve S = S0;
  double st, ct, Ep[3];
  sincos_any(theta, st, ct);
  elbow_position_cs(S, ct, st, Ep);
  const bool proj = elbow_projection_fires(A, Ep);
  get_joints_cs(A, S, ct, st, prev0, prev2, j, E);
  return proj;
}

// get_elbow_position(*theta) on that circle (NaN without one).  Returns whether the elbow projection fires there.
R2IK_HD bool elbow_on_circle(const ArmConst &A, const Solve &S, bool circle, const double *theta, double E[3]) {
  E[0] = NAN; E[1] = NAN; E[2] = NAN;
  if (!circle) return false;
  double st, ct;
  sincos_any(*theta, st, ct);
  elbow_position_cs(S, ct, st, E);
  return elbow_projection_fires(A, E);
}

}  // namespace r2ik
