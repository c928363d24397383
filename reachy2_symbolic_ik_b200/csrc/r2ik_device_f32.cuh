// r2ik_device_f32.cuh -- FP32 fast path of the per-pose solver (is_reachable + get_joints), sm_100a.
//
// BASELINE.json north_star: "the FP64 path is the correctness reference and an FP32 fast path is
// optional ... FP32 path within a stated 1e-4 rad".  This header restates the K1 part of
// r2ik_device.cuh (sik:121-282 is_reachable, sik:697-863 get_joints and what they call) in single
// precision: float4 pose loads, MUFU.RSQ / MUFU.RCP seeds used as they are (no Newton steps), 5-term
// polynomials, 32-bit registers -- twice the arithmetic rate of the FP64 pipe and half the bytes.  The few
// differences that cancel catastrophically for a nearly straight arm (wrist centre, its distance to the
// shoulder, the radicand of the elbow-circle radius) stay in FP64 on the exactly-widened inputs, and the
// circle linking uses the in-plane form of r2ik_device.cuh, which divides one well-conditioned scalar by
// r rho instead of locating points of a small circle from FP32 coordinates.
//
// What FP32 cannot do is take the reference's DECISIONS (state codes, interval order, branch cuts of
// atan2, the elbow-projection predicate) when a pose sits within rounding distance of one of them, and
// it cannot resolve the exact-zero special cases.  The fast / literal duality of the FP64 solver is
// therefore extended by one level: every decision of the FP32 solve tests its margin against an error
// band of a few FP32 ulps of the quantities involved and ORs "too close to call" into an `esc` flag;
// a flagged pose is solved again by the FP64 solver (a second kernel over the compacted list of flagged
// poses, from the same FP32 inputs widened to double) and its results are narrowed to float.  States and
// flags of the FP32 path are thereby the FP64 path's states on the same inputs; joints and intervals
// carry FP32 rounding (5e-7 rad median, 1.6e-5 at the 99.9th percentile), amplified where the geometry
// itself is ill-conditioned (a point on a joint axis, interval ends of a tiny elbow circle) -- those poses
// are also escalated when the lever is visible in the fast solve (the squared length under an atan2,
// (r rho sin alpha)^2 for the interval ends).  The same machinery decides the (voxel, orientation) pairs of
// the workspace reachability map (reach_flag_mixed, K4).
//
// "sik" = src/reachy2_symbolic_ik/symbolic_ik.py, "utl" = .../utils.py (reference checkout).
#pragma once

#include "r2ik_device.cuh"

#ifdef R2IK_F32_DEBUG
static float g_dbg[16]; static int g_dbg_n = 0;
static inline void r2ik_f32_dbg(float v) { if (g_dbg_n < 16) g_dbg[g_dbg_n++] = v; }
#endif
// escalation test n: ORs "too close to call" into `esc` (the debug build of tests/hostsim also records which test fired)
#ifdef R2IK_F32_DEBUG
static unsigned g_dbg_cause = 0;
#define R2IK_ESC(n, cond) do { if (cond) { esc = true; g_dbg_cause |= 1u << (n); } } while (0)
#else
#define R2IK_ESC(n, cond) esc = esc || (cond)
#endif
namespace r2ik {
namespace f32 {

// ArmConst narrowed to float (derived on the host from the FP64 constants, r2ik_create).
struct ArmConstF {
  float s[3];
  float L1, L2, L12, L1sq, L2sq;
  float wo[3], to[3];
  float max_arm_length, max_arm_length_sq;
  float d_min, proj_margin, backward_limit;
  float rLsq, hL;
  float Mst[9], Pst[3];
  float es0, es2, sing_coeff, sing_offset;
  float plP[3], plV[3], plC[3], plRho;
  float elbow_limit;
};

inline void narrow_constants(const ArmConst &A, ArmConstF &F) {
  for (int k = 0; k < 3; ++k) {
    F.s[k] = (float)A.s[k]; F.wo[k] = (float)A.wo[k]; F.to[k] = (float)A.to[k]; F.Pst[k] = (float)A.Pst[k];
    F.plP[k] = (float)A.plP[k]; F.plV[k] = (float)A.plV[k]; F.plC[k] = (float)A.plC[k];
  }
  for (int k = 0; k < 9; ++k) F.Mst[k] = (float)A.Mst[k];
  F.L1 = (float)A.L1; F.L2 = (float)A.L2; F.L12 = (float)A.L12; F.L1sq = (float)A.L1sq; F.L2sq = (float)A.L2sq;
  F.max_arm_length = (float)A.max_arm_length; F.max_arm_length_sq = (float)(A.max_arm_length * A.max_arm_length);
  F.d_min = (float)A.d_min; F.proj_margin = (float)A.proj_margin; F.backward_limit = (float)A.backward_limit;
  F.rLsq = (float)A.rLsq; F.hL = (float)A.hL;
  F.es0 = (float)A.es[0]; F.es2 = (float)A.es[2]; F.sing_coeff = (float)A.sing_coeff; F.sing_offset = (float)A.sing_offset;
  F.plRho = (float)A.plRho; F.elbow_limit = (float)A.elbow_limit;
}

// ---------------------------------------------------------------------------------------
// elementary functions: one MUFU each on the device
// ---------------------------------------------------------------------------------------
R2IK_HD float rsqrt_f(float x) {
#if defined(__CUDA_ARCH__)
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return 1.0f / sqrtf(x);
#endif
}
R2IK_HD float rcp_f(float x) {
#if defined(__CUDA_ARCH__)
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return 1.0f / x;
#endif
}
R2IK_HD float sqrt_f(float x) {
#if defined(__CUDA_ARCH__)
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return sqrtf(x);
#endif
}

constexpr float kPiF = 3.14159265358979323846f;
constexpr float kHalfPiF = 1.57079632679489661923f;
constexpr float kQuarterPiF = 0.78539816339744830962f;
constexpr float kTwoPiF = 6.28318530717958647692f;

// Error bands of the decisions, in units of the quantities compared (metres, cosines, radians).  They
// cover the accumulated FP32 rounding of the straight-line solve (a few 1e-7 on O(1) quantities) with a
// margin of ~10x; the measured share of escalated poses is reported by the tests / bench.
constexpr float kBandLen = 4e-6f;      // lengths and coordinates [m]
constexpr float kBandSin = 1e-5f;      // |sin| below which an angle sits on the +-pi / 0 branch cut
constexpr double kBandD2 = 4e-8;       // squared wrist distance [m^2] around the range / minimum-distance spheres
constexpr float kMinH2 = 4e-6f;        // squared length under an atan2 below which the angle is ill-conditioned (2 mm)
// The two angles whose lever collapses on ordinary poses -- shoulder pitch (the elbow near the pitch axis) and elbow
// yaw (a nearly straight arm: lever = forearm x sin(elbow pitch)) -- amplify the FP32 noise of the frame chain (a few
// 1e-6 m, measured) to more than 1e-4 rad well before 2 mm: they are handed to FP64 below 1.7 cm / 3.2 cm.  Host soak of
// 1.44 M reachable FK samples (profiles/r2_experiments.md): joints over 1e-4 rad 39 -> 5, max 4.8e-4 -> 1.4e-4,
// escalated 0.5 % -> 4.6 %.
constexpr float kMinH2ShoulderPitch = 3e-4f;
constexpr float kMinH2ElbowYaw = 1e-3f;
constexpr float kMinRadius2 = 1e-9f;   // elbow-circle radius^2 below which 1 / r is not trusted (0.03 mm)
constexpr float kMinLever2 = 1e-5f;    // (r rho sin alpha)^2 below which the interval ends are ill-conditioned (3 mm: interval error <= 2e-5 rad)

// atan2(s, c) of a UNIT vector (see angle_of_unit in r2ik_math.cuh): asin polynomial of 5 terms on
// |u| <= sin(pi/8), scripts/gen_atan_coeffs.py 0.3826834323650898 5 asin (max rel err 4.4e-9).
R2IK_HD float angle_of_unit_f(float c, float s) {
  const float ac = fabsf(c), as = fabsf(s);
  const bool swap = as > ac;
  const float mx = swap ? as : ac;
  const float mn = swap ? ac : as;
  const bool big = mn > 0.38268343236508978f;
  const float u = big ? (mn - mx) * 0.70710678118654752f : mn;
  const float v = u * u;
  float q = 0.04036556994867018f;
  q = fmaf(q, v, 0.04328442168484191f);
  q = fmaf(q, v, 0.07507298136377127f);
  q = fmaf(q, v, 0.16666531438030124f);
  float r = fmaf(u * v, q, u);
  if (big) r = kQuarterPiF + r;
  if (swap) r = kHalfPiF - r;
  if (c < 0.0f) r = kPiF - r;
  return copysignf(r, s);
}

// (cos a, sin a) and a = atan2(y, x).  esc: the vector is too short for the angle to be determined to
// 1e-4 from FP32 coordinates, or a sits on the +-pi branch cut.
R2IK_HD float cs_and_angle_f(float y, float x, float &c, float &s, bool &esc, float min_h2 = kMinH2) {
  const float h2 = x * x + y * y;
  const float ih = rsqrt_f(h2);
  c = x * ih; s = y * ih;
#ifdef R2IK_F32_DEBUG
  r2ik_f32_dbg(h2);
#endif
  R2IK_ESC(1, !(h2 > min_h2) || (c < 0.0f && fabsf(s) < kBandSin));
  return angle_of_unit_f(c, s);
}

// sin / cos for |x| up to a few turns: Cody-Waite reduction by pi/2 in three parts, cephes kernels.
R2IK_HD void sincos_f(float x, float &sn, float &cs) {
  const float kf = rintf(x * 0.63661977236758134308f);
  const int k = (int)kf;
  float r = fmaf(-kf, 1.5707962512969971f, x);      // pi/2 split: hi (24 bits)
  r = fmaf(-kf, 7.5497894158615964e-08f, r);        //             mid
  r = fmaf(-kf, 5.3903025299577648e-15f, r);        //             lo
  const float z = r * r;
  float ps = -1.9515295891e-4f;
  ps = fmaf(ps, z, 8.3321608736e-3f);
  ps = fmaf(ps, z, -1.6666654611e-1f);
  const float sr = fmaf(r * z, ps, r);
  float pc = 2.443315711809948e-5f;
  pc = fmaf(pc, z, -1.388731625493765e-3f);
  pc = fmaf(pc, z, 4.166664568298827e-2f);
  const float cr = fmaf(z * z, pc, fmaf(z, -0.5f, 1.0f));
  const float a = (k & 1) ? cr : sr;
  const float b = (k & 1) ? sr : cr;
  sn = (k & 2) ? -a : a;
  cs = ((k + 1) & 2) ? -b : b;
}

// ---------------------------------------------------------------------------------------
// solve state
// ---------------------------------------------------------------------------------------
struct SolveF {
  float p[3], R[9], w[3], c[3], r, a1[3], a2[3];
};
struct ReachF {
  int state;
  float i0, i1, c0, s0;
};

// Goal rotation from the 3x4 top of a row-major 4x4 (see rotation_from_mat4): an orthonormal,
// right-handed block away from the Euler gimbal band is used as it is; anything else is escalated.
R2IK_HD void rotation_from_mat4_f(const float m[12], float R[9], bool &esc) {
  const float r[9] = {m[0], m[1], m[2], m[4], m[5], m[6], m[8], m[9], m[10]};
  bool direct = true;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = i; j < 3; ++j) {
      const float g = r[3 * i] * r[3 * j] + r[3 * i + 1] * r[3 * j + 1] + r[3 * i + 2] * r[3 * j + 2];
      const float e = (i == j) ? 1.0f : 0.0f;
      if (!(fabsf(g - e) <= 2e-6f)) direct = false;
    }
  if (!(r[0] * r[0] + r[3] * r[3] > 1e-6f)) direct = false;   // cos^2(pitch): scipy's gimbal band, widened
  const float det = r[0] * (r[4] * r[8] - r[5] * r[7]) - r[1] * (r[3] * r[8] - r[5] * r[6]) + r[2] * (r[3] * r[7] - r[4] * r[6]);
  if (!(det > 0.5f)) direct = false;
  R2IK_ESC(2, !direct);
#pragma unroll
  for (int k = 0; k < 9; ++k) R[k] = r[k];
}

// R.from_euler("xyz", e).as_matrix() = Rz(e2) Ry(e1) Rx(e0)
// The six sines / cosines are taken in FP64 (the straight-line kernel of r2ik_math.cuh on the exactly widened angles) and
// the matrix is rounded once at the end: the FP32 construction carries ~2e-7 per element, which the near-straight-arm
// levers turn into 4e-4 rad (12 M host soak: 84 poses over 1e-4 with the FP32 matrix, against 18 for the same poses given
// as float matrices); this costs ~90 FP64 instructions on the euler layout only.
R2IK_HD void rot_from_euler_xyz_f(float e0, float e1, float e2, float R[9], bool &esc) {
  R2IK_ESC(3, !(fabsf(e0) <= 64.0f && fabsf(e1) <= 64.0f && fabsf(e2) <= 64.0f));
  double sx, cx, sy, cy, sz, cz;
  sincos_small((double)e0, sx, cx); sincos_small((double)e1, sy, cy); sincos_small((double)e2, sz, cz);
  R[0] = (float)(cz * cy); R[1] = (float)(cz * sy * sx - sz * cx); R[2] = (float)(cz * sy * cx + sz * sx);
  R[3] = (float)(sz * cy); R[4] = (float)(sz * sy * sx + cz * cx); R[5] = (float)(sz * sy * cx - cz * sx);
  R[6] = (float)(-sy);     R[7] = (float)(cy * sx);                R[8] = (float)(cy * cx);
}

R2IK_HD void wrist_from_goal_f(const ArmConstF &A, const float p[3], const float R[9], float w[3]) {
  w[0] = R[0] * A.wo[0] + R[1] * A.wo[1] + R[2] * A.wo[2] + p[0];
  w[1] = R[3] * A.wo[0] + R[4] * A.wo[1] + R[5] * A.wo[2] + p[1];
  w[2] = R[6] * A.wo[0] + R[7] * A.wo[1] + R[8] * A.wo[2] + p[2];
}

// utl:59-81 columns of rotation_matrix_from_vector for a UNIT vector u.  (1 - ux) / (uy^2 + uz^2) is
// taken as 1 / (1 + ux): the same number for a unit vector, without the cancellation.
R2IK_HD void rmfv_columns_f(float ux, float uy, float uz, float c0[3], float a1[3], float a2[3], bool &esc) {
  R2IK_ESC(4, (fabsf(uy) < 3e-5f && fabsf(uz) < 3e-5f));   // the isclose special cases (u = +-e_x)
  const float f = rcp_f(1.0f + ux);
  c0[0] = ux; c0[1] = uy; c0[2] = uz;
  a1[0] = -uy; a1[1] = 1.0f - (uy * uy) * f; a1[2] = -(uy * uz) * f;
  a2[0] = -uz; a2[1] = -(uy * uz) * f;        a2[2] = 1.0f - (uz * uz) * f;
}

// sik:121-282 is_reachable on a goal position + goal rotation (S.R set by the caller).
//
// Mixed precision front end.  The wrist centre, its distance to the shoulder and the radicand of the
// elbow-circle radius are differences of nearly equal O(0.5 m) quantities whenever the arm is close to
// straight (4 d^2 L1^2 - k^2 -> 0 as d -> L1 + L2): in FP32 their rounding alone moves elbow yaw / wrist
// yaw by > 1e-4 rad for elbow pitches below ~0.2 rad.  These ~25 operations are therefore done in FP64
// on the exactly-widened FP32 inputs (A64 = the FP64 constants) -- which also makes the reach / range
// decisions of sik:284-307, 146-171 exact instead of banded -- and everything downstream (frames, circle
// linking, angles, get_joints) runs in FP32 on the narrowed results.
R2IK_HD ReachF is_reachable_f(const ArmConst &A64, const ArmConstF &A, float pxf, float pyf, float pzf, SolveF &S, bool &esc) {
  ReachF out;
  out.i0 = NAN; out.i1 = NAN; out.c0 = NAN; out.s0 = NAN;
  double p[3] = {(double)pxf, (double)pyf, (double)pzf};
  // --- sik:284-307 reach pre-checks
  {
    const double dx = p[0] - A64.s[0], dy = p[1] - A64.s[1], dz = p[2] - A64.s[2];
    const double dg2 = dx * dx + dy * dy + dz * dz, Lm2 = A64.max_arm_length * A64.max_arm_length;
    R2IK_ESC(5, fabs(dg2 - Lm2) <= 1e-12);
    int pre = -1;
    if (dg2 > Lm2) {
      // the projected x decides between "Pose out of reach" and "Backward pose"
      const float sc = A.max_arm_length * rsqrt_f((float)dg2);
      const float pxp = A.s[0] + (float)dx * sc;
      R2IK_ESC(6, fabsf(pxp - A.backward_limit) < kBandLen);
      pre = R2IK_STATE_POSE_OUT_OF_REACH;
      if (pxp < A.backward_limit) pre = R2IK_STATE_BACKWARD_POSE;
    } else if (p[0] < A64.backward_limit) {
      // inside the sphere the goal itself is tested (sik:303); outside, only its projection is (a backward_limit
      // behind the shoulder can admit the projection of a goal that lies behind it)
      pre = R2IK_STATE_BACKWARD_POSE;
    }
    if (pre >= 0) { out.state = pre; return out; }
  }
  // --- sik:418-425 wrist centre, sik:146-153 kept in front of the torso plane
  double w[3];
#pragma unroll
  for (int k = 0; k < 3; ++k)
    w[k] = (double)S.R[3 * k] * A64.wo[0] + (double)S.R[3 * k + 1] * A64.wo[1] + (double)S.R[3 * k + 2] * A64.wo[2] + p[k];
  if (w[0] < A64.backward_limit) {
    const double diff = A64.backward_limit - w[0];
    p[0] += diff; w[0] += diff;
  }
  double P[3] = {w[0] - A64.s[0], w[1] - A64.s[1], w[2] - A64.s[2]};
  double d2 = P[0] * P[0] + P[1] * P[1] + P[2] * P[2];
  // The FP64 arithmetic above is exact on its inputs, but the rotation is the FP32 one: it differs from the FP64 solver's
  // (polar factor of the same float matrix / euler angles in double) by ~6e-8 per element, i.e. ~1e-8 m in the wrist
  // centre and ~2e-8 in d^2.  A wrist within that of the range sphere or of the minimum-distance sphere (a fully
  // stretched or fully folded arm: FK samples with elbow pitch < 1e-3 rad) is decided by the FP64 solver.
  R2IK_ESC(23, fabs(d2 - A64.L12 * A64.L12) < kBandD2 || fabs(d2 - A64.d_min * A64.d_min) < kBandD2);
  if (d2 > A64.L12 * A64.L12) { out.state = R2IK_STATE_WRIST_OUT_OF_RANGE; return out; }
  if (d2 < A64.d_min * A64.d_min) {
    // sik:166-171, 337-349: wrist pushed out radially to d_min, the goal follows, the wrist is recomputed
    double invd64;
    const double d = sqrt_rsqrt_nonneg(d2, invd64);
    R2IK_ESC(7, !(d2 > 1e-12));
    const double sc = div_fast(A64.d_min, d + A64.proj_margin);
#pragma unroll
    for (int k = 0; k < 3; ++k) p[k] += (A64.s[k] + P[k] * sc) - w[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      w[k] = (double)S.R[3 * k] * A64.wo[0] + (double)S.R[3 * k + 1] * A64.wo[1] + (double)S.R[3 * k + 2] * A64.wo[2] + p[k];
      P[k] = w[k] - A64.s[k];
    }
    d2 = P[0] * P[0] + P[1] * P[1] + P[2] * P[2];
  }
  // --- sik:366-399 elbow circle: radicand and centre offset in FP64, then narrowed
  const double kk = d2 - A64.L2sq + A64.L1sq;
  const double rad = 4.0 * d2 * A64.L1sq - kk * kk;
  const float invd = rsqrt_f((float)d2);
  const float inv2d = 0.5f * invd;
  const float radf = (float)rad;
  R2IK_ESC(8, !(radf * inv2d * inv2d > kMinRadius2));
  S.r = sqrt_f(fmaxf(radf, 0.0f)) * inv2d;
  const float cd = (float)kk * inv2d;
  const float n2[3] = {(float)P[0] * invd, (float)P[1] * invd, (float)P[2] * invd};
#pragma unroll
  for (int k = 0; k < 3; ++k) { S.p[k] = (float)p[k]; S.w[k] = (float)w[k]; S.c[k] = n2[k] * cd + A.s[k]; }
  float c0[3];
  rmfv_columns_f(n2[0], n2[1], n2[2], c0, S.a1, S.a2, esc);

  // --- sik:401-416 wrist-limit circle and sik:427-568 circle linking, in the plane of the elbow circle.
  // Both circles lie on the forearm sphere (centre w, radius L2), so the points where the reference's
  // plane-plane line meets the limit circle (sik:588-645) ARE the points of the elbow circle that lie in
  // the limit plane n1 . (X - p1) = 0.  With X(theta) = p2 + r (a1 cos theta + a2 sin theta) the signed
  // x of X in the limitation frame -- the reference's mid-arc test quantity, sik:541-558 -- is
  //     xl(theta) = Xc + r (A cos theta + B sin theta) = Xc + r rho cos(theta - phi),
  //     A = n1 . a1, B = n1 . a2, rho = |n1 x n2|, Xc = n1 . (p2 - p1)   (sik:466-467),
  // so the intersection angles are phi -+ acos(kappa), kappa = -Xc / (r rho), the reference's
  // discriminant test is |kappa| <= 1, and its sort + mid-arc test selects the arc on which xl > 0: the
  // interval runs counter-clockwise from phi - alpha to phi + alpha.  Unlike the 3-D construction
  // (whose point coordinates carry ~1e-7 m of FP32 rounding against a circle of radius r: 1e-4 rad at
  // r = 1 cm) this form only divides the well-conditioned scalar Xc by r rho.
  const float nLx = (float)(w[0] - p[0]), nLy = (float)(w[1] - p[1]), nLz = (float)(w[2] - p[2]);
  const float inL = rsqrt_f(nLx * nLx + nLy * nLy + nLz * nLz);
  const float n1[3] = {nLx * inL, nLy * inL, nLz * inL};
  R2IK_ESC(9, (fabsf(n1[1]) < 3e-5f && fabsf(n1[2]) < 3e-5f));   // rmfv(n1) special cases (sik:455)
  // c - w = n2 (k / 2d - d) = n2 (k - 2 d^2) / 2d: the difference is taken in FP64
  const float cdw = (float)(kk - 2.0 * d2) * inv2d;
  const float Ca = n1[0] * n2[0] + n1[1] * n2[1] + n1[2] * n2[2];
  const float Aa = n1[0] * S.a1[0] + n1[1] * S.a1[1] + n1[2] * S.a1[2];
  const float Ba = n1[0] * S.a2[0] + n1[1] * S.a2[1] + n1[2] * S.a2[2];
  const float rho2 = Aa * Aa + Ba * Ba;
  R2IK_ESC(10, !(rho2 > 1e-6f));                                   // sik:475-483 parallel planes (and close to it)
  const float irho = rsqrt_f(rho2);
  const float Xc = cdw * Ca - A.hL;                               // n1 . (p2 - p1), |n1| = 1
  {
    // sik:570-586 the reference gives up when its two line parameters are np.isclose
    const float t = (cdw - A.hL * Ca) * irho, u = Xc * irho;
    R2IK_ESC(11, fabsf(u - t) <= 4.0f * (1e-8f + 1e-5f * fabsf(t)) + kBandLen);
  }
  const float kappa = -Xc * irho * rcp_f(S.r);
  const float sp2 = (1.0f - kappa) * (1.0f + kappa);
  // conditioning of theta: d(theta) = d(Xc) / (r rho sin(alpha)); also covers |kappa| ~ 1 (the discriminant sign)
  R2IK_ESC(12, fabsf(sp2) * (S.r * S.r * rho2) < kMinLever2);
  if (!(sp2 >= 0.0f)) {
    if (Xc > 0.0f) { out.state = R2IK_STATE_REACHABLE; out.i0 = -kPiF; out.i1 = kPiF; out.c0 = -1.0f; out.s0 = -0.0f; }
    else out.state = R2IK_STATE_LIMITED_BY_WRIST;
    return out;
  }
  const float sp = sqrt_f(sp2);
  const float cph = Aa * irho, sph = Ba * irho;
  const float c_lo = cph * kappa + sph * sp, s_lo = sph * kappa - cph * sp;   // phi - alpha
  const float c_hi = cph * kappa - sph * sp, s_hi = sph * kappa + cph * sp;   // phi + alpha
  R2IK_ESC(13, (c_lo < 0.0f && fabsf(s_lo) < kBandSin) || (c_hi < 0.0f && fabsf(s_hi) < kBandSin));
  out.state = R2IK_STATE_REACHABLE;
  out.i0 = angle_of_unit_f(c_lo, s_lo);
  out.i1 = angle_of_unit_f(c_hi, s_hi);
  out.c0 = c_lo; out.s0 = s_lo;
  return out;
}

struct P3f { float x, y, z; };
R2IK_HD void rot_y_f(P3f &p, float c, float s) { const float x = c * p.x + s * p.z, z = -s * p.x + c * p.z; p.x = x; p.z = z; }
R2IK_HD void rot_z_f(P3f &p, float c, float s) { const float x = c * p.x - s * p.y, y = s * p.x + c * p.y; p.x = x; p.y = y; }
R2IK_HD void rot_x_f(P3f &p, float c, float s) { const float y = c * p.y - s * p.z, z = s * p.y + c * p.z; p.y = y; p.z = z; }
R2IK_HD P3f to_shoulder_f(const ArmConstF &A, const float X[3]) {
  P3f o;
  o.x = A.Mst[0] * X[0] + A.Mst[1] * X[1] + A.Mst[2] * X[2] + A.Pst[0];
  o.y = A.Mst[3] * X[0] + A.Mst[4] * X[1] + A.Mst[5] * X[2] + A.Pst[1];
  o.z = A.Mst[6] * X[0] + A.Mst[7] * X[1] + A.Mst[8] * X[2] + A.Pst[2];
  return o;
}

// sik:697-863 get_joints from (cos theta, sin theta); see get_joints_impl for the frame chain.
R2IK_HD void get_joints_f(const ArmConstF &A, SolveF &S, float ct, float st, float joints[7], float E[3], bool &esc) {
  const float y = S.r * ct, z = S.r * st;
#pragma unroll
  for (int k = 0; k < 3; ++k) E[k] = S.a1[k] * y + S.a2[k] * z + S.c[k];
  const float plane = E[2] - ((E[0] - A.es0) * A.sing_coeff + A.es2 - A.sing_offset);
  R2IK_ESC(14, fabsf(plane) < kBandLen);
  if (plane > 0.0f) {
    // sik:647-682 make_elbow_projection
    const float dist = (E[0] - A.plP[0]) * A.plV[0] + (E[1] - A.plP[1]) * A.plV[1] + (E[2] - A.plP[2]) * A.plV[2];
    const float vc[3] = {E[0] - dist * A.plV[0] - A.plC[0], E[1] - dist * A.plV[1] - A.plC[1], E[2] - dist * A.plV[2] - A.plC[2]};
    const float v2 = vc[0] * vc[0] + vc[1] * vc[1] + vc[2] * vc[2];
    R2IK_ESC(15, !(v2 > kMinH2));
    const float sc = A.plRho * rsqrt_f(v2);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float ne = A.plC[k] + vc[k] * sc;
      S.p[k] += ne - E[k];
      E[k] = ne;
    }
    wrist_from_goal_f(A, S.p, S.R, S.w);
  }
  const float tipw[3] = {S.R[0] * A.to[0] + S.R[1] * A.to[1] + S.R[2] * A.to[2] + S.p[0],
                         S.R[3] * A.to[0] + S.R[4] * A.to[1] + S.R[5] * A.to[2] + S.p[1],
                         S.R[6] * A.to[0] + S.R[7] * A.to[1] + S.R[8] * A.to[2] + S.p[2]};
  const float ptw[3] = {S.R[0] * 0.1f + tipw[0], S.R[3] * 0.1f + tipw[1], S.R[6] * 0.1f + tipw[2]};
  P3f el = to_shoulder_f(A, E), wr = to_shoulder_f(A, S.w), tp = to_shoulder_f(A, tipw), pt = to_shoulder_f(A, ptw);
  float s, c, at[7];
  at[0] = cs_and_angle_f(el.z, el.x, c, s, esc, kMinH2ShoulderPitch);  // sik:751-758
  rot_y_f(el, c, s); rot_y_f(wr, c, s); rot_y_f(tp, c, s); rot_y_f(pt, c, s);
  at[1] = -cs_and_angle_f(-el.y, el.x, c, s, esc);                     // sik:766-769
  rot_z_f(wr, c, s); rot_z_f(tp, c, s); rot_z_f(pt, c, s);
  wr.x -= A.L1; tp.x -= A.L1; pt.x -= A.L1;
  {
    float ca, sa;
    at[2] = cs_and_angle_f(wr.z, -wr.y, ca, sa, esc, kMinH2ElbowYaw);  // sik:782-789
    c = sa; s = -ca;
  }
  rot_x_f(wr, c, s); rot_x_f(tp, c, s); rot_x_f(pt, c, s);
  at[3] = cs_and_angle_f(wr.z, wr.x, c, s, esc);                       // sik:797-800
  rot_y_f(tp, c, s); rot_y_f(pt, c, s);
  tp.x -= A.L2; pt.x -= A.L2;
  {
    float ca, sa;
    at[4] = cs_and_angle_f(tp.y, -tp.x, ca, sa, esc);                  // sik:815-820
    R2IK_ESC(16, (ca > 0.0f && fabsf(sa) < kBandSin));                  // wrist_roll = pi - a wraps at a = 0
    c = -ca; s = -sa;
  }
  rot_z_f(tp, c, s); rot_z_f(pt, c, s);
  at[5] = cs_and_angle_f(tp.z, tp.x, c, s, esc);                       // sik:826-829
  rot_y_f(pt, c, s);
  {
    float ca, sa;
    at[6] = cs_and_angle_f(pt.y, pt.z, ca, sa, esc);                   // sik:848
  }
  joints[0] = -at[0];
  joints[1] = at[1];
  joints[2] = -kHalfPiF + at[2];
  float ep = -at[3];
  ep = fminf(A.elbow_limit, fmaxf(-A.elbow_limit, ep));                // sik:853-861
  joints[3] = ep;
  float wrist_roll = kPiF - at[4];
  if (wrist_roll > kPiF) wrist_roll -= kTwoPiF;
  joints[4] = wrist_roll;
  joints[5] = -at[5];
  joints[6] = at[6];
}

// ---------------------------------------------------------------------------------------
// Flag-only solve for the workspace reachability map (K4): is (voxel centre p, orientation o) reachable?
//
// What depends on the orientation alone is hoisted into OriConst: wv = R wo (so that the wrist is p + wv: 3 adds instead
// of a 3x3 product per pair) and the limit-plane normal n1 = (w - p) / |w - p| = wv / |wo| (no normalisation per pair).
// Per pair, the cancelling front end (wrist, distance, radicand) runs in FP64 -- ~15 operations -- and the in-plane
// linking test sign(r^2 rho^2 - Xc^2) in FP32, with the same error bands as the K1 fast path; a pair that is too
// close to call is decided by the FP64 solver (solve_core<false, true>), so the COUNTS are those of the FP64 path.
// ---------------------------------------------------------------------------------------
struct OriConst {
  double wv[3];   // R wo
  float n1[3];    // wv / |wv|
  int special;    // rotation_matrix_from_vector(n1) would take one of its isclose special cases: always escalate
};

R2IK_HD OriConst make_ori_const(const ArmConst &A, const double R[9]) {
  OriConst O;
  for (int k = 0; k < 3; ++k) O.wv[k] = R[3 * k] * A.wo[0] + R[3 * k + 1] * A.wo[1] + R[3 * k + 2] * A.wo[2];
  const double n = sqrt(O.wv[0] * O.wv[0] + O.wv[1] * O.wv[1] + O.wv[2] * O.wv[2]);
  for (int k = 0; k < 3; ++k) O.n1[k] = (float)(O.wv[k] / n);
  O.special = !(n > 1e-6) || (fabsf(O.n1[1]) < 3e-5f && fabsf(O.n1[2]) < 3e-5f);
  return O;
}

// ps = p - s (FP64, p already through the reach pre-checks), px = p.x.  Returns the state; esc: decide in FP64 instead.
R2IK_HD int reach_flag_mixed(const ArmConst &A64, const ArmConstF &A, const double ps[3], double px, const OriConst &O, bool &esc) {
  esc = O.special != 0;
  double P[3] = {ps[0] + O.wv[0], ps[1] + O.wv[1], ps[2] + O.wv[2]};
  const double wx = px + O.wv[0];
  if (wx < A64.backward_limit) P[0] += A64.backward_limit - wx;          // sik:146-153: p and w move together
  double d2 = P[0] * P[0] + P[1] * P[1] + P[2] * P[2];
  if (d2 > A64.L12 * A64.L12) return R2IK_STATE_WRIST_OUT_OF_RANGE;
  if (d2 < A64.d_min * A64.d_min) {
    // sik:166-171, 337-349: the wrist is pushed out radially to d_min d / (d + margin), the goal follows and the wrist is
    // recomputed from it: P scales by sc (the recomputed wrist is the pushed one up to rounding)
    double invd64;
    const double d = sqrt_rsqrt_nonneg(d2, invd64);
    esc = esc || !(d2 > 1e-12);
    const double sc = div_fast(A64.d_min, d + A64.proj_margin);
    P[0] *= sc; P[1] *= sc; P[2] *= sc;
    d2 = P[0] * P[0] + P[1] * P[1] + P[2] * P[2];
  }
  const double kk = d2 - A64.L2sq + A64.L1sq;
  const double rad = 4.0 * d2 * A64.L1sq - kk * kk;
  const float invd = rsqrt_f((float)d2);
  const float inv2d = 0.5f * invd;
  const float r2 = (float)rad * inv2d * inv2d;
  R2IK_ESC(18, !(r2 > kMinRadius2));
  const float n2[3] = {(float)P[0] * invd, (float)P[1] * invd, (float)P[2] * invd};
  const float Ca = O.n1[0] * n2[0] + O.n1[1] * n2[1] + O.n1[2] * n2[2];
  const float rho2 = fmaf(-Ca, Ca, 1.0f);
  R2IK_ESC(19, !(rho2 > 1e-4f));                                   // (nearly) parallel planes, and the cancellation in 1 - Ca^2
  const float cdw = (float)(kk - 2.0 * d2) * inv2d;                // |c - w| with sign: c - w = n2 cdw
  const float Xc = cdw * Ca - A.hL, nb = cdw - A.hL * Ca;
  R2IK_ESC(20, fabsf(Xc - nb) <= 4.0f * (1e-8f + 1e-5f * fabsf(nb)) + kBandLen);   // np.isclose(u, t), sik:581
  const float rr = r2 * rho2, xx = Xc * Xc;
  const float dl = rr - xx;
  // error of dl: rho2 = 1 - Ca^2 carries the absolute rounding of Ca (~2e-7, relative 1e-4 at 3 degrees between the
  // planes), Xc that of cdw Ca (~5e-8): r2 d(rho2) + 2 |Xc| d(Xc), plus the relative rounding of the products
  R2IK_ESC(21, fabsf(dl) <= 1e-5f * (rr + xx) + 1.5e-6f * r2 + 4e-7f * fabsf(Xc));
  if (dl < 0.0f) {
    R2IK_ESC(22, fabsf(Xc) < kBandLen);
    return Xc > 0.0f ? R2IK_STATE_REACHABLE : R2IK_STATE_LIMITED_BY_WRIST;
  }
  return R2IK_STATE_REACHABLE;
}

// The state of one (voxel p, orientation) pair: reach_flag_mixed, and where it is too close to call in FP32 (esc) the
// FP64 flag solve on the orientation's xyz Euler angles e.
R2IK_HD int reach_pair(const ArmConst &A64, const ArmConstF &A, const double ps[3], double px, double py, double pz,
                       const OriConst &O, const double *e, bool &esc) {
  int st = reach_flag_mixed(A64, A, ps, px, O, esc);
  if (esc) {
    Solve S;
    S.p[0] = px; S.p[1] = py; S.p[2] = pz;
    rot_from_euler_xyz(e[0], e[1], e[2], S.R);
    st = solve_core<false, true>(A64, S).state;
  }
  return st;
}

// ---------------------------------------------------------------------------------------
// per-pose bodies of K1-f32
// ---------------------------------------------------------------------------------------
// out[12] = theta interval (2), joints (7), elbow (3); NaN when unreachable.
// in[]: KIND == R2IK_POSE_MAT4: the 3x4 top of the row-major 4x4 (12 floats); EULER6: x y z roll pitch yaw.
// Returns true when the pose must be solved again in FP64 (state / out are then meaningless).
template <int KIND>
R2IK_HD bool symik_pose_fast(const ArmConst &A64, const ArmConstF &A, const float *in, bool has_theta, float theta, int &state, float out[12]) {
  bool esc = false;
  SolveF S;
  float px, py, pz;
  if (KIND == R2IK_POSE_EULER6) {
    px = in[0]; py = in[1]; pz = in[2];
    rot_from_euler_xyz_f(in[3], in[4], in[5], S.R, esc);
  } else {
    px = in[3]; py = in[7]; pz = in[11];
    rotation_from_mat4_f(in, S.R, esc);
  }
  ReachF rc = is_reachable_f(A64, A, px, py, pz, S, esc);
  state = rc.state;
  out[0] = rc.i0; out[1] = rc.i1;
  if (rc.state == R2IK_STATE_REACHABLE) {
    float ct = rc.c0, st = rc.s0;
    if (has_theta) {
      R2IK_ESC(17, !(fabsf(theta) <= 64.0f));
      sincos_f(theta, st, ct);
    }
    get_joints_f(A, S, ct, st, out + 2, out + 9, esc);
  } else {
#pragma unroll
    for (int k = 2; k < 12; ++k) out[k] = NAN;
  }
  return esc;
}

// The escalation target: the FP64 solver on the same inputs widened to double, results narrowed
// (body of k_symik_escalated_f32; a few poses in 10^3 take it).
template <int KIND>
R2IK_HD void symik_pose_escalated(const ArmConst &A, const float *in, bool has_theta, float theta, float prev0, float prev2,
                          int *state, float *out) {
  double pos[3];
  Solve S;
  bool valid = true;
  if (KIND == R2IK_POSE_EULER6) {
    pos[0] = in[0]; pos[1] = in[1]; pos[2] = in[2];
    rot_from_euler_xyz((double)in[3], (double)in[4], (double)in[5], S.R);
  } else {
    double m[16];
    for (int k = 0; k < 12; ++k) m[k] = (double)in[k];
    m[12] = 0.0; m[13] = 0.0; m[14] = 0.0; m[15] = 1.0;
    pos[0] = m[3]; pos[1] = m[7]; pos[2] = m[11];
    valid = rotation_from_mat4(m, false, S.R);
  }
  Reach rc;
  if (valid) rc = is_reachable_R<false>(A, pos, S);
  else { rc.state = R2IK_STATE_INVALID_ROTATION; rc.i0 = NAN; rc.i1 = NAN; }
  *state = rc.state;
  out[0] = (float)rc.i0; out[1] = (float)rc.i1;
  if (rc.state == R2IK_STATE_REACHABLE) {
    double ct = rc.c0, st = rc.s0, j[7], E[3];
    if (has_theta) sincos_any((double)theta, st, ct);
    get_joints_cs(A, S, ct, st, (double)prev0, (double)prev2, j, E);
    for (int k = 0; k < 7; ++k) out[2 + k] = (float)j[k];
    for (int k = 0; k < 3; ++k) out[9 + k] = (float)E[k];
  } else {
    for (int k = 2; k < 12; ++k) out[k] = NAN;
  }
}

}  // namespace f32
}  // namespace r2ik
