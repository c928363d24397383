// r2ik_control.cuh -- ControlIK policies on top of the per-pose solver: elbow-angle selection
// (discrete search / rate-limited continuous tracking), (re)initialisation by ternary search,
// and the safety chain (Orbita3D wrist cone, multi-turn unwrap, +-6pi clamp, continuity check).
// "ctl" = src/reachy2_symbolic_ik/control_ik.py, "utl" = .../utils.py.
#pragma once

#include "r2ik_device.cuh"

namespace r2ik {

// is_elbow_ok(get_elbow_position(theta)) (utl:443-465 on sik:684-695) as two half-plane tests in
// (cos theta, sin theta): the elbow point is c + a1 r cos + a2 r sin, and both conditions of the
// predicate are linear in it:
//   E.y side < -0.2                                   <=>  C1 + A1 cos + B1 sin < 0
//   E.z < (E.x - es.x) coeff + es.z - offset          <=>  C2 + A2 cos + B2 sin < 0
// Hoisting the six coefficients out of the K-sample loop leaves 4 FMA + 2 compares per sample
// (algebraically the same predicate; it can differ from the literal evaluation only for an elbow
// within rounding of a limit plane).
struct ElbowTest { double A1, B1, C1, A2, B2, C2; };

R2IK_HD ElbowTest make_elbow_test(const ArmConst &A, const Solve &S) {
  ElbowTest T;
  T.A1 = A.side * S.a1[1] * S.r;
  T.B1 = A.side * S.a2[1] * S.r;
  T.C1 = A.side * S.c[1] + 0.2;
  T.A2 = (S.a1[2] - A.sing_coeff * S.a1[0]) * S.r;
  T.B2 = (S.a2[2] - A.sing_coeff * S.a2[0]) * S.r;
  T.C2 = (S.c[2] - A.sing_coeff * S.c[0]) + (A.sing_coeff * A.es[0] - A.es[2] + A.sing_offset);
  return T;
}
R2IK_HD bool elbow_ok_cs(const ElbowTest &T, double c, double s) {
  return (T.C1 + T.A1 * c + T.B1 * s < 0.0) && (T.C2 + T.A2 * c + T.B2 * s < 0.0);
}

// The K samples of the search (utl:366-390) for one pose: theta_k = linspace(start, stop, K)[k].
// cos / sin of the samples a thread visits (k0, k0 + stride, ...) follow from one sincos and a
// fixed rotation by stride * step per sample instead of a sincos each.
struct SearchPlan {
  Linspace L;
  ElbowTest T;
  double preferred_theta;
};

// Lowest cost among samples k0, k0 + stride, ... < nb (strict <: the first minimum wins, utl:386).
R2IK_HD void search_strided(const SearchPlan &P, int nb, int k0, int stride, double &best, int &best_k) {
  best = INFINITY;
  best_k = 0x7fffffff;
  if (k0 >= nb) return;
  double c, s, cd, sd;
  const double th0 = linspace_value(P.L, k0), dth = (double)stride * P.L.step;
  sincos_any(th0, s, c);
  sincos_any(dth, sd, cd);
  for (int k = k0; k < nb; k += stride) {
    if (elbow_ok_cs(P.T, c, s)) {
      double cost = fabs(angle_diff(linspace_value(P.L, k), P.preferred_theta));
      if (cost < best) { best = cost; best_k = k; }
    }
    double cn = c * cd - s * sd;
    s = s * cd + c * sd;
    c = cn;
  }
}

// The same arg-min WITHOUT visiting the K samples.  On the sampled range (an interval of theta of length
// <= 2 pi) the cost |angle_diff(theta, preferred)| falls linearly to 0 at the point congruent to the
// preferred theta and rises to pi at its antipode, and each half-plane test C + A cos + B sin < 0 holds on
// one arc of the circle (phi + acos(g), phi + 2 pi - acos(g)), g = -C / hypot(A, B), phi = atan2(B, A).
// The valid samples therefore form a few runs of consecutive indices, and on a run the cheapest sample is
// either next to the preferred point or at an end of the run -- i.e. next to a crossing of one of the two
// tests or at an end of the range.  Candidates: the 3 samples around each of the <= 4 crossings, the 3
// around the preferred point, the first and the last sample; each is evaluated like a visited sample
// (theta_k from linspace, its cos / sin, the two tests, the wrapped cost) and the minimum is taken in
// (cost, index) order = the reference's strict-< scan.  17 evaluations instead of K, no cooperation
// between lanes.  Returns false when an atan2 argument is outside the fast routine's range (the caller
// scans instead).
R2IK_HD void search_eval_cs(const SearchPlan &P, int nb, int k, double c, double s, double &best, int &best_k) {
  if (k < 0 || k >= nb) return;
  if (!elbow_ok_cs(P.T, c, s)) return;
  const double cost = fabs(angle_diff(linspace_value(P.L, k), P.preferred_theta));
  if (cost < best || (cost == best && k < best_k)) { best = cost; best_k = k; }
}
R2IK_HD bool search_analytic(const SearchPlan &P, int nb, double &best, int &best_k) {
  best = INFINITY;
  best_k = 0x7fffffff;
  if (!(P.L.step > 0.0) || nb < 8) {                     // degenerate range or a handful of samples: just scan
    double b; int bk;
    search_strided(P, nb, 0, 1, b, bk);
    best = b; best_k = bk;
    return true;
  }
  const double inv_step = 1.0 / P.L.step;
  bool ok = true;
  // angles whose neighbouring samples are candidates: the crossings phi +- alpha of each test, the preferred theta
  // (NaN = no such crossing; its candidates are skipped)
  double cand[5];
  const double A_[2] = {P.T.A1, P.T.A2}, B_[2] = {P.T.B1, P.T.B2}, C_[2] = {P.T.C1, P.T.C2};
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const double R2 = A_[t] * A_[t] + B_[t] * B_[t];
    const double s2 = R2 - C_[t] * C_[t];                // R^2 sin^2(alpha): < 0 => the test never changes sign
    const bool cross = s2 >= 0.0;
    ok = ok && (!cross || (atan2_core_ok(B_[t], A_[t]) && (R2 > 1e-280)));
    const double phi = atan2_core(B_[t], A_[t]);
    const double alpha = atan2_core(sqrt_nonneg(cross ? s2 : 0.0), -C_[t]);   // acos(-C / R)
    cand[2 * t] = cross ? phi + alpha : NAN;
    cand[2 * t + 1] = cross ? phi - alpha : NAN;
  }
  cand[4] = P.preferred_theta;
  // cos / sin of a candidate's two neighbours follow from its own by the fixed rotation of one sample step -- the way
  // search_strided walks the samples -- so the 17 evaluations take 7 sincos (+ 1 for the step).  One copy of the body
  // in the instruction stream (unrolled the kernel no longer fits the instruction cache).
  double sd, cd;
  sincos_any(P.L.step, sd, cd);
#pragma unroll 1
  for (int g = 0; g < 7; ++g) {
    int k;
    if (g < 5) {
      // sample position of the angle congruent to the candidate in [start, start + 2 pi)
      // (+ 4 pi keeps the argument inside pymod_2pi's exact fast range; the candidate index tolerates the rounding)
      const double x = pymod_2pi((cand[g] - P.L.start) + 2.0 * kTwoPi) * inv_step;
      if (!(x <= (double)nb)) continue;                  // NaN, or beyond the last sample (ranges shorter than 2 pi)
      k = (int)rint(x);
      if (k >= nb) k = nb - 1;                           // x rounded up past the last sample: its neighbourhood is the range's end
    } else {
      k = g == 5 ? 0 : nb - 1;
    }
    double s, c;
    sincos_any(linspace_value(P.L, k), s, c);
    search_eval_cs(P, nb, k, c, s, best, best_k);
    if (g < 5) {
      search_eval_cs(P, nb, k - 1, c * cd + s * sd, s * cd - c * sd, best, best_k);
      search_eval_cs(P, nb, k + 1, c * cd - s * sd, s * cd + c * sd, best, best_k);
    }
  }
  return ok;
}

// utl:357-364: preferred_theta is tried first
R2IK_HD bool preferred_theta_works(const ArmConst &A, const Solve &S, double i0, double i1, double preferred_theta) {
  if (!is_valid_angle(preferred_theta, i0, i1)) return false;
  double E[3];
  elbow_position(S, preferred_theta, E);
  return is_elbow_ok(A, E);
}

// utl:334-396 get_best_discrete_theta, serial form (one thread scans all samples; strict <
// keeps the first minimum).  Returns false when no sample is valid.
R2IK_HD bool best_discrete_theta(const ArmConst &A, const Solve &S, double i0, double i1, int nb,
                                 double preferred_theta, double &theta) {
  if (preferred_theta_works(A, S, i0, i1, preferred_theta)) { theta = preferred_theta; return true; }
  double start, stop;
  search_range(i0, i1, start, stop);
  SearchPlan P;
  P.L = make_linspace(start, stop, nb);
  P.T = make_elbow_test(A, S);
  P.preferred_theta = preferred_theta;
  double best;
  int best_k;
  search_strided(P, nb, 0, 1, best, best_k);
  if (!(best < INFINITY)) { theta = 0.0; return false; }
  theta = linspace_value(P.L, best_k);
  return true;
}

// Step toward a target theta by at most d_theta_max (utl:252-264, utl:123-127)
R2IK_HD double step_toward(double target, double previous_theta, double d_theta_max) {
  double ad = angle_diff(target, previous_theta);
  if (fabs(ad) < d_theta_max) return target;
  // ad / fabs(ad) of the reference is exactly +-1 (0 / 0 = nan when d_theta_max <= 0 lets ad = 0 through): no division
  const double sign = ad == 0.0 ? NAN : copysign(1.0, ad);
  return previous_theta + sign * d_theta_max;
}

// ctl:464-497 safety_checks after the (stateless) Orbita3D limit: multi-turn unwrap against the previous
// solution and the +-6 pi clamp.  Returns the emergency bits raised by multiturn_safety_check.
R2IK_HD int safety_multiturn(double j[7], const double previous_sol[7]) {
  for (int i = 0; i < 7; ++i)                               // utl:493-505 allow_multiturn
    j[i] = previous_sol[i] + angle_diff(j[i], previous_sol[i]);
  int bits = 0;                                             // utl:535-568
  const double lim = 6.0 * kPi;
  if (j[0] > lim) { j[0] = lim; bits |= R2IK_EMG_SHOULDER_PITCH; }
  if (j[0] < -lim) { j[0] = -lim; bits |= R2IK_EMG_SHOULDER_PITCH; }
  if (j[2] > lim) { j[2] = lim; bits |= R2IK_EMG_ELBOW_YAW; }
  if (j[2] < -lim) { j[2] = -lim; bits |= R2IK_EMG_ELBOW_YAW; }
  if (j[6] > lim) { j[6] = lim; bits |= R2IK_EMG_WRIST_YAW; }
  if (j[6] < -lim) { j[6] = -lim; bits |= R2IK_EMG_WRIST_YAW; }
  return bits;
}

// ctl:464-497 safety_checks
R2IK_HD int safety_checks(double j[7], const double previous_sol[7], double orbita_max) {
  limit_orbita3d_wrist(j, orbita_max);                      // utl:522-532
  return safety_multiturn(j, previous_sol);
}

R2IK_HD double joints_angle_distance(const double a[7], const double b[7]) {
  double s = 0.0;
  for (int i = 0; i < 7; ++i) { double d = angle_diff(a[i], b[i]); s += d * d; }
  return sqrt(s);
}

// utl:267-331 get_best_theta_to_current_joints: ternary search of the theta whose joints are
// closest to current_joints.  get_joints mutates S exactly like the reference (the state leak
// is part of the reference result when the elbow projection fires, SURVEY.md A.6.1).
R2IK_HD double best_theta_to_current_joints(const ArmConst &A, Solve &S, const double current_joints[7],
                                            double preferred_theta) {
  double low = -kPi, high = kPi;
  if (A.side < 0) { low = 0.0; high = kTwoPi; }
  const double tolerance = 0.01;
  double j1[7], j2[7], E[3];
  get_joints(A, S, preferred_theta, 0.0, 0.0, j1, E);
  if (joints_angle_distance(j1, current_joints) < tolerance) return preferred_theta;
  while ((high - low) > tolerance) {
    double mid1 = low + (high - low) / 3;
    double mid2 = high - (high - low) / 3;
    get_joints(A, S, mid1, 0.0, 0.0, j1, E);
    get_joints(A, S, mid2, 0.0, 0.0, j2, E);
    double f1 = joints_angle_distance(j1, current_joints);
    double f2 = joints_angle_distance(j2, current_joints);
    if (f1 < f2) high = mid2; else low = mid1;
  }
  double best = (low + high) / 2;
  get_joints(A, S, best, 0.0, 0.0, j1, E);  // utl:324: one more call (its state leak is observable)
  return best;
}

// The same search as ControlIK's CONSTRUCTOR runs it (ctl:142-159): there `current_joints` is the list of BOTH arms' joint
// lists, so the reference's cost loops over i < len(current_joints) = n_rows and broadcasts joints[i] against the whole
// row i:  cost^2 = sum_{i < n_rows} sum_{k < 7} angle_diff(joints[i], rows[i][k])^2  (SURVEY.md A.6.11).  The value
// seeds ControlIK.previous_theta, a visible attribute that no output depends on.
R2IK_HD double ctor_rows_distance(const double j[7], const double *rows, int n_rows) {
  double s = 0.0;
  for (int i = 0; i < n_rows; ++i)
    for (int k = 0; k < 7; ++k) { double d = angle_diff(j[i], rows[7 * i + k]); s += d * d; }
  return sqrt(s);
}
R2IK_HD double ctor_previous_theta(const ArmConst &A, Solve &S, const double *rows, int n_rows, double preferred_theta) {
  double low = -kPi, high = kPi;
  if (A.side < 0) { low = 0.0; high = kTwoPi; }
  const double tolerance = 0.01;
  double j1[7], j2[7], E[3];
  get_joints(A, S, preferred_theta, 0.0, 0.0, j1, E);
  if (ctor_rows_distance(j1, rows, n_rows) < tolerance) return preferred_theta;
  while ((high - low) > tolerance) {
    double mid1 = low + (high - low) / 3;
    double mid2 = high - (high - low) / 3;
    get_joints(A, S, mid1, 0.0, 0.0, j1, E);
    get_joints(A, S, mid2, 0.0, 0.0, j2, E);
    if (ctor_rows_distance(j1, rows, n_rows) < ctor_rows_distance(j2, rows, n_rows)) high = mid2; else low = mid1;
  }
  return (low + high) / 2;
}

// ControlIK.__init__'s seed of previous_theta (ctl:142-159): is_reachable_no_limits on the current pose (identity snap of
// ctl:142), then the constructor's form of the ternary search.  NaN for a pose without an elbow circle.
R2IK_HD double ctl_ctor_theta(const ArmConst &A, const double *current_pose, const double *rows, int n_rows,
                              double preferred_theta) {
  Solve S;
  const double cpos[3] = {current_pose[3], current_pose[7], current_pose[11]};
  double theta = NAN;
  if (rotation_from_mat4(current_pose, true, S.R) && is_reachable_R<true>(A, cpos, S).state == R2IK_STATE_REACHABLE)
    theta = ctor_previous_theta(A, S, rows, n_rows, preferred_theta);
  return theta;
}

// Selection + joints + safety for one pose whose is_reachable result is already known.
// Shared tail of the discrete path (ctl:454-462).
R2IK_HD int discrete_finish(const ArmConst &A, const R2ikCtlParams &par, Solve &S, bool found, double theta,
                            const double prev_joints[7], const double current_joints[7], double joints[7]) {
  if (found) {
    theta = limit_theta_to_interval(theta, par.interval_limit[0], par.interval_limit[1]);
    double E[3];
    get_joints(A, S, theta, prev_joints[0], prev_joints[2], joints, E);
  } else {
    for (int i = 0; i < 7; ++i) joints[i] = current_joints[i];
  }
  return safety_checks(joints, prev_joints, par.orbita3d_max_angle);
}

// Discrete mode, per pose (k_ctl_discrete, k_ctl_discrete_scan and the three passes of r2ik_discrete_compact.cuh).
// Classify: the rotation with the near-identity snap (ctl:212-217), is_reachable, and for a reachable pose the
// preferred theta first (utl:357-364); a reachable pose without that shortcut needs the K-sample search.  false:
// invalid rotation (rc.state = INVALID_ROTATION).
R2IK_HD bool disc_classify(const ArmConst &A, const R2ikCtlParams &par, const double *row, Solve &S, Reach &rc,
                           bool &shortcut, bool &need_search) {
  double pos[3];
  shortcut = false;
  need_search = false;
  rc.state = R2IK_STATE_INVALID_ROTATION;
  rc.literal = false;
  if (!load_pose<R2IK_POSE_MAT4>(row, true, pos, S.R)) return false;
  rc = is_reachable_R<false>(A, pos, S);
  if (rc.state == R2IK_STATE_REACHABLE) {
    shortcut = preferred_theta_works(A, S, rc.i0, rc.i1, par.preferred_theta);
    need_search = !shortcut;
  }
  return true;
}

// The K samples of a pose's search (utl:366-375); the elbow tests P.T are the caller's
R2IK_HD SearchPlan disc_search_plan(const R2ikCtlParams &par, double i0, double i1) {
  SearchPlan P;
  P.preferred_theta = par.preferred_theta;
  double start, stop;
  search_range(i0, i1, start, stop);
  P.L = make_linspace(start, stop, par.nb_search_points);
  return P;
}
// ... with the elbow tests of the solved pose
R2IK_HD SearchPlan disc_search_plan(const ArmConst &A, const R2ikCtlParams &par, const Solve &S, const Reach &rc) {
  SearchPlan P = disc_search_plan(par, rc.i0, rc.i1);
  P.T = make_elbow_test(A, S);
  return P;
}

// The arg-min of the K-sample search (utl:376-390) from a plan: search_analytic, or the exhaustive scan where its atan2
// arguments are out of range.  false: no valid sample (theta untouched).
R2IK_HD bool disc_search(const SearchPlan &P, int nb, double &theta) {
  double best;
  int best_k;
  if (!search_analytic(P, nb, best, best_k)) search_strided(P, nb, 0, 1, best, best_k);
  const bool found = best < INFINITY;
  if (found) theta = linspace_value(P.L, best_k);
  return found;
}

// ---------------------------------------------------------------------------------------
// Continuous mode (ctl:276-407), cut at its data dependences.  Of one waypoint's work only two thin
// strands depend on the trajectory's past: the rate-limited elbow angle (previous_theta) and the
// unwrap / continuity / emergency chain (previous_sol).  Everything else -- the goal rotation,
// is_reachable, the 10-sample search for the target theta, get_joints for a GIVEN theta, the Orbita3D
// limit -- is a function of the waypoint alone.  The four pieces below are exactly the statements of
// the reference's function, regrouped; continuous_step composes them for one waypoint (serial kernel,
// host harness) and the phased kernels run (1) and (3) over all waypoints in parallel and (2), (4) as
// short per-trajectory scans, with the same flags / states and joints equal to rounding.
// ---------------------------------------------------------------------------------------
#define R2IK_WP_INVALID 0        // rotation block with det <= 0
#define R2IK_WP_TARGET 1         // reachable, a target theta was found                       (ctl:350-361)
#define R2IK_WP_NO_SAMPLE 2      // reachable, no valid sample: theta = previous, "limited by shoulder" (ctl:362-363)
#define R2IK_WP_UNREACHABLE 3    // not reachable: no-limits solve, tend to preferred_theta   (ctl:368-388)
#define R2IK_WP_SERIAL 0x80      // get_joints hit a degenerate input: phase (4) redoes this waypoint in order

// (1) stateless: classify the waypoint and find its target theta.  S holds the goal rotation on exit
// (and the is_reachable solve for codes 1, 2).
R2IK_HD int cont_target(const ArmConst &A, const R2ikCtlParams &par, const double *M, Solve &S, double pos[3], double &goal,
                        int &st_out) {
  pos[0] = M[3]; pos[1] = M[7]; pos[2] = M[11];
  goal = 0.0;
  if (!rotation_from_mat4(M, true, S.R)) { st_out = R2IK_STATE_INVALID_ROTATION; return R2IK_WP_INVALID; }
  Reach rc = is_reachable_R<false>(A, pos, S);
  if (rc.state != R2IK_STATE_REACHABLE) { st_out = rc.state; return R2IK_WP_UNREACHABLE; }
  if (best_discrete_theta(A, S, rc.i0, rc.i1, par.nb_search_points_continuous, par.preferred_theta_ctor, goal)) {
    st_out = R2IK_STATE_EMPTY;
    return R2IK_WP_TARGET;
  }
  st_out = R2IK_STATE_LIMITED_BY_SHOULDER;
  return R2IK_WP_NO_SAMPLE;
}

// (2) scan over previous_theta: ctl:306-325 (re)initialisation
R2IK_HD double cont_initial_theta(const ArmConst &A, const R2ikCtlParams &par, const double current_joints[7],
                                  const double *current_pose) {
  Solve S;
  double cpos[3] = {current_pose[3], current_pose[7], current_pose[11]};
  rotation_from_mat4(current_pose, true, S.R);
  is_reachable_R<true>(A, cpos, S);
  return best_theta_to_current_joints(A, S, current_joints, par.preferred_theta);
}
// ... and the step of the scan (ctl:350-366, 379-381)
R2IK_HD double cont_next_theta(const R2ikCtlParams &par, int code, double goal, double previous_theta) {
  double theta;
  if (code == R2IK_WP_TARGET) theta = step_toward(goal, previous_theta, par.d_theta_max);
  else if (code == R2IK_WP_NO_SAMPLE) theta = previous_theta;
  else theta = step_toward(par.preferred_theta, previous_theta, par.d_theta_max);
  return limit_theta_to_interval(theta, par.interval_limit[0], par.interval_limit[1]);
}

// (3) stateless for a given theta: joints + Orbita3D limit.  S.R / pos as left by cont_target; an
// unreachable waypoint is solved without limits first (ctl:369).  prev0 / prev2 only matter at the exact
// singularities of get_joints.
R2IK_HD void cont_raw_joints(const ArmConst &A, const R2ikCtlParams &par, int code, const double pos[3], Solve &S, double theta,
                             double prev0, double prev2, double joints[7]) {
  if (code == R2IK_WP_UNREACHABLE) is_reachable_R<true>(A, pos, S);
  double E[3];
  get_joints(A, S, theta, prev0, prev2, joints, E);
  limit_orbita3d_wrist(joints, par.orbita3d_max_angle);                        // ctl:393, first link of safety_checks
}

// (4) scan over previous_sol: unwrap + clamp, continuity check, emergency latch (ctl:393-405)
R2IK_HD void cont_finish(R2ikTrajState &cs, double joints[7]) {
  int bits = safety_multiturn(joints, cs.previous_sol);
  if (bits) { cs.emergency_stop = 1; cs.emergency_bits |= bits; }
  if (!cs.init) {                                            // ctl:395-400, utl:571-589
    const double max_step[7] = {0.5, 0.5, 0.5, 0.5, 1.0, 1.0, 1.0};
    bool discontinuity = false;
    for (int i = 0; i < 7; ++i)
      if (fabs(angle_diff(joints[i], cs.previous_sol[i])) > max_step[i]) discontinuity = true;
    if (discontinuity) {
      for (int i = 0; i < 7; ++i) joints[i] = cs.previous_sol[i];
      cs.emergency_stop = 1;
      cs.emergency_bits |= R2IK_EMG_DISCONTINUITY;
    }
  }
  cs.init = 0;
  if (!cs.emergency_stop)
    for (int i = 0; i < 7; ++i) cs.previous_sol[i] = joints[i];
}

// ctl:276-407 symbolic_inverse_kinematics_continuous for one waypoint of one trajectory.
R2IK_HD void continuous_step(const ArmConst &A, const R2ikCtlParams &par, const double *M,
                             const double current_joints[7], const double *current_pose, R2ikTrajState &cs,
                             double joints[7], uint8_t &reachable, uint8_t &state) {
  if (cs.emergency_stop) {                                   // ctl:205-210
    for (int i = 0; i < 7; ++i) joints[i] = cs.previous_sol[i];
    reachable = 0; state = R2IK_STATE_EMERGENCY;
    return;
  }
  Solve S;
  double pos[3], goal;
  int st_out;
  const int code = cont_target(A, par, M, S, pos, goal, st_out);
  if (code == R2IK_WP_INVALID) {
    for (int i = 0; i < 7; ++i) joints[i] = NAN;
    reachable = 0; state = R2IK_STATE_INVALID_ROTATION;
    return;
  }
  if (!cs.has_previous_sol) {                                // ctl:306-325
    for (int i = 0; i < 7; ++i) cs.previous_sol[i] = current_joints[i];
    cs.has_previous_sol = 1;
    cs.init = 1;
    cs.previous_theta = cont_initial_theta(A, par, current_joints, current_pose);
  }
  const double theta = cont_next_theta(par, code, goal, cs.previous_theta);
  cs.previous_theta = theta;
  cont_raw_joints(A, par, code, pos, S, theta, cs.previous_sol[0], cs.previous_sol[2], joints);
  cont_finish(cs, joints);
  reachable = code == R2IK_WP_TARGET ? 1 : 0;
  state = (uint8_t)st_out;
}

}  // namespace r2ik
