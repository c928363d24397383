/* TEST-ONLY: the CPU oracle's get_best_theta_to_current_joints (oracle/r2ik_oracle.c, utils.py:267-331) batched over
 * poses with per-pose current joints, for tests/test_best_theta_host.py and tests/test_gpu_best_theta.py, which compile
 * it with the oracle's flags (oracle/Makefile) into a temporary directory.  The oracle source is included as it is, so
 * the solve, get_joints and the search below are the oracle's own functions.  Never part of the package. */
#include "../../oracle/r2ik_oracle.c"

/* utl:267-331 with the decision margins of one search: *cmp_margin = the smallest |f1 - f2| over the search's
 * comparisons (INFINITY when the shortcut returns), *shortcut_margin = |f(preferred_theta) - 0.01|.  The comparisons and
 * the get_joints calls are those of get_best_theta_to_current_joints, in the same order on the same solver. */
static double best_theta_with_margins(orc_solver *s, const double current_joints[7], double preferred_theta,
                                      double *cmp_margin, double *shortcut_margin) {
  static const double zero7[7] = {0, 0, 0, 0, 0, 0, 0};
  double low = -ORC_PI, high = ORC_PI;
  if (s->cfg.side < 0) { low = 0; high = 2 * ORC_PI; }
  const double tolerance = 0.01;
  double j[7], j2[7];
  *cmp_margin = INFINITY;
  solver_get_joints(s, preferred_theta, zero7, j, 0);
  const double f0 = joints_angle_dist(j, current_joints);
  *shortcut_margin = fabs(f0 - tolerance);
  if (f0 < tolerance) return preferred_theta;
  while ((high - low) > tolerance) {
    double mid1 = low + (high - low) / 3;
    double mid2 = high - (high - low) / 3;
    solver_get_joints(s, mid1, zero7, j, 0);
    solver_get_joints(s, mid2, zero7, j2, 0);
    double f1 = joints_angle_dist(j, current_joints);
    double f2 = joints_angle_dist(j2, current_joints);
    if (fabs(f1 - f2) < *cmp_margin) *cmp_margin = fabs(f1 - f2);
    if (f1 < f2) high = mid2; else low = mid1;
  }
  return (low + high) / 2;
}

/* Solve pose i on a fresh solver (is_reachable, or is_reachable_no_limits); returns the state (no_limits: reachable
 * with an elbow circle, else "out of reach - should not happen", as r2ik_symik_best_theta_f64 reports it). */
static int solve_fresh(orc_solver *s, const orc_arm_config *cfg, int kind, const double *row, int no_limits) {
  double pos[3], eul[3], itv[2];
  solver_init(s, cfg);
  if (load_pose(kind, row, pos, eul)) return ORC_STATE_INVALID_ROTATION;
  if (no_limits) return solver_is_reachable_no_limits(s, pos, eul) ? ORC_STATE_REACHABLE : ORC_STATE_SHOULD_NOT_HAPPEN;
  int st;
  solver_is_reachable(s, pos, eul, itv, &st);
  return st;
}

/* For each pose: state; theta = get_best_theta_to_current_joints on the pose's solve (NaN unless reachable); joints =
 * get_joints(theta) as the first call on a fresh solve; the two margins of the search (NaN unless reachable);
 * theta_check (nullable) = the oracle's get_best_theta_to_current_joints itself on another fresh solve.
 * current_joints: row i at current_joints + cj_stride * i (cj_stride 0 or 7). */
void orc_best_theta_batch(const orc_arm_config *cfg, int kind, const double *poses, int64_t n, const double *current_joints,
                          int cj_stride, double preferred_theta, int no_limits, uint8_t *state, double *theta,
                          double *joints, double *cmp_margin, double *shortcut_margin, double *theta_check) {
  static const double zero7[7] = {0, 0, 0, 0, 0, 0, 0};
  const int stride = kind == ORC_POSE_EULER6 ? 6 : 16;
#pragma omp parallel for schedule(dynamic, 64)
  for (int64_t i = 0; i < n; i++) {
    const double *row = poses + i * stride, *cj = current_joints + (int64_t)cj_stride * i;
    orc_solver s;
    const int st = solve_fresh(&s, cfg, kind, row, no_limits);
    state[i] = (uint8_t)st;
    fill_nan(joints + 7 * i, 7);
    theta[i] = cmp_margin[i] = shortcut_margin[i] = NAN;
    if (theta_check) theta_check[i] = NAN;
    if (st != ORC_STATE_REACHABLE) continue;
    theta[i] = best_theta_with_margins(&s, cj, preferred_theta, cmp_margin + i, shortcut_margin + i);
    solve_fresh(&s, cfg, kind, row, no_limits);
    solver_get_joints(&s, theta[i], zero7, joints + 7 * i, 0);
    if (theta_check) {
      solve_fresh(&s, cfg, kind, row, no_limits);
      theta_check[i] = get_best_theta_to_current_joints(&s, cj, preferred_theta);
    }
  }
}
