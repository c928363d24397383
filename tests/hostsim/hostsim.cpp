// TEST-ONLY host harness: compiles the device solver source (the csrc headers, all __host__ __device__) with g++ and
// loops over poses / waypoints / pairs on the CPU, calling the same per-item functions the kernels call, so the kernel
// *logic* is checked against the golden fixtures in the GPU-less CI.  It is not part of libr2ik.so, is never imported
// by the package, and is no fallback for anything.
#include <cstring>
#include <vector>
#include <cstdint>
#include <type_traits>

#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_control.cuh"
#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_cont_codes.cuh"
#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_discrete_compact.cuh"
#define R2IK_F32_DEBUG 1
#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_device_f32.cuh"
#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_host.h"

using namespace r2ik;

// f(std::integral_constant<int, KIND>) for the pose layout `kind` (EULER6, anything else MAT4)
template <typename F>
static void by_kind(int kind, F f) {
  if (kind == R2IK_POSE_EULER6) f(std::integral_constant<int, R2IK_POSE_EULER6>());
  else f(std::integral_constant<int, R2IK_POSE_MAT4>());
}

extern "C" {

// r2ik_math.cuh: the straight-line atan2 (host build: '/' instead of the MUFU seed + Newton).
void hs_atan2_core(const double *y, const double *x, int64_t n, double *out, uint8_t *ok) {
  for (int64_t i = 0; i < n; ++i) {
    ok[i] = atan2_core_ok(y[i], x[i]);
    out[i] = atan2_core(y[i], x[i]);
  }
}

// angle_of_unit on (x, y) / |(x, y)| normalised the way cs_of_atan2 does
void hs_angle_of_unit(const double *y, const double *x, int64_t n, double *out) {
  for (int64_t i = 0; i < n; ++i) {
    double c, s;
    bool degenerate = false;
    cs_of_atan2<false>(y[i], x[i], c, s, degenerate);
    out[i] = degenerate ? NAN : angle_of_unit(c, s);
  }
}

void hs_sincos_small(const double *x, int64_t n, double *sn, double *cs) {
  for (int64_t i = 0; i < n; ++i) sincos_small(x[i], sn[i], cs[i]);
}

// utl:508-519 on n wrist triples (joints[4:7])
void hs_limit_orbita3d(const double *w, int64_t n, double max_angle, double *out) {
  for (int64_t i = 0; i < n; ++i) {
    double j[7] = {0, 0, 0, 0, w[3 * i], w[3 * i + 1], w[3 * i + 2]};
    limit_orbita3d_wrist(j, max_angle);
    out[3 * i] = j[4]; out[3 * i + 1] = j[5]; out[3 * i + 2] = j[6];
  }
}

void hs_constants(const R2ikArmConfig *cfg, R2ikArmConstants *pub) {
  ArmConst A;
  derive_constants(*cfg, A, *pub);
}

void hs_symik_batch(const R2ikArmConfig *cfg, int kind, const double *poses, const double *theta, int64_t n,
                    uint8_t *reach, uint8_t *state, double *interval, double *joints, double *elbow) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  by_kind(kind, [&](auto K) {
    for (int64_t i = 0; i < n; ++i) {
      Solve S;
      const Reach rc = symik_reach<K()>(A, poses + pose_stride(K()) * i, S);
      reach[i] = rc.state == R2IK_STATE_REACHABLE;
      state[i] = (uint8_t)rc.state;
      interval[2 * i] = rc.i0; interval[2 * i + 1] = rc.i1;
      symik_joints(A, S, rc, theta ? theta + i : nullptr, 0.0, 0.0, joints + 7 * i, elbow + 3 * i);
    }
  });
}

void hs_no_limits_batch(const R2ikArmConfig *cfg, int kind, const double *poses, const double *theta, int64_t n,
                        double *joints, double *elbow) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  by_kind(kind, [&](auto K) {
    for (int64_t i = 0; i < n; ++i)
      symik_no_limits<K()>(A, poses + pose_stride(K()) * i, theta + i, nullptr, joints + 7 * i, elbow + 3 * i);
  });
}

void hs_ctl_discrete_batch(const R2ikArmConfig *cfg, const R2ikCtlParams *par, const double *M, int64_t n,
                           const double *prev, const double *cur, double *joints, uint8_t *reach, uint8_t *state,
                           uint8_t *emg) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  for (int64_t i = 0; i < n; ++i) {
    Solve S;
    Reach rc;
    bool found, need_search;
    double theta = 0.0;
    const bool valid = disc_classify(A, *par, M + 16 * i, S, rc, found, need_search);
    int st = rc.state;
    if (found) theta = par->preferred_theta;
    if (need_search) {
      found = disc_search(disc_search_plan(A, *par, S, rc), par->nb_search_points, theta);
      if (!found) st = R2IK_STATE_LIMITED_BY_SHOULDER;
    }
    if (valid) emg[i] = (uint8_t)discrete_finish(A, *par, S, found, theta, prev, cur, joints + 7 * i);
    else {
      for (int k = 0; k < 7; ++k) joints[7 * i + k] = NAN;
      emg[i] = 0;
    }
    reach[i] = found; state[i] = (uint8_t)st;
  }
}

// The three passes of r2ik_ctl_discrete_compact_f64 one after the other over the same lists, with the appends in `order`
// (0: ascending, 1: descending pose index) to show that the result does not depend on the order the blocks arrive in.
// n_lists[0..2] receive the list lengths and the number of finish entries that carry the literal-solve flag.
void hs_ctl_discrete_compact_batch(const R2ikArmConfig *cfg, const R2ikCtlParams *par, const double *M, int64_t n,
                                   const double *prev, const double *cur, int order, double *joints, uint8_t *reach,
                                   uint8_t *state, uint8_t *emg, int64_t *n_lists) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  DiscHeader hdr;
  disc_header_init(&hdr, *par, prev, cur);
  std::vector<uint32_t> search_idx((size_t)n), finish_idx((size_t)n);
  std::vector<double> plan(8 * (size_t)n), finish_theta((size_t)n);
  for (int64_t q = 0; q < n; ++q) {   // k_disc_classify
    const int64_t i = order ? n - 1 - q : q;
    Solve S;
    Reach rc;
    bool shortcut, need_search;
    uint32_t tag = (uint32_t)i;
    disc_classify(A, *par, M + 16 * i, S, rc, shortcut, need_search);
    if (rc.literal) tag |= kDiscLiteral;
    if (need_search) {
      const size_t k = hdr.n_search++;
      search_idx[k] = tag;
      disc_plan_pack(&plan[8 * k], A, S, rc.i0, rc.i1);
    } else if (shortcut) {
      const size_t k = hdr.n_finish++;
      finish_idx[k] = tag; finish_theta[k] = par->preferred_theta;
    } else {
      disc_store_final(&hdr, i, rc.state, joints, reach, state, emg);
    }
  }
  n_lists[0] = hdr.n_search;
  for (size_t k = 0; k < hdr.n_search; ++k) {   // k_disc_search
    const uint32_t tag = search_idx[k];
    double theta;
    if (disc_search(disc_plan_unpack(*par, &plan[8 * k]), par->nb_search_points, theta)) {
      const size_t f = hdr.n_finish++;
      finish_idx[f] = tag; finish_theta[f] = theta;
    } else {
      disc_store_final(&hdr, (int64_t)(tag & ~kDiscLiteral), R2IK_STATE_LIMITED_BY_SHOULDER, joints, reach, state, emg);
    }
  }
  n_lists[1] = hdr.n_finish;
  n_lists[2] = 0;
  for (size_t k = 0; k < hdr.n_finish; ++k) {   // k_disc_finish
    const uint32_t tag = finish_idx[k];
    n_lists[2] += (tag & kDiscLiteral) != 0;
    const int64_t i = tag & ~kDiscLiteral;
    emg[i] = (uint8_t)disc_finish_listed(A, *par, M + 16 * i, (tag & kDiscLiteral) != 0, finish_theta[k], prev, joints + 7 * i);
    reach[i] = 1; state[i] = R2IK_STATE_REACHABLE;
  }
}

void hs_ctl_continuous_batch(const R2ikArmConfig *cfg, const R2ikCtlParams *par, const double *M, int64_t T, int32_t W,
                             const double *cur_joints, const double *cur_pose, R2ikTrajState *st, double *joints,
                             uint8_t *reach, uint8_t *state) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  for (int64_t t = 0; t < T; ++t)
    for (int32_t w = 0; w < W; ++w) {
      size_t k = (size_t)t * W + w;
      continuous_step(A, *par, M + 16 * k, cur_joints + 7 * t, cur_pose + 16 * t, st[t], joints + 7 * k, reach[k], state[k]);
    }
}

// The phased K3 on the host, phase after phase over the whole batch with the device functions the kernels call:
// k_cont_targets, k_cont_thetas, then k_cont_raw_joints_codes
// (raw joints + the 16-bit code of every waypoint against its predecessor; the first waypoint of a trajectory is irregular) and k_cont_finish_codes (cont_finish_codes_trajectory, the same function the kernel calls).
void hs_ctl_continuous_phased_batch(const R2ikArmConfig *cfg, const R2ikCtlParams *par, const double *M, int64_t T, int32_t W,
                                   const double *cur_joints, const double *cur_pose, R2ikTrajState *st, double *joints,
                                   uint8_t *reach, uint8_t *state, double *ws, uint16_t *codes, int force_serial_mod) {   // codes: in / out
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  const int64_t n_wp = T * W;
  for (int64_t k = 0; k < n_wp; ++k) {                       // k_cont_targets
    Solve S; double pos[3], goal; int sto;
    int c = cont_target(A, *par, M + 16 * k, S, pos, goal, sto);
    ws[k] = goal; reach[k] = (uint8_t)c; state[k] = (uint8_t)sto;
  }
  for (int64_t t = 0; t < T; ++t) {                          // k_cont_thetas
    if (st[t].emergency_stop) continue;
    double theta = st[t].previous_theta;
    bool has = st[t].has_previous_sol != 0;
    for (int32_t w = 0; w < W; ++w) {
      size_t k = (size_t)t * W + w;
      int c = reach[k];
      if (c == R2IK_WP_INVALID) continue;
      if (!has) { theta = cont_initial_theta(A, *par, cur_joints + 7 * t, cur_pose + 16 * t); has = true; }
      theta = cont_next_theta(*par, c, ws[k], theta);
      ws[k] = theta;
    }
  }
  for (int64_t t = 0; t < T; ++t) {                          // k_cont_raw_joints_codes
    bool prev_ordinary = false;
    double jp[7];
    for (int32_t w = 0; w < W; ++w) {
      size_t k = (size_t)t * W + w;
      int c = reach[k];
      double j[7];
      bool serial = false;
      for (int q = 0; q < 7; ++q) j[q] = NAN;
      if (c != R2IK_WP_INVALID) serial = cont_raw_joints_item(A, *par, M + 16 * k, c, ws + k, k, force_serial_mod, j);
      const bool ordinary = c != R2IK_WP_INVALID && !serial;
      unsigned cd = (ordinary && w > 0 && prev_ordinary) ? cont_wind_code(j, jp) : cont_irregular_code(serial ? (c | R2IK_WP_SERIAL) : c);
      codes[k] = (uint16_t)cd;
      reach[k] = c == R2IK_WP_TARGET ? 1 : 0;
      for (int q = 0; q < 7; ++q) { joints[7 * k + q] = j[q]; jp[q] = j[q]; }
      prev_ordinary = ordinary;
    }
  }
  for (int64_t t = 0; t < T; ++t) {                          // k_cont_finish_codes
    const double *Mt = M + 16 * (size_t)t * W;
    auto serial = [&](int w, int kind, double theta, double p0, double p2, double *out) {
      cont_serial_joints(A, *par, Mt + 16 * (size_t)w, kind, theta, p0, p2, out);
    };
    const size_t base = (size_t)t * W;
    cont_finish_codes_trajectory(W, cur_joints + 7 * t, st[t], ws + base, codes + base, joints + 7 * base, reach + base, state + base, serial);
  }
}

double hs_ctl_ctor_theta(const R2ikArmConfig *cfg, double preferred_theta, const double *rows, int n_rows, const double *current_pose) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  return ctl_ctor_theta(A, current_pose, rows, n_rows, preferred_theta);
}

void hs_elbow_positions(const R2ikArmConfig *cfg, int kind, const double *poses, const double *thetas, int K, int64_t n,
                        int no_limits, double *elbows, uint8_t *projected) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  by_kind(kind, [&](auto KI) {
    for (int64_t i = 0; i < n; ++i) {
      const double *row = poses + pose_stride(KI()) * i;
      Solve S;
      const bool circle = no_limits ? pose_elbow_circle<KI(), true>(A, row, S) : pose_elbow_circle<KI(), false>(A, row, S);
      for (int k = 0; k < K; ++k)
        projected[i * K + k] = elbow_on_circle(A, S, circle, thetas + (i * K + k), elbows + (i * K + k) * 3);
    }
  });
}

// K1-f32 (r2ik_device_f32.cuh): the FP32 fast solve with FP64 escalation, as k_symik_solve_f32 + k_symik_escalated_f32.
// mode: 0 = as the kernels (escalate flagged poses), 1 = never escalate (raw FP32 results, to measure them).
void hs_symik_batch_f32(const R2ikArmConfig *cfg, int kind, const float *poses, const float *theta, int64_t n, int mode,
                        uint8_t *reach, uint8_t *state, float *interval, float *joints, float *elbow, uint8_t *escalated) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  f32::ArmConstF F;
  f32::narrow_constants(A, F);
  const int stride = kind == R2IK_POSE_EULER6 ? 6 : 16;
  for (int64_t i = 0; i < n; ++i) {
    const float *in = poses + i * stride;
    float out[12];
    int st;
    const bool has_theta = theta != nullptr;
    g_dbg_n = 0;
    const float th = has_theta ? theta[i] : 0.0f;
    bool esc = kind == R2IK_POSE_EULER6 ? f32::symik_pose_fast<R2IK_POSE_EULER6>(A, F, in, has_theta, th, st, out)
                                        : f32::symik_pose_fast<R2IK_POSE_MAT4>(A, F, in, has_theta, th, st, out);
    escalated[i] = esc;
    if (mode == 2) { for (int k = 0; k < 12; ++k) out[k] = k < g_dbg_n ? g_dbg[k] : NAN; }
    if (mode == 3) { out[0] = (float)g_dbg_cause; }
    g_dbg_n = 0; g_dbg_cause = 0;
    if (esc && mode == 0) {
      if (kind == R2IK_POSE_EULER6) f32::symik_pose_escalated<R2IK_POSE_EULER6>(A, in, has_theta, th, 0.0f, 0.0f, &st, out);
      else f32::symik_pose_escalated<R2IK_POSE_MAT4>(A, in, has_theta, th, 0.0f, 0.0f, &st, out);
    }
    state[i] = (uint8_t)st;
    reach[i] = st == R2IK_STATE_REACHABLE;
    interval[2 * i] = out[0]; interval[2 * i + 1] = out[1];
    for (int k = 0; k < 7; ++k) joints[7 * i + k] = out[2 + k];
    for (int k = 0; k < 3; ++k) elbow[3 * i + k] = out[9 + k];
  }
}

// search_analytic vs the exhaustive scan (search_strided, stride 1) on n random search plans:
// plans[i] = start, stop, A1, B1, C1, A2, B2, C2, preferred (9 doubles).
void hs_search_compare(const double *plans, int64_t n, int nb, double *best_scan, int32_t *k_scan, double *best_ana,
                       int32_t *k_ana, uint8_t *ok) {
  for (int64_t i = 0; i < n; ++i) {
    const double *q = plans + 9 * i;
    SearchPlan P;
    P.L = make_linspace(q[0], q[1], nb);
    P.T.A1 = q[2]; P.T.B1 = q[3]; P.T.C1 = q[4]; P.T.A2 = q[5]; P.T.B2 = q[6]; P.T.C2 = q[7];
    P.preferred_theta = q[8];
    int ks, ka;
    search_strided(P, nb, 0, 1, best_scan[i], ks);
    ok[i] = search_analytic(P, nb, best_ana[i], ka);
    k_scan[i] = ks; k_ana[i] = ka;
  }
}

// K4 with the mixed-precision flag and FP64 escalation (reach_pair, as k_reach_map).
// mode 0: as the kernel; mode 1: never escalate (to measure what the bands catch).  n_esc: escalated pairs.
void hs_reach_map_mixed(const R2ikArmConfig *cfg, const double *origin, const double *step, const int32_t *dims,
                        const double *ori_euler, int32_t ori_begin, int32_t ori_end, int mode, uint32_t *counts,
                        uint64_t *n_esc, uint64_t *n_live_pairs) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  f32::ArmConstF F;
  f32::narrow_constants(A, F);
  const int no = ori_end - ori_begin;
  std::vector<f32::OriConst> O((size_t)no);
  for (int o = 0; o < no; ++o) {
    const double *e = ori_euler + 3 * (size_t)(ori_begin + o);
    double R[9];
    rot_from_euler_xyz(e[0], e[1], e[2], R);
    O[o] = f32::make_ori_const(A, R);
  }
  *n_esc = 0; *n_live_pairs = 0;
  for (int ix = 0; ix < dims[0]; ++ix)
    for (int iy = 0; iy < dims[1]; ++iy)
      for (int iz = 0; iz < dims[2]; ++iz) {
        double px = origin[0] + ix * step[0], py = origin[1] + iy * step[1], pz = origin[2] + iz * step[2];
        uint32_t count = 0;
        if (reach_prechecks(A, px, py, pz) < 0) {
          const double ps[3] = {px - A.s[0], py - A.s[1], pz - A.s[2]};
          for (int o = 0; o < no; ++o) {
            bool esc = false;
            const int st = mode == 1 ? f32::reach_flag_mixed(A, F, ps, px, O[o], esc)
                                     : f32::reach_pair(A, F, ps, px, py, pz, O[o], ori_euler + 3 * (size_t)(ori_begin + o), esc);
            ++*n_live_pairs;
            if (esc) ++*n_esc;
            count += st == R2IK_STATE_REACHABLE;
          }
        }
        counts[((size_t)ix * dims[1] + iy) * dims[2] + iz] = count;
      }
}

}  // extern "C"
