// r2ik_kernels.cu -- sm_100a kernels and the C ABI of libr2ik.so (include/r2ik.h).
//
//   K1     k_symik_solve                        one thread / pose: is_reachable + get_joints (FP64)
//   K1-f32 k_symik_solve_f32 + k_symik_escalated_f32   the FP32 fast path; undecidable poses re-solved in FP64
//   K1b    k_symik_no_limits, k_elbow_positions    is_reachable_no_limits, get_elbow_position
//   K1s    k_symik_sweep                        one solve per pose, get_joints at K elbow angles spread over the block
//   K2     k_ctl_discrete                       one lane / pose, analytic arg-min over the K elbow samples
//          k_ctl_discrete_scan                  the exhaustive warp-cooperative scan of the K samples (cross-check)
//   K3     k_cont_targets / k_cont_thetas / k_cont_raw_joints_codes / k_cont_finish_codes / k_cont_apply_windings
//                                               continuous mode cut at its data dependences: per-waypoint kernels
//                                               and per-trajectory scans;  k_ctl_continuous = the one-kernel form
//   K4     k_reach_map                          one thread / voxel, mixed-precision flag with FP64 escalation
//          k_reach_map_f64                      every pair by the FP64 flag solve (cross-check)
//
// The work is scalar FP64 / FP32 (sincos / atan2 / sqrt / FMA chains): it runs on the FP64 and FP32 pipes, not on
// tensor cores; HBM traffic is a few hundred bytes per pose.  There is no host implementation
// of any entry point in this library.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "r2ik_control.cuh"
#include "r2ik_device_f32.cuh"
#include "r2ik_host.h"

using namespace r2ik;

#ifndef R2IK_BLOCK
#define R2IK_BLOCK 128
#endif
#ifndef R2IK_K1_MINBLOCKS
#define R2IK_K1_MINBLOCKS 4   // resident blocks / SM the register allocation of K1 is held to
#endif

// ---------------------------------------------------------------------------------------
// K1: SymbolicIK.is_reachable + theta_to_joints
// ---------------------------------------------------------------------------------------
// Launched as a programmatic dependent of what precedes it on the stream (launch_pdl): back-to-back launches (two arms,
// pipeline chunks) overlap their launch latency, 0.1305 -> 0.1250 ms per 2 x 1M poses.
template <int KIND>
__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K1_MINBLOCKS)
k_symik_solve(const __grid_constant__ ArmConst A, const double *__restrict__ poses, const double *__restrict__ theta,
              const double *__restrict__ prev_joints, int64_t n, uint8_t *__restrict__ reachable,
              uint8_t *__restrict__ state, double *__restrict__ interval, double *__restrict__ joints,
              double *__restrict__ elbow) {
  // the next kernel on the stream may be scheduled as soon as every block of this one has started; this one touches
  // memory only once its own predecessor has completed
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double prev0 = 0.0, prev2 = 0.0;
  if (prev_joints) { prev0 = prev_joints[0]; prev2 = prev_joints[2]; }
  Solve S;
  const Reach rc = symik_reach<KIND>(A, poses + pose_stride(KIND) * i, S);
  if (reachable) reachable[i] = rc.state == R2IK_STATE_REACHABLE ? 1 : 0;   // nullable: state == R2IK_STATE_REACHABLE says the same (lean host record)
  state[i] = (uint8_t)rc.state;
  if (interval) { interval[2 * i] = rc.i0; interval[2 * i + 1] = rc.i1; }
  if (!joints && !elbow) return;
  double j[7], E[3];
  symik_joints(A, S, rc, theta ? theta + i : nullptr, prev0, prev2, j, E);
  if (joints) {
#pragma unroll
    for (int k = 0; k < 7; ++k) joints[7 * i + k] = j[k];
  }
  if (elbow) { elbow[3 * i] = E[0]; elbow[3 * i + 1] = E[1]; elbow[3 * i + 2] = E[2]; }
}

// ---------------------------------------------------------------------------------------
// K1-f32: the FP32 fast path of K1 (r2ik_device_f32.cuh), two kernels:
//   k_symik_solve_f32      one thread / pose: float4 / float2 pose loads (64 B per 4x4 pose, 48 B read), the FP32
//                          solve; a pose whose decisions or conditioning FP32 cannot settle is not stored but
//                          appended to a list (one atomicAdd per warp);
//   k_symik_escalated_f32  the FP64 solver on the listed poses (same float inputs widened), results narrowed.
// Keeping the FP64 solver out of the first kernel matters more than the few poses suggest: inlined behind a
// branch it cost a 130 KB kernel whose divergent excursions (7 % of the warps, one lane each) thrashed the
// instruction cache -- 125 us per 1M poses, slower than the FP64 kernel (profiles/r1_s8_symik_f32_ncu_full.txt).
// ---------------------------------------------------------------------------------------
#ifndef R2IK_K1F_MINBLOCKS
#define R2IK_K1F_MINBLOCKS 6
#endif
template <int KIND>
__device__ __forceinline__ void load_pose_f32(const float *__restrict__ poses, int64_t i, float in[12]) {
  if (KIND == R2IK_POSE_EULER6) {
    const float2 *p = reinterpret_cast<const float2 *>(poses + 6 * i);
    float2 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
    in[0] = a.x; in[1] = a.y; in[2] = b.x; in[3] = b.y; in[4] = c.x; in[5] = c.y;
  } else {
    const float4 *p = reinterpret_cast<const float4 *>(poses + 16 * i);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      float4 v = __ldg(p + r);
      in[4 * r] = v.x; in[4 * r + 1] = v.y; in[4 * r + 2] = v.z; in[4 * r + 3] = v.w;
    }
  }
}

__device__ __forceinline__ void store_pose_f32(int64_t i, int st, const float out[12], uint8_t *__restrict__ reachable,
                                               uint8_t *__restrict__ state, float *__restrict__ interval,
                                               float *__restrict__ joints, float *__restrict__ elbow) {
  reachable[i] = st == R2IK_STATE_REACHABLE ? 1 : 0;
  state[i] = (uint8_t)st;
  if (interval) reinterpret_cast<float2 *>(interval)[i] = make_float2(out[0], out[1]);
  if (joints) {
#pragma unroll
    for (int k = 0; k < 7; ++k) joints[7 * i + k] = out[2 + k];
  }
  if (elbow) { elbow[3 * i] = out[9]; elbow[3 * i + 1] = out[10]; elbow[3 * i + 2] = out[11]; }
}

// resets the escalation count (a kernel instead of a memset node, so that the three launches of a call and the last
// launch of the previous call form one chain of programmatic dependents)
__global__ void k_zero_u32(unsigned *p) {
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (threadIdx.x == 0 && blockIdx.x == 0) *p = 0u;
}

template <int KIND>
__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K1F_MINBLOCKS)
k_symik_solve_f32(const __grid_constant__ ArmConst A64, const __grid_constant__ f32::ArmConstF A,
                  const float *__restrict__ poses, const float *__restrict__ theta, int64_t n,
                  uint8_t *__restrict__ reachable, uint8_t *__restrict__ state, float *__restrict__ interval,
                  float *__restrict__ joints, float *__restrict__ elbow, uint32_t *__restrict__ esc_list,
                  unsigned *__restrict__ n_escalated) {
  asm volatile("griddepcontrol.launch_dependents;");   // k_symik_escalated_f32 may be scheduled under this kernel's tail
  asm volatile("griddepcontrol.wait;" ::: "memory");   // k_zero_u32 (and whatever preceded it) has completed
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < n;
  bool esc = false;
  float out[12];
  int st = 0;
  if (active) {
    float in[12];
    load_pose_f32<KIND>(poses, i, in);
    const bool has_theta = theta != nullptr;
    const float th = has_theta ? theta[i] : 0.0f;
    esc = f32::symik_pose_fast<KIND>(A64, A, in, has_theta, th, st, out);
  }
  // warp-aggregated append of the escalated poses
  const unsigned m = __ballot_sync(0xffffffffu, esc);
  if (m) {
    const int lane = threadIdx.x & 31;
    unsigned base = 0;
    if (lane == __ffs(m) - 1) base = atomicAdd(n_escalated, (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (esc) esc_list[base + __popc(m & ((1u << lane) - 1))] = (uint32_t)i;
  }
  if (active && !esc) store_pose_f32(i, st, out, reachable, state, interval, joints, elbow);
}

template <int KIND>
__global__ void __launch_bounds__(R2IK_BLOCK)
k_symik_escalated_f32(const __grid_constant__ ArmConst A64, const float *__restrict__ poses, const float *__restrict__ theta,
                      const float *__restrict__ prev_joints, uint8_t *__restrict__ reachable, uint8_t *__restrict__ state,
                      float *__restrict__ interval, float *__restrict__ joints, float *__restrict__ elbow,
                      const uint32_t *__restrict__ esc_list, const unsigned *__restrict__ n_escalated) {
  // launched as a programmatic dependent of k_symik_solve_f32: its blocks may be resident before that kernel has drained
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const unsigned count = *n_escalated;
  float prev0 = 0.0f, prev2 = 0.0f;
  if (prev_joints) { prev0 = prev_joints[0]; prev2 = prev_joints[2]; }
  for (unsigned k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += gridDim.x * blockDim.x) {
    const int64_t i = esc_list[k];
    float in[12], out[12];
    load_pose_f32<KIND>(poses, i, in);
    const bool has_theta = theta != nullptr;
    int st;
    f32::symik_pose_escalated<KIND>(A64, in, has_theta, has_theta ? theta[i] : 0.0f, prev0, prev2, &st, out);
    store_pose_f32(i, st, out, reachable, state, interval, joints, elbow);
  }
}

template <int KIND>
__global__ void __launch_bounds__(R2IK_BLOCK)
k_symik_no_limits(const __grid_constant__ ArmConst A, const double *__restrict__ poses, const double *__restrict__ theta,
                  const double *__restrict__ prev_joints, int prev_stride, int64_t n, double *__restrict__ joints,
                  double *__restrict__ elbow, uint8_t *__restrict__ projected) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double j[7], E[3];
  const bool proj = symik_no_limits<KIND>(A, poses + pose_stride(KIND) * i, theta + i,
                                          prev_joints ? prev_joints + (size_t)prev_stride * i : nullptr, j, E);
  for (int k = 0; k < 7; ++k) joints[7 * i + k] = j[k];
  if (elbow) { elbow[3 * i] = E[0]; elbow[3 * i + 1] = E[1]; elbow[3 * i + 2] = E[2]; }
  if (projected) projected[i] = proj ? 1 : 0;
}

template <int KIND, bool NO_LIMITS>
__global__ void __launch_bounds__(R2IK_BLOCK)
k_elbow_positions(const __grid_constant__ ArmConst A, const double *__restrict__ poses, const double *__restrict__ thetas,
                  int K, int64_t n, double *__restrict__ elbows, uint8_t *__restrict__ projected) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Solve S;
  const bool circle = pose_elbow_circle<KIND, NO_LIMITS>(A, poses + pose_stride(KIND) * i, S);
  for (int k = 0; k < K; ++k) {
    double E[3];
    const bool proj = elbow_on_circle(A, S, circle, thetas + ((size_t)i * K + k), E);
    double *o = elbows + ((size_t)i * K + k) * 3;
    o[0] = E[0]; o[1] = E[1]; o[2] = E[2];
    if (projected) projected[(size_t)i * K + k] = proj ? 1 : 0;
  }
}

// ---------------------------------------------------------------------------------------
// K1s: elbow-angle sweep, get_joints at K angles per pose from one solve of the pose.
// A block owns a tile of P poses x Kt samples (sweep_tile): threads < P solve one pose each and leave its Solve and
// Reach in shared memory, then the block walks the P * Kt items pose-major, sample-minor, so consecutive threads store
// consecutive 56-byte joint rows.  A pose whose K samples span several tiles is solved once per tile.
// ---------------------------------------------------------------------------------------
// 4 blocks / SM (128 registers, ~145 B of spills): 10-28 % faster than 2 blocks at 255 registers without spills on every
// shape of scripts/experiments/exp_sweep.py (profiles/r3_exp_sweep*.txt)
#ifndef R2IK_K1S_MINBLOCKS
#define R2IK_K1S_MINBLOCKS 4
#endif
template <int KIND, bool NO_LIMITS>
__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K1S_MINBLOCKS)
k_symik_sweep(const __grid_constant__ ArmConst A, const double *__restrict__ poses, int64_t n, const double *__restrict__ thetas,
              int theta_stride, int K, int P, int Kt, int n_ktiles, const double *__restrict__ prev_joints,
              uint8_t *__restrict__ state, double *__restrict__ interval, double *__restrict__ thetas_used,
              double *__restrict__ joints, double *__restrict__ elbow, uint8_t *__restrict__ projected) {
  __shared__ Solve sS[R2IK_BLOCK];
  __shared__ Reach sR[R2IK_BLOCK];
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  double prev0 = 0.0, prev2 = 0.0;
  if (prev_joints) { prev0 = prev_joints[0]; prev2 = prev_joints[2]; }
  const int64_t p0 = (int64_t)(blockIdx.x / n_ktiles) * P;
  const int kt = (int)(blockIdx.x % n_ktiles), k0 = kt * Kt;
  const int np = (int)min((int64_t)P, n - p0), nk = min(Kt, K - k0);
  if (threadIdx.x < np) {
    const int64_t i = p0 + threadIdx.x;
    Solve S;
    const Reach rc = symik_reach<KIND, NO_LIMITS>(A, poses + pose_stride(KIND) * i, S);
    sS[threadIdx.x] = S;
    sR[threadIdx.x] = rc;
    if (kt == 0) {
      state[i] = (uint8_t)rc.state;
      if (interval) { interval[2 * i] = rc.i0; interval[2 * i + 1] = rc.i1; }
    }
  }
  __syncthreads();
  for (int f = threadIdx.x; f < np * nk; f += blockDim.x) {
    const int p = f / nk, k = k0 + (f - p * nk);
    const int64_t i = p0 + p;
    const Reach rc = sR[p];
    const double th = sweep_theta(rc, thetas ? thetas + (size_t)theta_stride * i : nullptr, K, k);
    double j[7], E[3];
    const bool proj = sweep_sample(A, sS[p], rc, th, prev0, prev2, j, E);
    const size_t o = (size_t)i * K + k;
#pragma unroll
    for (int q = 0; q < 7; ++q) joints[7 * o + q] = j[q];
    if (elbow) { elbow[3 * o] = E[0]; elbow[3 * o + 1] = E[1]; elbow[3 * o + 2] = E[2]; }
    if (thetas_used) thetas_used[o] = th;
    if (projected) projected[o] = proj ? 1 : 0;
  }
}

// The reference's scalar call sequence in ONE launch of one thread: is_reachable (or is_reachable_no_limits), then
// get_elbow_position(theta) and get_joints(theta, previous_joints).  The query travels as a kernel parameter (no
// input buffer) and the record may live in mapped pinned host memory, so a scalar facade call is one launch + one
// stream synchronisation (the consumer of the reference calls it once per control tick, src/example/example_control.py:9-27).
template <bool NO_LIMITS>
__device__ __forceinline__ void scalar_body(const ArmConst &A, const R2ikScalarQuery &q, R2ikScalarResult &r) {
  const double pos[3] = {q.goal_pose[0], q.goal_pose[1], q.goal_pose[2]};
  Solve S;
  rot_from_euler_xyz(q.goal_pose[3], q.goal_pose[4], q.goal_pose[5], S.R);
  // the pre-checked position is what the reference stores in self.goal_pose (sik:143); is_reachable_R recomputes it
  const Reach rc = is_reachable_R<NO_LIMITS>(A, pos, S);
  r.state = rc.state;
  r.reachable = rc.state == R2IK_STATE_REACHABLE ? 1 : 0;
  const bool attrs = NO_LIMITS || rc.state == R2IK_STATE_REACHABLE || rc.state == R2IK_STATE_LIMITED_BY_WRIST ||
                     rc.state == R2IK_STATE_WRIST_OUT_OF_RANGE || rc.state == R2IK_STATE_SHOULD_NOT_HAPPEN;
  if (attrs) {
    for (int k = 0; k < 3; ++k) { r.goal_position_solved[k] = S.p[k]; r.wrist_position_solved[k] = S.w[k]; }
  }
  if (r.reachable) { r.interval[0] = rc.i0; r.interval[1] = rc.i1; }
  const bool circle = r.reachable || (!NO_LIMITS && rc.state == R2IK_STATE_LIMITED_BY_WRIST);
  if (circle && (q.has_theta || r.reachable)) {
    double st = rc.s0, ct = rc.c0;
    if (q.has_theta) sincos_any(q.theta, st, ct);
    elbow_position_cs(S, ct, st, r.elbow_on_circle);
    if (r.reachable) {
      r.projected = elbow_projection_fires(A, r.elbow_on_circle) ? 1 : 0;
      get_joints_cs(A, S, ct, st, q.previous_joints[0], q.previous_joints[2], r.joints, r.elbow);
      for (int k = 0; k < 3; ++k) { r.goal_position[k] = S.p[k]; r.wrist_position[k] = S.w[k]; }
    }
  }
}

__global__ void __launch_bounds__(32)
k_symik_scalar(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikScalarQuery q, R2ikScalarResult *__restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  R2ikScalarResult r;
  r.interval[0] = NAN; r.interval[1] = NAN;
  for (int k = 0; k < 7; ++k) r.joints[k] = NAN;
  for (int k = 0; k < 3; ++k) {
    r.elbow[k] = NAN; r.elbow_on_circle[k] = NAN; r.goal_position_solved[k] = NAN; r.wrist_position_solved[k] = NAN;
    r.goal_position[k] = NAN; r.wrist_position[k] = NAN;
  }
  r.reachable = 0; r.state = 0; r.projected = 0; r.reserved = 0;
  if (q.no_limits) scalar_body<true>(A, q, r);
  else scalar_body<false>(A, q, r);
  *out = r;
}

// ControlIK.__init__'s seed of previous_theta (ctl_ctor_theta).  One thread; arguments by value; result to any
// device-accessible address.
struct CtorThetaArgs { double rows[49]; double current_pose[16]; double preferred_theta; int n_rows; int pad; };
__global__ void __launch_bounds__(32)
k_ctl_ctor_theta(const __grid_constant__ ArmConst A, const __grid_constant__ CtorThetaArgs a, double *__restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  out[0] = ctl_ctor_theta(A, a.current_pose, a.rows, a.n_rows, a.preferred_theta);
}

// ---------------------------------------------------------------------------------------
// K2: ControlIK discrete mode, two forms with identical results.
//
// k_ctl_discrete (default): one lane / pose end to end.  The K-sample search of get_best_discrete_theta
// (utl:366-390) is replaced by search_analytic (r2ik_control.cuh): the arg-min over the K samples is found
// among 17 candidate samples located from the crossings of the two elbow half-plane tests, each evaluated
// exactly like a visited sample -- the cost of a pose no longer depends on K.
//
// k_ctl_discrete_scan: the exhaustive form.  Each lane solves its own pose (is_reachable, preferred-theta
// shortcut); poses that need the K-sample search are then served one at a time by the whole
// warp: the circle is broadcast with shuffles, lane l evaluates samples l, l+32, ..., and a
// shuffle arg-min with lowest-index tie-break reproduces the reference's strict-< scan
// (utl:381-390).  Each lane finally runs get_joints + safety_checks for its own pose.  Kept as the
// cross-check of the analytic search (tests compare the two on every sampled pose) and for K < 8.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// The scan form spends most of its time in the warp-serial K-sample search, a short dependent chain per lane that
// only more resident warps can overlap: holding the kernel to 64 registers (8 blocks / SM; the solve
// phases spill ~1.1 KB to L1-resident local memory) measured 0.89 ms per 1M poses x 360 samples against
// 1.18 ms at 128 registers and 1.77 ms unconstrained (176 registers), profiles/r1_experiments.md.
#ifndef R2IK_K2_MINBLOCKS
#define R2IK_K2_MINBLOCKS 8
#endif
__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K2_MINBLOCKS)
k_ctl_discrete_scan(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikCtlParams par,
               const double *__restrict__ M, int64_t n, const double *__restrict__ prev_joints,
               const double *__restrict__ current_joints, double *__restrict__ joints, uint8_t *__restrict__ reachable,
               uint8_t *__restrict__ state, uint8_t *__restrict__ emergency) {
  const int lane = threadIdx.x & 31;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < n;
  double prev[7], cur[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) { prev[k] = prev_joints[k]; cur[k] = current_joints[k]; }

  Solve S;
  int st = R2IK_STATE_INVALID_ROTATION;
  bool found = false, need_search = false, valid_pose = false;
  double theta = 0.0;
  const int nb = par.nb_search_points;
  SearchPlan plan;
  if (active) {
    Reach rc;
    valid_pose = disc_classify(A, par, M + 16 * i, S, rc, found, need_search);
    st = rc.state;
    if (found) theta = par.preferred_theta;
    if (need_search) plan = disc_search_plan(A, par, S, rc);
  }
  unsigned pending = __ballot_sync(0xffffffffu, need_search);
  while (pending) {
    const int src = __ffs(pending) - 1;
    pending &= pending - 1;
    SearchPlan B;   // the plan of lane `src`, broadcast
    B.preferred_theta = par.preferred_theta;
    B.L.div = nb - 1;
    B.L.start = shfl_d(plan.L.start, src); B.L.stop = shfl_d(plan.L.stop, src);
    B.L.delta = shfl_d(plan.L.delta, src); B.L.step = shfl_d(plan.L.step, src);
    B.T.A1 = shfl_d(plan.T.A1, src); B.T.B1 = shfl_d(plan.T.B1, src); B.T.C1 = shfl_d(plan.T.C1, src);
    B.T.A2 = shfl_d(plan.T.A2, src); B.T.B2 = shfl_d(plan.T.B2, src); B.T.C2 = shfl_d(plan.T.C2, src);
    double best;
    int best_k;
    search_strided(B, nb, lane, 32, best, best_k);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      double ob = __shfl_xor_sync(0xffffffffu, best, off);
      int ok = __shfl_xor_sync(0xffffffffu, best_k, off);
      if (ob < best || (ob == best && ok < best_k)) { best = ob; best_k = ok; }
    }
    if (lane == src) {
      found = best < INFINITY;
      if (found) theta = linspace_value(plan.L, best_k);
      else st = R2IK_STATE_LIMITED_BY_SHOULDER;
    }
  }
  if (!active) return;
  double j[7];
  int bits = 0;
  if (valid_pose) {
    bits = discrete_finish(A, par, S, found, theta, prev, cur, j);
  } else {
#pragma unroll
    for (int k = 0; k < 7; ++k) j[k] = NAN;
  }
#pragma unroll
  for (int k = 0; k < 7; ++k) joints[7 * i + k] = j[k];
  reachable[i] = found ? 1 : 0;
  state[i] = (uint8_t)st;
  if (emergency) emergency[i] = (uint8_t)bits;
}

#ifndef R2IK_K2A_MINBLOCKS
#define R2IK_K2A_MINBLOCKS 8
#endif
__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K2A_MINBLOCKS)
k_ctl_discrete(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikCtlParams par,
               const double *__restrict__ M, int64_t n, const double *__restrict__ prev_joints,
               const double *__restrict__ current_joints, double *__restrict__ joints, uint8_t *__restrict__ reachable,
               uint8_t *__restrict__ state, uint8_t *__restrict__ emergency) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned wmask = __ballot_sync(0xffffffffu, i < n);
  if (i >= n) return;
  double prev[7], cur[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) { prev[k] = prev_joints[k]; cur[k] = current_joints[k]; }
  Solve S;
  Reach rc;
  bool found, need_search;
  double theta = 0.0, j[7];
  int bits = 0;
  // The three sections below are kept apart by warp barriers: without them the compiler threads the preferred-theta
  // and the search paths separately through their own copies of the tail (get_joints + safety chain), and a warp runs
  // that tail twice at half the lanes (ncu: get_joints at 10 of 32 lanes for 64 % of the poses found).
  const bool valid = disc_classify(A, par, M + 16 * i, S, rc, found, need_search);
  int st = rc.state;
  if (found) theta = par.preferred_theta;
  __syncwarp(wmask);
  if (need_search) {
    found = disc_search(disc_search_plan(A, par, S, rc), par.nb_search_points, theta);
    if (!found) st = R2IK_STATE_LIMITED_BY_SHOULDER;
  }
  __syncwarp(wmask);
  if (valid) {
    bits = discrete_finish(A, par, S, found, theta, prev, cur, j);
  } else {
#pragma unroll
    for (int k = 0; k < 7; ++k) j[k] = NAN;
  }
#pragma unroll
  for (int k = 0; k < 7; ++k) joints[7 * i + k] = j[k];
  reachable[i] = found ? 1 : 0;
  state[i] = (uint8_t)st;
  if (emergency) emergency[i] = (uint8_t)bits;
}

// ---------------------------------------------------------------------------------------
// K3: ControlIK continuous mode.  A trajectory is a sequential recursion over its waypoints
// (previous_theta / previous_sol / init / emergency latch), so one thread owns one trajectory
// and keeps the controller state in registers; parallelism comes from the trajectories.
// ---------------------------------------------------------------------------------------
// Launch shape of K3: 65 536 trajectories are only 2 048 warps, 13.8 per SM.  Blocks of 64 threads held
// to 128 registers (7 blocks = 14 warps per SM) make the whole batch resident in one wave and spread
// it evenly over the 148 SMs; the unconstrained allocation (240 registers, 8 warps / SM) needed two
// waves, the second 73 % full: 49 ms vs 32 ms for cfg 4 (profiles/r1_experiments.md).
#ifndef R2IK_K3_BLOCK
#define R2IK_K3_BLOCK 64
#endif
#ifndef R2IK_K3_MINBLOCKS
#define R2IK_K3_MINBLOCKS 7
#endif
__global__ void __launch_bounds__(R2IK_K3_BLOCK, R2IK_K3_MINBLOCKS)
k_ctl_continuous(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikCtlParams par,
                 const double *__restrict__ M, int64_t T, int W, const double *__restrict__ current_joints,
                 const double *__restrict__ current_pose, R2ikTrajState *__restrict__ states,
                 double *__restrict__ joints, uint8_t *__restrict__ reachable, uint8_t *__restrict__ state) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  R2ikTrajState cs = states[t];
  double cj[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) cj[k] = current_joints[7 * t + k];
  for (int w = 0; w < W; ++w) {
    size_t k = (size_t)t * W + w;
    double m[16], cp[16];
    load_mat4(M + 16 * k, m);
    if (!cs.has_previous_sol && !cs.emergency_stop) load_mat4(current_pose + 16 * t, cp);
    double j[7];
    uint8_t r, s;
    continuous_step(A, par, m, cj, cp, cs, j, r, s);
#pragma unroll
    for (int q = 0; q < 7; ++q) joints[7 * k + q] = j[q];
    reachable[k] = r;
    state[k] = s;
  }
  states[t] = cs;
}

// ---------------------------------------------------------------------------------------
// K3, phased form (needs 10 bytes of workspace per waypoint).  See r2ik_control.cuh "Continuous mode, cut at its
// data dependences" and r2ik_cont_codes.cuh:
//   k_cont_targets           1 thread / waypoint    classify + target theta                       -> code, state, ws = goal
//   k_cont_thetas            1 thread / trajectory  rate-limited theta scan (tiles through shared memory) -> ws = theta
//   k_cont_raw_joints_codes  1 thread / waypoint    get_joints(theta) + Orbita3D limit, winding code against the predecessor
//                                                                                                 -> joints (raw), codes16, reachable
//   k_cont_finish_codes      1 thread / trajectory  unwrap / continuity / emergency scan on the 16-bit codes; the reference's
//                                                   statements verbatim on irregular waypoints    -> codes16 (absolute windings),
//                                                                                                    joints / state where irregular, states
//   k_cont_apply_windings    1 thread / 8 waypoints j + 2 pi k on the wound rows                  -> joints
// The two per-waypoint kernels hold ~95 % of the arithmetic and run at full parallelism (T x W threads); the scans are a
// 1 000-step recursion per trajectory that only all trajectories in flight at once can hide.  `reachable` carries the
// waypoint code and `state` the reference state between the phases.
// ---------------------------------------------------------------------------------------
#ifndef R2IK_K3T_MINBLOCKS
#define R2IK_K3T_MINBLOCKS 6    // 80 registers: 4 / 5 (96 registers) / 6 / 7 / 8 blocks -> 7.70 / 7.71 / 7.51 / 7.58 / 7.63 ms for cfg 4 (s46)
#endif
__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K3T_MINBLOCKS)
k_cont_targets(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikCtlParams par, const double *__restrict__ M,
               int64_t n_wp, double *__restrict__ ws, uint8_t *__restrict__ code, uint8_t *__restrict__ state) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_wp) return;
  double m[16], pos[3], goal;
  load_mat4(M + 16 * k, m);
  Solve S;
  int st;
  const int c = cont_target(A, par, m, S, pos, goal, st);
  ws[k] = goal;
  code[k] = (uint8_t)c;
  state[k] = (uint8_t)st;
}

// The theta scan walks each trajectory's row in order, one thread per trajectory: read directly, every warp request
// touches 32 different sectors (the rows of 32 trajectories are W waypoints apart; ncu on the first form of the
// scans: 35.7 GB between L1 and L2 for 7.3 GB of payload, long_scoreboard 11 cycles per issue,
// profiles/r1_s16_continuous_ncu_full.txt).  It therefore moves tiles of (block trajectories) x 8 waypoints
// through shared memory with cooperative, row-contiguous loads and stores; each thread then walks its own row of the
// tile.  Row stride 9 doubles: bank-conflict free for the 64-bit accesses of a half warp.  1.33 -> 1.05 ms for cfg 4.
#define R2IK_TH_TILE 8    // waypoints per tile of the theta scan (64 B of thetas per trajectory)

__global__ void __launch_bounds__(R2IK_K3_BLOCK, R2IK_K3_MINBLOCKS)
k_cont_thetas(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikCtlParams par, int64_t T, int W,
              const double *__restrict__ current_joints, const double *__restrict__ current_pose,
              const R2ikTrajState *__restrict__ states, double *__restrict__ ws, const uint8_t *__restrict__ code) {
  __shared__ double s_th[R2IK_K3_BLOCK][R2IK_TH_TILE + 1];
  __shared__ uint8_t s_code[R2IK_K3_BLOCK][R2IK_TH_TILE];
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x;
  const int64_t t = t0 + threadIdx.x;
  const bool live = t < T && !states[t].emergency_stop;   // a latched trajectory answers every waypoint with its solution
  double theta = 0.0;
  bool has = false;
  if (live) { theta = states[t].previous_theta; has = states[t].has_previous_sol != 0; }
  for (int w0 = 0; w0 < W; w0 += R2IK_TH_TILE) {
    const int nw = min(R2IK_TH_TILE, W - w0);
    for (int f = threadIdx.x; f < R2IK_K3_BLOCK * R2IK_TH_TILE; f += R2IK_K3_BLOCK) {
      const int r = f / R2IK_TH_TILE, e = f % R2IK_TH_TILE;
      if (t0 + r < T && e < nw) {
        const size_t g = (size_t)(t0 + r) * W + w0 + e;
        s_th[r][e] = ws[g];
        s_code[r][e] = code[g];
      }
    }
    __syncthreads();
    if (live) {
      for (int e = 0; e < nw; ++e) {
        const int c = s_code[threadIdx.x][e];
        if (c == R2IK_WP_INVALID) continue;
        if (!has) {                                                // ctl:306-325, at the first valid waypoint
          double cj[7], cp[16];
#pragma unroll
          for (int q = 0; q < 7; ++q) cj[q] = current_joints[7 * t + q];
          load_mat4(current_pose + 16 * t, cp);
          theta = cont_initial_theta(A, par, cj, cp);
          has = true;
        }
        theta = cont_next_theta(par, c, s_th[threadIdx.x][e], theta);
        s_th[threadIdx.x][e] = theta;
      }
    }
    __syncthreads();
    for (int f = threadIdx.x; f < R2IK_K3_BLOCK * R2IK_TH_TILE; f += R2IK_K3_BLOCK) {
      const int r = f / R2IK_TH_TILE, e = f % R2IK_TH_TILE;
      if (t0 + r < T && e < nw) ws[(size_t)(t0 + r) * W + w0 + e] = s_th[r][e];
    }
    __syncthreads();
  }
}

#include "r2ik_cont_codes.cuh"
#include "r2ik_discrete_compact.cuh"

// ---------------------------------------------------------------------------------------
// K4: workspace reachability map.  One thread per voxel.  Voxels outside the reach sphere or behind the torso plane
// leave before the orientation loop (those two states do not depend on the orientation, sik:284-307), and a block
// without a live voxel (3/4 of the bounding cube) leaves before staging anything.
//
// Per (voxel, orientation) pair only a flag is needed.  k_reach_map decides it with reach_flag_mixed
// (r2ik_device_f32.cuh): what depends on the orientation alone (R wo and the limit-plane normal) is staged once per
// block in shared memory, the cancelling front end of a pair runs in FP64 (~15 operations) and the in-plane linking
// test in FP32; a pair within the FP32 error bands of a decision (3e-4 of them) is decided by the FP64 flag solve,
// so the counts are those of the all-FP64 kernel k_reach_map_f64 (kept: tests compare the two volumes).
// ---------------------------------------------------------------------------------------
// Orientations staged at once.  In the FP64 kernel, 64 meant two block barriers per chunk and `barrier` as the first
// stall reason (4.3 cycles per issue: voxels of a block leave the solve at different depths); 512 = the whole
// orientation set of cfg 5 (36 KB of rotation matrices / 20 KB of OriConst), two barriers per block.
#ifndef R2IK_ORI_CHUNK
#define R2IK_ORI_CHUNK 512
#endif

__device__ __forceinline__ bool voxel_live(const ArmConst &A, int64_t v, int64_t nv, double ox, double oy, double oz, double sx,
                                           double sy, double sz, int d1, int d2, double &px, double &py, double &pz) {
  px = 0; py = 0; pz = 0;
  if (v >= nv) return false;
  int ix, iy, iz;
  if (nv <= 0x7fffffffLL) {      // 32-bit index arithmetic whenever the volume allows it (the 64-bit divisions are emulated)
    const unsigned u = (unsigned)v, row = u / (unsigned)d2;
    iz = (int)(u - row * (unsigned)d2);
    ix = (int)(row / (unsigned)d1);
    iy = (int)(row - (unsigned)ix * (unsigned)d1);
  } else {
    iz = (int)(v % d2);
    iy = (int)((v / d2) % d1);
    ix = (int)(v / ((int64_t)d2 * d1));
  }
  px = ox + ix * sx; py = oy + iy * sy; pz = oz + iz * sz;
  return reach_prechecks(A, px, py, pz) < 0;
}

// CT = uint32_t, or uint16_t for the sharded map: orientation shards of at most 65 535 orientations sum without a carry
// when two 16-bit counts travel in one 32-bit lane of the all-reduce.  [v_begin, nv) = the voxel range of this launch
// (slabs of the volume are launched one after the other so that the reduction of one overlaps the kernel of the next).
template <typename CT>
__global__ void __launch_bounds__(R2IK_BLOCK)
k_reach_map(const __grid_constant__ ArmConst A, const __grid_constant__ f32::ArmConstF AF, double ox, double oy, double oz,
            double sx, double sy, double sz, int d0, int d1, int d2, const double *__restrict__ ori_euler, int ori_begin,
            int ori_end, int64_t v_begin, int64_t nv, int row_mod, int row_rem, CT *__restrict__ counts) {
  __shared__ f32::OriConst sO[R2IK_ORI_CHUNK];
  int64_t v = v_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row_mod > 1) {
    // interleaved sharding: of the rows (ix, iy, :) of [v_begin, nv) this launch owns those with row % row_mod == row_rem
    // (v_begin is row-aligned); the launch index enumerates the owned rows densely
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t row0 = v_begin / d2;
    const int64_t first = row0 + ((row_rem - row0 % row_mod) + row_mod) % row_mod;
    v = (first + (u / d2) * row_mod) * d2 + u % d2;
  }
  double px, py, pz;
  const bool live = voxel_live(A, v, nv, ox, oy, oz, sx, sy, sz, d1, d2, px, py, pz);
  if (!__syncthreads_or(live ? 1 : 0)) {
    if (v < nv) counts[v] = 0;
    return;
  }
  const double ps[3] = {px - A.s[0], py - A.s[1], pz - A.s[2]};
  uint32_t count = 0;
  for (int base = ori_begin; base < ori_end; base += R2IK_ORI_CHUNK) {
    const int m = min(R2IK_ORI_CHUNK, ori_end - base);
    if (base != ori_begin) __syncthreads();
    for (int o = threadIdx.x; o < m; o += blockDim.x) {
      const double *e = ori_euler + 3 * (size_t)(base + o);
      double R[9];
      rot_from_euler_xyz(e[0], e[1], e[2], R);
      sO[o] = f32::make_ori_const(A, R);
    }
    __syncthreads();
    if (live) {
      for (int o = 0; o < m; ++o) {
        bool esc;   // too close to call in FP32: 3e-4 of the pairs
        const int st = f32::reach_pair(A, AF, ps, px, py, pz, sO[o], ori_euler + 3 * (size_t)(base + o), esc);
        count += (st == R2IK_STATE_REACHABLE) ? 1u : 0u;
      }
    }
  }
  if (v < nv) counts[v] = (CT)count;
}

// The all-FP64 form (every pair through solve_core<false, true>): the cross-check of k_reach_map.
__global__ void __launch_bounds__(R2IK_BLOCK)
k_reach_map_f64(const __grid_constant__ ArmConst A, double ox, double oy, double oz, double sx, double sy, double sz,
                int d0, int d1, int d2, const double *__restrict__ ori_euler, int ori_begin, int ori_end,
                uint32_t *__restrict__ counts) {
  __shared__ double sR[R2IK_ORI_CHUNK][9];
  const int64_t nv = (int64_t)d0 * d1 * d2;
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double px, py, pz;
  const bool live = voxel_live(A, v, nv, ox, oy, oz, sx, sy, sz, d1, d2, px, py, pz);
  if (!__syncthreads_or(live ? 1 : 0)) {
    if (v < nv) counts[v] = 0;
    return;
  }
  uint32_t count = 0;
  for (int base = ori_begin; base < ori_end; base += R2IK_ORI_CHUNK) {
    int m = min(R2IK_ORI_CHUNK, ori_end - base);
    if (base != ori_begin) __syncthreads();
    for (int o = threadIdx.x; o < m; o += blockDim.x) {
      const double *e = ori_euler + 3 * (size_t)(base + o);
      double R[9];
      rot_from_euler_xyz(e[0], e[1], e[2], R);
#pragma unroll
      for (int k = 0; k < 9; ++k) sR[o][k] = R[k];
    }
    __syncthreads();
    if (live) {
      for (int o = 0; o < m; ++o) {
        Solve S;
        S.p[0] = px; S.p[1] = py; S.p[2] = pz;
#pragma unroll
        for (int k = 0; k < 9; ++k) S.R[k] = sR[o][k];
        Reach rc = solve_core<false, true>(A, S);
        count += (rc.state == R2IK_STATE_REACHABLE) ? 1u : 0u;
      }
    }
  }
  if (v < nv) counts[v] = count;
}

// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void affine_mul(double A[12], const double B[12]) {
  double o[12];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      double v = A[4 * r] * B[c] + A[4 * r + 1] * B[4 + c] + A[4 * r + 2] * B[8 + c];
      if (c == 3) v += A[4 * r + 3];
      o[4 * r + c] = v;
    }
  }
#pragma unroll
  for (int k = 0; k < 12; ++k) A[k] = o[k];
}

__global__ void __launch_bounds__(R2IK_BLOCK)
k_fk(const __grid_constant__ R2ikFkChain ch, const double *__restrict__ joints, int64_t n, double *__restrict__ M) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double T[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    affine_mul(T, ch.fixed[k]);
    double s, c;
    sincos(joints[7 * i + k], &s, &c);
    const double ax = ch.axis[k][0], ay = ch.axis[k][1], az = ch.axis[k][2], v = 1.0 - c;
    // R = I + sin q K + (1 - cos q) K^2
    double Rj[12] = {1.0 - v * (ay * ay + az * az), -s * az + v * ax * ay, s * ay + v * ax * az, 0.0,
                     s * az + v * ax * ay, 1.0 - v * (ax * ax + az * az), -s * ax + v * ay * az, 0.0,
                     -s * ay + v * ax * az, s * ax + v * ay * az, 1.0 - v * (ax * ax + ay * ay), 0.0};
    affine_mul(T, Rj);
  }
  affine_mul(T, ch.fixed[7]);
  double2 *o = reinterpret_cast<double2 *>(M + 16 * i);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    o[2 * r] = make_double2(T[4 * r], T[4 * r + 1]);
    o[2 * r + 1] = make_double2(T[4 * r + 2], T[4 * r + 3]);
  }
  o[6] = make_double2(0.0, 0.0);
  o[7] = make_double2(0.0, 1.0);
}

// ---------------------------------------------------------------------------------------
// FP64 FMA peak probe (roofline denominator for bench.py; MEASURED_PEAKS.json has no FP64 entry)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dfma_probe(int iters, double seed, double *sink) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 0.999999, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 123.456) sink[0] = s;  // never true: keeps the chains alive
}

// FP32 counterpart (roofline denominator of K1-f32)
__global__ void __launch_bounds__(256) k_ffma_probe(int iters, float seed, float *sink) {
  float a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const float m = 0.999999f, c = 1e-9f;
  for (int i = 0; i < iters; ++i) {
    a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
    a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
  }
  float s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 123.456f) sink[0] = s;
}

// ---------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------
struct r2ik_context {
  int device;
  R2ikArmConfig cfg;
  ArmConst A;
  f32::ArmConstF AF;   // A narrowed to float for K1-f32
  R2ikArmConstants pub;
};

static thread_local char g_err[256] = "";

static int fail_arg(int code, const char *msg) {
  snprintf(g_err, sizeof g_err, "%s", msg);
  return code;
}
static int fail_cuda(cudaError_t e, const char *where) {
  snprintf(g_err, sizeof g_err, "%s: %s", where, cudaGetErrorString(e));
  return -(int)e;
}
#define R2IK_CUDA(call, where)                        \
  do {                                                \
    cudaError_t e_ = (call);                          \
    if (e_ != cudaSuccess) return fail_cuda(e_, where); \
  } while (0)

// Every entry runs on its handle's device and leaves the calling thread's current device as it found it (the caller --
// torch, or any other runtime user in the process -- keeps its own notion of the current device).
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
    else if (err == cudaSuccess) prev = -1;     // nothing to restore
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

static inline bool misaligned16(const void *p) { return ((uintptr_t)p & 15) != 0; }
static inline unsigned blocks_for(int64_t n) { return (unsigned)((n + R2IK_BLOCK - 1) / R2IK_BLOCK); }

// Tile of k_symik_sweep: Kt samples of each of P poses, about 1024 items (8 per thread).  Few angles per pose: P = 128,
// every thread solves a pose.  Many angles: fewer poses per tile, and while the grid would leave the 148 SMs short of
// 8 tiles each the samples of a pose are split over more tiles (down to 128 samples a tile), each of which solves the
// pose again.
static void sweep_tile(int64_t n, int K, int &P, int &Kt) {
  constexpr int kItems = 1024, kMinKt = 128;
  constexpr int64_t kFullGrid = 148 * 8;
  Kt = K < kItems ? K : kItems;
  P = kItems / Kt < R2IK_BLOCK ? kItems / Kt : R2IK_BLOCK;
  while (Kt > kMinKt && (n + P - 1) / P * ((K + Kt - 1) / Kt) < kFullGrid) Kt = (Kt + 1) / 2;
}

// Launch as a programmatic dependent of the preceding work on the stream: the kernel's blocks may be scheduled under its
// predecessor's tail, and the kernel waits (griddepcontrol.wait) before it touches memory.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, cudaStream_t s, Args... args) {
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.stream = s;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

extern "C" {

int r2ik_abi_version(void) { return R2IK_ABI_VERSION; }
const char *r2ik_last_error(void) { return g_err; }

int r2ik_create(const R2ikArmConfig *cfg, int device, r2ik_handle *out) {
  if (!cfg || !out) return fail_arg(R2IK_ERR_NULL, "r2ik_create: null argument");
  if (cfg->side != 1 && cfg->side != -1) return fail_arg(R2IK_ERR_ARM, "r2ik_create: side must be +1 (r_arm) or -1 (l_arm)");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess) return fail_cuda(e, "cudaGetDeviceCount");
  if (count == 0 || device < 0 || device >= count) return fail_arg(R2IK_ERR_NO_DEVICE, "r2ik_create: no such CUDA device");
  r2ik_context *h = new (std::nothrow) r2ik_context;
  if (!h) return fail_arg(R2IK_ERR_ARG, "r2ik_create: out of host memory");
  h->device = device;
  h->cfg = *cfg;
  derive_constants(*cfg, h->A, h->pub);
  f32::narrow_constants(h->A, h->AF);
  *out = h;
  return 0;
}

int r2ik_destroy(r2ik_handle h) {
  delete h;
  return 0;
}

int r2ik_get_constants(r2ik_handle h, R2ikArmConstants *out) {
  if (!h || !out) return fail_arg(R2IK_ERR_NULL, "r2ik_get_constants: null argument");
  *out = h->pub;
  return 0;
}

int r2ik_interval_limit(int side, int low_elbow, double *out) {
  if (!out) return fail_arg(R2IK_ERR_NULL, "r2ik_interval_limit: null argument");
  // ctl:225-252
  double il0 = low_elbow ? -4 * kPi / 5 : 3 * kPi / 4;
  double il1 = low_elbow ? 0.0 : -2 * kPi / 6;
  if (side < 0) {
    double a = -kPi - il1, b = -kPi - il0;
    il0 = a; il1 = b;
    if (il0 < -kPi) il0 = pymod(il0, kTwoPi);
    if (il1 < -kPi) il1 = pymod(il1, kTwoPi);
    if (il0 > kPi) il0 = pymod(il0, -kTwoPi);
    if (il1 > kPi) il1 = pymod(il1, -kTwoPi);
  }
  out[0] = il0; out[1] = il1;
  return 0;
}

int r2ik_symik_solve_f64(r2ik_handle h, int pose_kind, const double *poses, const double *theta, const double *prev_joints,
                         int64_t n, uint8_t *reachable, uint8_t *state, double *interval, double *joints, double *elbow,
                         void *stream) {
  if (n < 0 || (pose_kind != R2IK_POSE_EULER6 && pose_kind != R2IK_POSE_MAT4 && pose_kind != R2IK_POSE_MAT34))
    return fail_arg(R2IK_ERR_ARG, "r2ik_symik_solve_f64: bad n or pose_kind");
  if (!h) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_solve_f64: null handle");
  if (n == 0) return 0;  // empty batch: nothing to read or write
  if (!poses || !state) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_solve_f64: null argument");
  if (misaligned16(poses)) return fail_arg(R2IK_ERR_ARG, "r2ik_symik_solve_f64: poses must be 16-byte aligned");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned g = blocks_for(n);
  cudaError_t e;
  if (pose_kind == R2IK_POSE_MAT4)
    e = launch_pdl(k_symik_solve<R2IK_POSE_MAT4>, g, R2IK_BLOCK, s, h->A, poses, theta, prev_joints, n, reachable, state, interval, joints, elbow);
  else if (pose_kind == R2IK_POSE_MAT34)
    e = launch_pdl(k_symik_solve<R2IK_POSE_MAT34>, g, R2IK_BLOCK, s, h->A, poses, theta, prev_joints, n, reachable, state, interval, joints, elbow);
  else
    e = launch_pdl(k_symik_solve<R2IK_POSE_EULER6>, g, R2IK_BLOCK, s, h->A, poses, theta, prev_joints, n, reachable, state, interval, joints, elbow);
  R2IK_CUDA(e, "k_symik_solve launch");
  R2IK_CUDA(cudaGetLastError(), "k_symik_solve launch");
  return 0;
}

int r2ik_symik_solve_f32(r2ik_handle h, int pose_kind, const float *poses, const float *theta, const float *prev_joints,
                         int64_t n, uint8_t *reachable, uint8_t *state, float *interval, float *joints, float *elbow,
                         uint32_t *escalated_idx, uint32_t *n_escalated, void *stream) {
  if (n < 0 || n > 0xffffffffLL || (pose_kind != R2IK_POSE_EULER6 && pose_kind != R2IK_POSE_MAT4))
    return fail_arg(R2IK_ERR_ARG, "r2ik_symik_solve_f32: bad n (0 .. 2^32-1) or pose_kind");
  if (!h) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_solve_f32: null handle");
  if (n == 0) {   // the contract "the call sets n_escalated" holds for an empty batch too
    if (n_escalated) {
      DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
      R2IK_CUDA(cudaMemsetAsync(n_escalated, 0, sizeof(uint32_t), (cudaStream_t)stream), "cudaMemsetAsync");
    }
    return 0;
  }
  if (!poses || !reachable || !state || !escalated_idx || !n_escalated)
    return fail_arg(R2IK_ERR_NULL, "r2ik_symik_solve_f32: null argument");
  if (((uintptr_t)poses & (pose_kind == R2IK_POSE_MAT4 ? 15 : 7)) != 0 || ((uintptr_t)interval & 7) != 0)
    return fail_arg(R2IK_ERR_ARG, "r2ik_symik_solve_f32: poses must be 16-byte (MAT4) / 8-byte (EULER6) aligned, interval 8-byte aligned");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaStream_t s = (cudaStream_t)stream;
  // second pass: a fixed grid striding over the (device-side) count -- a few percent of the poses.  One-warp blocks: the
  // FP64 solver takes 188 registers (10 warps / SM), and 46 k escalated poses per million are 1 438 warps -- as blocks of
  // 32 threads they are all resident in one wave, as blocks of 128 they needed two (296 of 360 blocks at a time).
  const int64_t ew = (n + 31) / 32;
  const unsigned eb = (unsigned)(ew < 2368 ? ew : 2368);
  // count reset, first pass and second pass are a chain of programmatic dependents: each is scheduled under its
  // predecessor's tail and waits (griddepcontrol.wait) before it touches memory
  R2IK_CUDA(launch_pdl(k_zero_u32, 1, 32, s, n_escalated), "k_zero_u32 launch");
  const bool mat4 = pose_kind == R2IK_POSE_MAT4;
  const unsigned g = blocks_for(n);
  R2IK_CUDA(mat4 ? launch_pdl(k_symik_solve_f32<R2IK_POSE_MAT4>, g, R2IK_BLOCK, s, h->A, h->AF, poses, theta, n, reachable, state,
                              interval, joints, elbow, escalated_idx, n_escalated)
                 : launch_pdl(k_symik_solve_f32<R2IK_POSE_EULER6>, g, R2IK_BLOCK, s, h->A, h->AF, poses, theta, n, reachable, state,
                              interval, joints, elbow, escalated_idx, n_escalated),
            "k_symik_solve_f32 launch");
  R2IK_CUDA(mat4 ? launch_pdl(k_symik_escalated_f32<R2IK_POSE_MAT4>, eb, 32, s, h->A, poses, theta, prev_joints, reachable, state,
                              interval, joints, elbow, escalated_idx, n_escalated)
                 : launch_pdl(k_symik_escalated_f32<R2IK_POSE_EULER6>, eb, 32, s, h->A, poses, theta, prev_joints, reachable, state,
                              interval, joints, elbow, escalated_idx, n_escalated),
            "k_symik_escalated_f32 launch");
  R2IK_CUDA(cudaGetLastError(), "k_symik_solve_f32 launch");
  return 0;
}

int r2ik_symik_no_limits_f64(r2ik_handle h, int pose_kind, const double *poses, const double *theta, const double *prev_joints,
                             int32_t prev_stride, int64_t n, double *joints, double *elbow, uint8_t *projected, void *stream) {
  if (n < 0 || (pose_kind != R2IK_POSE_EULER6 && pose_kind != R2IK_POSE_MAT4) || (prev_stride != 0 && prev_stride != 7))
    return fail_arg(R2IK_ERR_ARG, "r2ik_symik_no_limits_f64: bad n, pose_kind or prev_stride (0 = broadcast, 7 = per pose)");
  if (!h) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_no_limits_f64: null handle");
  if (n == 0) return 0;
  if (!poses || !theta || !joints) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_no_limits_f64: null argument");
  if (misaligned16(poses)) return fail_arg(R2IK_ERR_ARG, "r2ik_symik_no_limits_f64: poses must be 16-byte aligned");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaStream_t s = (cudaStream_t)stream;
  if (pose_kind == R2IK_POSE_MAT4)
    k_symik_no_limits<R2IK_POSE_MAT4><<<blocks_for(n), R2IK_BLOCK, 0, s>>>(h->A, poses, theta, prev_joints, prev_stride, n, joints, elbow, projected);
  else
    k_symik_no_limits<R2IK_POSE_EULER6><<<blocks_for(n), R2IK_BLOCK, 0, s>>>(h->A, poses, theta, prev_joints, prev_stride, n, joints, elbow, projected);
  R2IK_CUDA(cudaGetLastError(), "k_symik_no_limits launch");
  return 0;
}

int r2ik_elbow_positions_f64(r2ik_handle h, int pose_kind, const double *poses, const double *thetas, int32_t K, int64_t n,
                             int32_t no_limits, double *elbows, uint8_t *projected, void *stream) {
  if (n < 0 || K < 0 || (pose_kind != R2IK_POSE_EULER6 && pose_kind != R2IK_POSE_MAT4))
    return fail_arg(R2IK_ERR_ARG, "r2ik_elbow_positions_f64: bad n, K or pose_kind");
  if (!h) return fail_arg(R2IK_ERR_NULL, "r2ik_elbow_positions_f64: null handle");
  if (n == 0 || K == 0) return 0;
  if (!poses || !thetas || !elbows) return fail_arg(R2IK_ERR_NULL, "r2ik_elbow_positions_f64: null argument");
  if (misaligned16(poses)) return fail_arg(R2IK_ERR_ARG, "r2ik_elbow_positions_f64: poses must be 16-byte aligned");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned g = blocks_for(n);
  if (pose_kind == R2IK_POSE_MAT4) {
    if (no_limits) k_elbow_positions<R2IK_POSE_MAT4, true><<<g, R2IK_BLOCK, 0, s>>>(h->A, poses, thetas, K, n, elbows, projected);
    else k_elbow_positions<R2IK_POSE_MAT4, false><<<g, R2IK_BLOCK, 0, s>>>(h->A, poses, thetas, K, n, elbows, projected);
  } else {
    if (no_limits) k_elbow_positions<R2IK_POSE_EULER6, true><<<g, R2IK_BLOCK, 0, s>>>(h->A, poses, thetas, K, n, elbows, projected);
    else k_elbow_positions<R2IK_POSE_EULER6, false><<<g, R2IK_BLOCK, 0, s>>>(h->A, poses, thetas, K, n, elbows, projected);
  }
  R2IK_CUDA(cudaGetLastError(), "k_elbow_positions launch");
  return 0;
}

int r2ik_symik_sweep_f64(r2ik_handle h, int pose_kind, const double *poses, int64_t n, const double *thetas,
                         int32_t theta_stride, int32_t K, int32_t no_limits, const double *prev_joints, uint8_t *state,
                         double *interval, double *thetas_used, double *joints, double *elbow, uint8_t *projected,
                         void *stream) {
  if (n < 0 || K < 1 || (pose_kind != R2IK_POSE_EULER6 && pose_kind != R2IK_POSE_MAT4 && pose_kind != R2IK_POSE_MAT34))
    return fail_arg(R2IK_ERR_ARG, "r2ik_symik_sweep_f64: bad n, K (>= 1) or pose_kind");
  if (theta_stride != 0 && theta_stride != K)
    return fail_arg(R2IK_ERR_ARG, "r2ik_symik_sweep_f64: theta_stride must be 0 (one shared row) or K (one row per pose)");
  if (n > INT64_MAX / K / 7) return fail_arg(R2IK_ERR_ARG, "r2ik_symik_sweep_f64: n * K * 7 overflows");
  if (!h) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_sweep_f64: null handle");
  if (n == 0) return 0;
  if (!poses || !state || !joints) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_sweep_f64: null argument");
  if (misaligned16(poses)) return fail_arg(R2IK_ERR_ARG, "r2ik_symik_sweep_f64: poses must be 16-byte aligned");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaStream_t s = (cudaStream_t)stream;
  int P, Kt;
  sweep_tile(n, K, P, Kt);
  const int n_ktiles = (K + Kt - 1) / Kt;
  const int64_t n_tiles = (n + P - 1) / P * n_ktiles;
  if (n_tiles > 0x7fffffffLL) return fail_arg(R2IK_ERR_ARG, "r2ik_symik_sweep_f64: more than 2^31 - 1 tiles");
  const unsigned g = (unsigned)n_tiles;
#define R2IK_SWEEP(KIND, NL) \
  launch_pdl(k_symik_sweep<KIND, NL>, g, R2IK_BLOCK, s, h->A, poses, n, thetas, (int)theta_stride, (int)K, P, Kt, n_ktiles, \
             prev_joints, state, interval, thetas_used, joints, elbow, projected)
  cudaError_t e;
  if (pose_kind == R2IK_POSE_MAT4) e = no_limits ? R2IK_SWEEP(R2IK_POSE_MAT4, true) : R2IK_SWEEP(R2IK_POSE_MAT4, false);
  else if (pose_kind == R2IK_POSE_MAT34) e = no_limits ? R2IK_SWEEP(R2IK_POSE_MAT34, true) : R2IK_SWEEP(R2IK_POSE_MAT34, false);
  else e = no_limits ? R2IK_SWEEP(R2IK_POSE_EULER6, true) : R2IK_SWEEP(R2IK_POSE_EULER6, false);
#undef R2IK_SWEEP
  R2IK_CUDA(e, "k_symik_sweep launch");
  R2IK_CUDA(cudaGetLastError(), "k_symik_sweep launch");
  return 0;
}

int r2ik_symik_scalar_f64(r2ik_handle h, const R2ikScalarQuery *query, R2ikScalarResult *out, void *stream) {
  if (!h || !query || !out) return fail_arg(R2IK_ERR_NULL, "r2ik_symik_scalar_f64: null argument");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  k_symik_scalar<<<1, 32, 0, (cudaStream_t)stream>>>(h->A, *query, out);
  R2IK_CUDA(cudaGetLastError(), "k_symik_scalar launch");
  return 0;
}

int r2ik_ctl_ctor_theta_f64(r2ik_handle h, double preferred_theta, const double *current_joints_rows, int32_t n_rows,
                            const double *current_pose, double *out_theta, void *stream) {
  if (!h || !current_joints_rows || !current_pose || !out_theta) return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_ctor_theta_f64: null argument");
  if (n_rows < 0 || n_rows > 7) return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_ctor_theta_f64: n_rows must be 0 .. 7 (the reference indexes joints[i] by the row)");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  CtorThetaArgs a;
  memset(&a, 0, sizeof a);
  memcpy(a.rows, current_joints_rows, sizeof(double) * 7 * (size_t)n_rows);
  memcpy(a.current_pose, current_pose, sizeof(double) * 16);
  a.preferred_theta = preferred_theta;
  a.n_rows = n_rows;
  k_ctl_ctor_theta<<<1, 32, 0, (cudaStream_t)stream>>>(h->A, a, out_theta);
  R2IK_CUDA(cudaGetLastError(), "k_ctl_ctor_theta launch");
  return 0;
}

int r2ik_stream_synchronize(void *stream) {
  R2IK_CUDA(cudaStreamSynchronize((cudaStream_t)stream), "cudaStreamSynchronize");
  return 0;
}

static int ctl_discrete_launch(bool scan, r2ik_handle h, const R2ikCtlParams *par, const double *M, int64_t n,
                               const double *prev_joints, const double *current_joints, double *joints, uint8_t *reachable,
                               uint8_t *state, uint8_t *emergency, void *stream) {
  if (!h || !par) return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_discrete_f64: null handle or parameters");
  if (n < 0 || par->nb_search_points < 2) return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_discrete_f64: bad n or nb_search_points");
  if (n == 0) return 0;
  if (!M || !prev_joints || !current_joints || !joints || !reachable || !state)
    return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_discrete_f64: null argument");
  if (misaligned16(M)) return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_discrete_f64: M must be 16-byte aligned");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  if (scan)
    k_ctl_discrete_scan<<<blocks_for(n), R2IK_BLOCK, 0, (cudaStream_t)stream>>>(h->A, *par, M, n, prev_joints, current_joints,
                                                                               joints, reachable, state, emergency);
  else
    k_ctl_discrete<<<blocks_for(n), R2IK_BLOCK, 0, (cudaStream_t)stream>>>(h->A, *par, M, n, prev_joints, current_joints, joints,
                                                                          reachable, state, emergency);
  R2IK_CUDA(cudaGetLastError(), "k_ctl_discrete launch");
  return 0;
}

int r2ik_ctl_discrete_f64(r2ik_handle h, const R2ikCtlParams *par, const double *M, int64_t n, const double *prev_joints,
                          const double *current_joints, double *joints, uint8_t *reachable, uint8_t *state,
                          uint8_t *emergency, void *stream) {
  return ctl_discrete_launch(false, h, par, M, n, prev_joints, current_joints, joints, reachable, state, emergency, stream);
}

int r2ik_ctl_discrete_scan_f64(r2ik_handle h, const R2ikCtlParams *par, const double *M, int64_t n, const double *prev_joints,
                               const double *current_joints, double *joints, uint8_t *reachable, uint8_t *state,
                               uint8_t *emergency, void *stream) {
  return ctl_discrete_launch(true, h, par, M, n, prev_joints, current_joints, joints, reachable, state, emergency, stream);
}

int64_t r2ik_ctl_discrete_workspace_bytes(int64_t n) { return n < 0 ? -1 : (int64_t)disc_ws_bytes(n); }

int r2ik_ctl_discrete_compact_f64(r2ik_handle h, const R2ikCtlParams *par, const double *M, int64_t n, const double *prev_joints,
                                  const double *current_joints, double *joints, uint8_t *reachable, uint8_t *state,
                                  uint8_t *emergency, void *workspace, int64_t workspace_bytes, void *stream) {
  if (!h || !par) return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_discrete_compact_f64: null handle or parameters");
  if (n < 0 || n >= ((int64_t)1 << 31) || par->nb_search_points < 2)
    return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_discrete_compact_f64: bad n or nb_search_points");
  if (n == 0) return 0;
  if (!M || !prev_joints || !current_joints || !joints || !reachable || !state || !workspace)
    return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_discrete_compact_f64: null argument");
  if (misaligned16(M) || misaligned16(workspace))
    return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_discrete_compact_f64: M and workspace must be 16-byte aligned");
  if (workspace_bytes < (int64_t)disc_ws_bytes(n))
    return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_discrete_compact_f64: workspace smaller than r2ik_ctl_discrete_workspace_bytes(n)");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaStream_t s = (cudaStream_t)stream;
  const DiscWs w = disc_ws_carve(workspace, n);
  const unsigned lb = blocks_for(n);   // the list passes: sized for n entries, blocks past the device-side counts leave at once
  // consts is an ordinary launch (it waits for everything before it on the stream); the three passes are programmatic
  // dependents of their predecessors (r2ik_discrete_compact.cuh)
  k_disc_consts<<<1, 32, 0, s>>>(*par, prev_joints, current_joints, w.hdr);
  R2IK_CUDA(launch_pdl(k_disc_classify, lb, R2IK_BLOCK, s, h->A, *par, M, n, w.hdr, w.plan, w.finish_theta, w.search_idx,
                       w.finish_idx, joints, reachable, state, emergency), "k_disc_classify launch");
  R2IK_CUDA(launch_pdl(k_disc_search, lb, R2IK_BLOCK, s, *par, w.hdr, w.plan, w.finish_theta, w.search_idx, w.finish_idx, joints,
                       reachable, state, emergency), "k_disc_search launch");
  R2IK_CUDA(launch_pdl(k_disc_finish, lb, R2IK_BLOCK, s, h->A, *par, M, prev_joints, w.hdr, w.finish_theta, w.finish_idx, joints,
                       reachable, state, emergency), "k_disc_finish launch");
  R2IK_CUDA(cudaGetLastError(), "k_disc_* launch");
  return 0;
}

int r2ik_ctl_continuous_f64(r2ik_handle h, const R2ikCtlParams *par, const double *M, int64_t T, int32_t W,
                            const double *current_joints, const double *current_pose, R2ikTrajState *st, double *joints,
                            uint8_t *reachable, uint8_t *state, void *stream) {
  if (!h || !par) return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_continuous_f64: null handle or parameters");
  if (T < 0 || W < 0 || par->nb_search_points_continuous < 2)
    return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_continuous_f64: bad T, W or nb_search_points_continuous");
  if (T == 0 || W == 0) return 0;
  if (!M || !current_joints || !current_pose || !st || !joints || !reachable || !state)
    return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_continuous_f64: null argument");
  if (misaligned16(M) || misaligned16(current_pose))
    return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_continuous_f64: M and current_pose must be 16-byte aligned");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  k_ctl_continuous<<<(unsigned)((T + R2IK_K3_BLOCK - 1) / R2IK_K3_BLOCK), R2IK_K3_BLOCK, 0, (cudaStream_t)stream>>>(h->A, *par, M, T, W, current_joints, current_pose, st,
                                                                          joints, reachable, state);
  R2IK_CUDA(cudaGetLastError(), "k_ctl_continuous launch");
  return 0;
}

int r2ik_ctl_continuous_phased_f64(r2ik_handle h, const R2ikCtlParams *par, const double *M, int64_t T, int32_t W,
                                  const double *current_joints, const double *current_pose, R2ikTrajState *st, double *joints,
                                  uint8_t *reachable, uint8_t *state, double *workspace, int32_t test_force_serial_mod,
                                  void *stream) {
  if (!h || !par) return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_continuous_phased_f64: null handle or parameters");
  if (T < 0 || W < 0 || par->nb_search_points_continuous < 2)
    return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_continuous_phased_f64: bad T, W or nb_search_points_continuous");
  if (T == 0 || W == 0) return 0;
  if (!M || !current_joints || !current_pose || !st || !joints || !reachable || !state || !workspace)
    return fail_arg(R2IK_ERR_NULL, "r2ik_ctl_continuous_phased_f64: null argument");
  if (misaligned16(M) || misaligned16(current_pose))
    return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_continuous_phased_f64: M and current_pose must be 16-byte aligned");
  const int64_t nblk = (W + R2IK_CODE_STORED - 1) / R2IK_CODE_STORED;
  if (T * nblk > 0x7fffffffLL) return fail_arg(R2IK_ERR_ARG, "r2ik_ctl_continuous_phased_f64: T * ceil(W / 127) exceeds the grid limit");
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n_wp = T * (int64_t)W;
  uint16_t *codes16 = reinterpret_cast<uint16_t *>(workspace + n_wp);       // the codes follow the T*W thetas
  const unsigned tb = (unsigned)((T + R2IK_K3_BLOCK - 1) / R2IK_K3_BLOCK);
  k_cont_targets<<<blocks_for(n_wp), R2IK_BLOCK, 0, s>>>(h->A, *par, M, n_wp, workspace, reachable, state);
  k_cont_thetas<<<tb, R2IK_K3_BLOCK, 0, s>>>(h->A, *par, T, W, current_joints, current_pose, st, workspace, reachable);
  k_cont_raw_joints_codes<<<(unsigned)(T * nblk), R2IK_CODE_BLOCK, 0, s>>>(h->A, *par, M, W, workspace, reachable, state, joints, codes16,
                                                                          test_force_serial_mod);
  k_cont_finish_codes<<<tb, R2IK_K3_BLOCK, 0, s>>>(h->A, *par, M, T, W, current_joints, st, workspace, codes16, joints, reachable, state);
  k_cont_apply_windings<<<(unsigned)(((n_wp + 7) / 8 + 255) / 256), 256, 0, s>>>(n_wp, codes16, joints);
  R2IK_CUDA(cudaGetLastError(), "k_cont_* launch");
  return 0;
}

static int reach_map_launch(bool all_f64, r2ik_handle h, const double *origin, const double *step, const int32_t *dims,
                            const double *orientations_euler, int32_t ori_begin, int32_t ori_end, uint32_t *counts,
                            void *stream) {
  if (!h || !origin || !step || !dims || !orientations_euler || !counts)
    return fail_arg(R2IK_ERR_NULL, "r2ik_reach_map_u32: null argument");
  if (dims[0] <= 0 || dims[1] <= 0 || dims[2] <= 0 || ori_begin < 0 || ori_end < ori_begin)
    return fail_arg(R2IK_ERR_ARG, "r2ik_reach_map_u32: bad dims or orientation range");
  int64_t nv = (int64_t)dims[0] * dims[1] * dims[2];
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  if (all_f64)
    k_reach_map_f64<<<blocks_for(nv), R2IK_BLOCK, 0, (cudaStream_t)stream>>>(h->A, origin[0], origin[1], origin[2], step[0],
                                                                            step[1], step[2], dims[0], dims[1], dims[2],
                                                                            orientations_euler, ori_begin, ori_end, counts);
  else
    k_reach_map<uint32_t><<<blocks_for(nv), R2IK_BLOCK, 0, (cudaStream_t)stream>>>(h->A, h->AF, origin[0], origin[1], origin[2], step[0],
                                                                                  step[1], step[2], dims[0], dims[1], dims[2],
                                                                                  orientations_euler, ori_begin, ori_end, 0, nv, 1, 0, counts);
  R2IK_CUDA(cudaGetLastError(), "k_reach_map launch");
  return 0;
}

int r2ik_reach_map_range_u16(r2ik_handle h, const double *origin, const double *step, const int32_t *dims,
                             const double *orientations_euler, int32_t ori_begin, int32_t ori_end, int64_t voxel_begin,
                             int64_t voxel_end, int32_t row_mod, int32_t row_rem, uint16_t *counts, void *stream) {
  if (!h || !origin || !step || !dims || !orientations_euler || !counts)
    return fail_arg(R2IK_ERR_NULL, "r2ik_reach_map_range_u16: null argument");
  if (dims[0] <= 0 || dims[1] <= 0 || dims[2] <= 0 || ori_begin < 0 || ori_end < ori_begin || ori_end - ori_begin > 65535)
    return fail_arg(R2IK_ERR_ARG, "r2ik_reach_map_range_u16: bad dims or orientation range (at most 65 535 orientations per call)");
  const int64_t nv = (int64_t)dims[0] * dims[1] * dims[2];
  if (voxel_begin < 0 || voxel_end > nv || voxel_end < voxel_begin)
    return fail_arg(R2IK_ERR_ARG, "r2ik_reach_map_range_u16: bad voxel range");
  if (row_mod < 1 || row_rem < 0 || row_rem >= row_mod || (row_mod > 1 && (voxel_begin % dims[2] || voxel_end % dims[2])))
    return fail_arg(R2IK_ERR_ARG, "r2ik_reach_map_range_u16: bad row interleave (0 <= row_rem < row_mod; row-aligned range when row_mod > 1)");
  if (voxel_end == voxel_begin) return 0;
  int64_t n_launch = voxel_end - voxel_begin;
  if (row_mod > 1) {
    const int64_t row0 = voxel_begin / dims[2], row1 = voxel_end / dims[2];
    const int64_t first = row0 + ((row_rem - row0 % row_mod) + row_mod) % row_mod;
    n_launch = first < row1 ? ((row1 - first + row_mod - 1) / row_mod) * dims[2] : 0;
    if (n_launch == 0) return 0;
  }
  DeviceGuard guard_(h->device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  k_reach_map<uint16_t><<<blocks_for(n_launch), R2IK_BLOCK, 0, (cudaStream_t)stream>>>(
      h->A, h->AF, origin[0], origin[1], origin[2], step[0], step[1], step[2], dims[0], dims[1], dims[2], orientations_euler,
      ori_begin, ori_end, voxel_begin, voxel_end, row_mod, row_rem, counts);
  R2IK_CUDA(cudaGetLastError(), "k_reach_map launch");
  return 0;
}

int r2ik_reach_map_u32(r2ik_handle h, const double *origin, const double *step, const int32_t *dims,
                       const double *orientations_euler, int32_t ori_begin, int32_t ori_end, uint32_t *counts, void *stream) {
  return reach_map_launch(false, h, origin, step, dims, orientations_euler, ori_begin, ori_end, counts, stream);
}

int r2ik_reach_map_f64_u32(r2ik_handle h, const double *origin, const double *step, const int32_t *dims,
                           const double *orientations_euler, int32_t ori_begin, int32_t ori_end, uint32_t *counts,
                           void *stream) {
  return reach_map_launch(true, h, origin, step, dims, orientations_euler, ori_begin, ori_end, counts, stream);
}

int r2ik_fk_f64(const R2ikFkChain *chain, int device, const double *joints, int64_t n, double *M, void *stream) {
  if (!chain) return fail_arg(R2IK_ERR_NULL, "r2ik_fk_f64: null chain");
  if (n < 0) return fail_arg(R2IK_ERR_ARG, "r2ik_fk_f64: bad n");
  if (n == 0) return 0;
  if (!joints || !M) return fail_arg(R2IK_ERR_NULL, "r2ik_fk_f64: null argument");
  DeviceGuard guard_(device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  k_fk<<<blocks_for(n), R2IK_BLOCK, 0, (cudaStream_t)stream>>>(*chain, joints, n, M);
  R2IK_CUDA(cudaGetLastError(), "k_fk launch");
  return 0;
}

int r2ik_copy2d_async(void *dst, size_t dst_pitch, const void *src, size_t src_pitch, size_t width_bytes, size_t rows,
                      void *stream) {
  if (!dst || !src) return fail_arg(R2IK_ERR_NULL, "r2ik_copy2d_async: null argument");
  if (width_bytes > dst_pitch || width_bytes > src_pitch) return fail_arg(R2IK_ERR_ARG, "r2ik_copy2d_async: width exceeds a pitch");
  if (width_bytes == 0 || rows == 0) return 0;
  R2IK_CUDA(cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width_bytes, rows, cudaMemcpyDefault, (cudaStream_t)stream),
            "cudaMemcpy2DAsync");
  return 0;
}

int r2ik_dfma_probe(int device, int32_t iters, double *out_ms, double *out_flop, void *stream) {
  if (!out_ms || !out_flop) return fail_arg(R2IK_ERR_NULL, "r2ik_dfma_probe: null argument");
  DeviceGuard guard_(device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaDeviceProp prop;
  R2IK_CUDA(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
  cudaStream_t s = (cudaStream_t)stream;
  double *sink = nullptr;
  R2IK_CUDA(cudaMalloc(&sink, sizeof(double)), "cudaMalloc");
  const int threads = 256, blocks = prop.multiProcessorCount * 8;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  k_dfma_probe<<<blocks, threads, 0, s>>>(iters / 8 + 1, 1.0, sink);  // warm-up
  cudaEventRecord(e0, s);
  k_dfma_probe<<<blocks, threads, 0, s>>>(iters, 1.0, sink);
  cudaEventRecord(e1, s);
  cudaError_t e = cudaEventSynchronize(e1);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(sink);
  if (e != cudaSuccess) return fail_cuda(e, "k_dfma_probe");
  *out_ms = (double)ms;
  *out_flop = 2.0 * 8.0 * (double)iters * (double)threads * (double)blocks;
  return 0;
}

int r2ik_ffma_probe(int device, int32_t iters, double *out_ms, double *out_flop, void *stream) {
  if (!out_ms || !out_flop) return fail_arg(R2IK_ERR_NULL, "r2ik_ffma_probe: null argument");
  DeviceGuard guard_(device);
  R2IK_CUDA(guard_.err, "cudaSetDevice");
  cudaDeviceProp prop;
  R2IK_CUDA(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
  cudaStream_t s = (cudaStream_t)stream;
  float *sink = nullptr;
  R2IK_CUDA(cudaMalloc(&sink, sizeof(float)), "cudaMalloc");
  const int threads = 256, blocks = prop.multiProcessorCount * 8;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  k_ffma_probe<<<blocks, threads, 0, s>>>(iters / 8 + 1, 1.0f, sink);  // warm-up
  cudaEventRecord(e0, s);
  k_ffma_probe<<<blocks, threads, 0, s>>>(iters, 1.0f, sink);
  cudaEventRecord(e1, s);
  cudaError_t e = cudaEventSynchronize(e1);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(sink);
  if (e != cudaSuccess) return fail_cuda(e, "k_ffma_probe");
  *out_ms = (double)ms;
  *out_flop = 2.0 * 8.0 * (double)iters * (double)threads * (double)blocks;
  return 0;
}

}  // extern "C"
