// r2ik_discrete_compact.cuh -- K2 (ControlIK discrete mode) for large batches as three dense passes.
//
// In the one-kernel form (k_ctl_discrete, r2ik_kernels.cu) a warp walks through three sections of very different
// population: every lane solves is_reachable, about half of the lanes search the K samples, two thirds of the lanes run
// get_joints + the safety chain -- 17 - 18 of 32 lanes active per executed instruction on the FK-sampled workload
// (profiles/r1_s43_discrete_ncu_full.txt).  Here the sections are separate kernels and the poses that need the next
// section are handed over through index lists in a caller-provided workspace, so every warp of every pass is full:
//
//   k_disc_consts    1 thread: resets the two list counters and evaluates once the result every pose without a valid
//                    theta shares (current_joints through safety_checks: ctl:454-462 with found = false)
//   k_disc_classify  all poses: rotation check, is_reachable, preferred-theta shortcut (utl:357-364).
//                    unreachable / invalid -> final result;  shortcut works -> finish list (theta = preferred);
//                    otherwise -> search list with the search plan (interval + the six elbow half-plane coefficients)
//   k_disc_search    search list: search_analytic (r2ik_control.cuh) from the stored plan.
//                    a sample found -> finish list (theta of the sample);  none -> final result (limited by shoulder)
//   k_disc_finish    finish list: the elbow circle again from the pose (carrying the 200-byte solve through memory instead
//                    would add 330 MB of traffic per 1M poses to save 15 M of 95 M warp instructions), get_joints, safety chain
//
// The per-pose device functions are the ones k_ctl_discrete calls, on the same inputs: results are identical.
// Lists are appended by block-aggregated atomics (one atomicAdd per block and list); their order is the arrival order of
// the blocks, so the scattered result rows stay roughly ascending.
#pragma once

#include "r2ik_control.cuh"

namespace r2ik {

struct DiscHeader {
  unsigned n_search, n_finish;     // list lengths: a line of their own (every block adds to them)
  unsigned pad_[30];
  double nf_joints[7];             // the result shared by every pose without a valid theta (read-only after k_disc_consts)
  int nf_bits, pad2_;
  double pad3_[8];
};
static_assert(sizeof(DiscHeader) == 256, "DiscHeader is two 128-byte lines");

constexpr uint32_t kDiscLiteral = 0x80000000u;   // flag bit of a list entry (n < 2^31)

R2IK_HD size_t disc_ws_bytes(int64_t n) { return sizeof(DiscHeader) + (size_t)n * (64 + 8 + 4 + 4); }

// The search plan of a listed pose, 8 doubles (64 bytes, 16-byte aligned): i0, i1, A1, B1, C1, A2, B2, C2
R2IK_HD void disc_plan_pack(double *p, const ArmConst &A, const Solve &S, double i0, double i1) {
  const ElbowTest T = make_elbow_test(A, S);
#if defined(__CUDA_ARCH__)
  double2 *q = reinterpret_cast<double2 *>(p);
  q[0] = make_double2(i0, i1);
  q[1] = make_double2(T.A1, T.B1);
  q[2] = make_double2(T.C1, T.A2);
  q[3] = make_double2(T.B2, T.C2);
#else
  p[0] = i0; p[1] = i1; p[2] = T.A1; p[3] = T.B1; p[4] = T.C1; p[5] = T.A2; p[6] = T.B2; p[7] = T.C2;
#endif
}

R2IK_HD SearchPlan disc_plan_unpack(const R2ikCtlParams &par, const double *p) {
  double q[8];
#if defined(__CUDA_ARCH__)
  const double2 *p2 = reinterpret_cast<const double2 *>(p);
  const double2 q0 = p2[0], q1 = p2[1], q2 = p2[2], q3 = p2[3];
  q[0] = q0.x; q[1] = q0.y; q[2] = q1.x; q[3] = q1.y; q[4] = q2.x; q[5] = q2.y; q[6] = q3.x; q[7] = q3.y;
#else
  for (int k = 0; k < 8; ++k) q[k] = p[k];
#endif
  SearchPlan P = disc_search_plan(par, q[0], q[1]);
  P.T.A1 = q[2]; P.T.B1 = q[3]; P.T.C1 = q[4]; P.T.A2 = q[5]; P.T.B2 = q[6]; P.T.C2 = q[7];
  return P;
}

// Finish a listed pose at its theta.  The elbow circle is all get_joints needs of the solve: the circle linking (a
// quarter of is_reachable) is not redone, except for the rare pose whose solve took the literal instantiation (its S is
// that instantiation's).  Returns the emergency bits.
R2IK_HD int disc_finish_listed(const ArmConst &A, const R2ikCtlParams &par, const double *row, bool literal, double theta,
                               const double prev[7], double j[7]) {
  Solve S;
  double pos[3];
  load_pose<R2IK_POSE_MAT4>(row, true, pos, S.R);       // valid and reachable: k_disc_classify listed it
  if (literal) is_reachable_R<false>(A, pos, S);
  else circle_of_reachable(A, pos, S);
  return discrete_finish(A, par, S, true, theta, prev, prev, j);
}

// Empty lists, and the result every pose without a valid theta shares (current_joints through safety_checks: ctl:454-462
// with found = false)
R2IK_HD void disc_header_init(DiscHeader *hdr, const R2ikCtlParams &par, const double *prev_joints, const double *current_joints) {
  double prev[7], j[7];
  for (int k = 0; k < 7; ++k) { prev[k] = prev_joints[k]; j[k] = current_joints[k]; }
  const int bits = safety_checks(j, prev, par.orbita3d_max_angle);
  for (int k = 0; k < 7; ++k) hdr->nf_joints[k] = j[k];
  hdr->nf_bits = bits;
  hdr->n_search = 0;
  hdr->n_finish = 0;
}

// the result of a pose without a valid theta (or NaN joints for an invalid rotation)
R2IK_HD void disc_store_final(const DiscHeader *hdr, int64_t i, int st, double *__restrict__ joints,
                              uint8_t *__restrict__ reachable, uint8_t *__restrict__ state, uint8_t *__restrict__ emergency) {
  const bool invalid = st == R2IK_STATE_INVALID_ROTATION;
#pragma unroll
  for (int k = 0; k < 7; ++k) joints[7 * i + k] = invalid ? NAN : hdr->nf_joints[k];
  reachable[i] = 0;
  state[i] = (uint8_t)st;
  if (emergency) emergency[i] = invalid ? 0 : (uint8_t)hdr->nf_bits;
}

#if defined(__CUDACC__)

struct DiscWs {
  DiscHeader *hdr;
  double *plan;           // 8 doubles per search-list entry (disc_plan_pack)
  double *finish_theta;
  uint32_t *search_idx, *finish_idx;
};
inline __host__ DiscWs disc_ws_carve(void *ws, int64_t n) {
  DiscWs w;
  char *p = static_cast<char *>(ws);
  w.hdr = reinterpret_cast<DiscHeader *>(p); p += sizeof(DiscHeader);
  w.plan = reinterpret_cast<double *>(p); p += (size_t)n * 64;
  w.finish_theta = reinterpret_cast<double *>(p); p += (size_t)n * 8;
  w.search_idx = reinterpret_cast<uint32_t *>(p); p += (size_t)n * 4;
  w.finish_idx = reinterpret_cast<uint32_t *>(p);
  return w;
}

// Programmatic dependent launch: the four kernels of a call are chained on one stream, each launched with
// cudaLaunchAttributeProgrammaticStreamSerialization.  A kernel lets its successor's blocks be scheduled early
// (disc_launch_dependents, at block start: the successor's launch latency and ramp-up overlap this kernel's tail) and
// waits for its predecessor's memory before the first access that depends on it (disc_wait_predecessor).
__device__ __forceinline__ void disc_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void disc_wait_predecessor() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Slots of this thread in the lists shared by the grid, one atomicAdd per BLOCK and list: same-address atomics are
// served one at a time by the L2 slice that owns the line (~1 / cycle), and with one per warp the 62 500 of a 1M-pose
// batch arrive in bursts -- all resident warps reach the append together.  Every thread of the block calls it.
// p0 / p1: this thread appends to list 0 / 1 (never both).  Returns the slot in the list the thread appends to.
__device__ __forceinline__ unsigned disc_append2(bool p0, bool p1, unsigned *counter0, unsigned *counter1) {
  __shared__ unsigned s_warp[2][R2IK_BLOCK / 32], s_base[2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned m0 = __ballot_sync(0xffffffffu, p0), m1 = __ballot_sync(0xffffffffu, p1);
  if (lane == 0) { s_warp[0][warp] = __popc(m0); s_warp[1][warp] = __popc(m1); }
  __syncthreads();
  if (threadIdx.x < 2) {
    unsigned tot = 0;
#pragma unroll
    for (int w = 0; w < R2IK_BLOCK / 32; ++w) tot += s_warp[threadIdx.x][w];
    s_base[threadIdx.x] = tot ? atomicAdd(threadIdx.x ? counter1 : counter0, tot) : 0u;
  }
  __syncthreads();
  const int l = p1 ? 1 : 0;
  unsigned slot = s_base[l] + __popc((l ? m1 : m0) & ((1u << lane) - 1));
  for (int w = 0; w < warp; ++w) slot += s_warp[l][w];
  return slot;          // one call per block (the shared counters are not reused)
}

__global__ void k_disc_consts(const __grid_constant__ R2ikCtlParams par, const double *__restrict__ prev_joints,
                              const double *__restrict__ current_joints, DiscHeader *hdr) {
  disc_launch_dependents();
  if (threadIdx.x || blockIdx.x) return;
  disc_header_init(hdr, par, prev_joints, current_joints);
}

#ifndef R2IK_K2C_CLASSIFY_MINBLOCKS
#define R2IK_K2C_CLASSIFY_MINBLOCKS 6
#endif
#ifndef R2IK_K2C_SEARCH_MINBLOCKS
#define R2IK_K2C_SEARCH_MINBLOCKS 8
#endif
#ifndef R2IK_K2C_FINISH_MINBLOCKS
#define R2IK_K2C_FINISH_MINBLOCKS 4
#endif

__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K2C_CLASSIFY_MINBLOCKS)
k_disc_classify(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikCtlParams par, const double *__restrict__ M,
                int64_t n, DiscHeader *hdr, double *__restrict__ plan, double *__restrict__ finish_theta,
                uint32_t *__restrict__ search_idx, uint32_t *__restrict__ finish_idx, double *__restrict__ joints,
                uint8_t *__restrict__ reachable, uint8_t *__restrict__ state, uint8_t *__restrict__ emergency) {
  disc_launch_dependents();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < n;
  Solve S;
  Reach rc;
  rc.state = R2IK_STATE_INVALID_ROTATION;
  bool shortcut = false, need_search = false;
  uint32_t tag = (uint32_t)i;      // list entry: pose index, bit 31 = the solve took the literal instantiation
  if (active) {
    disc_classify(A, par, M + 16 * i, S, rc, shortcut, need_search);
    if (rc.literal) tag |= kDiscLiteral;
  }
  disc_wait_predecessor();      // k_disc_consts: the counters are reset, the shared result is there (the poses are the caller's)
  const unsigned slot = disc_append2(need_search, shortcut, &hdr->n_search, &hdr->n_finish);
  if (need_search) {
    search_idx[slot] = tag;
    disc_plan_pack(plan + 8 * (size_t)slot, A, S, rc.i0, rc.i1);
  }
  if (shortcut) {
    finish_idx[slot] = tag;
    finish_theta[slot] = par.preferred_theta;
  }
  if (active && !need_search && !shortcut) disc_store_final(hdr, i, rc.state, joints, reachable, state, emergency);
}

__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K2C_SEARCH_MINBLOCKS)
k_disc_search(const __grid_constant__ R2ikCtlParams par, DiscHeader *hdr, const double *__restrict__ plan,
              double *__restrict__ finish_theta, const uint32_t *__restrict__ search_idx, uint32_t *__restrict__ finish_idx,
              double *__restrict__ joints, uint8_t *__restrict__ reachable, uint8_t *__restrict__ state,
              uint8_t *__restrict__ emergency) {
  // one thread per list entry; the grid is sized for n entries and the blocks past the (device-side) count leave at once
  disc_launch_dependents();
  disc_wait_predecessor();
  const unsigned count = hdr->n_search;
  if (blockIdx.x * blockDim.x >= count) return;
  const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = k < count;
  bool found = false;
  double theta = 0.0;
  uint32_t i = 0;
  if (active) {
    i = search_idx[k];
    found = disc_search(disc_plan_unpack(par, plan + 8 * (size_t)k), par.nb_search_points, theta);
  }
  const unsigned kf = disc_append2(false, found, &hdr->n_finish, &hdr->n_finish);
  if (found) {
    finish_idx[kf] = i;
    finish_theta[kf] = theta;
  } else if (active) {
    disc_store_final(hdr, (int64_t)(i & ~kDiscLiteral), R2IK_STATE_LIMITED_BY_SHOULDER, joints, reachable, state, emergency);
  }
}

__global__ void __launch_bounds__(R2IK_BLOCK, R2IK_K2C_FINISH_MINBLOCKS)
k_disc_finish(const __grid_constant__ ArmConst A, const __grid_constant__ R2ikCtlParams par, const double *__restrict__ M,
              const double *__restrict__ prev_joints, const DiscHeader *hdr, const double *__restrict__ finish_theta,
              const uint32_t *__restrict__ finish_idx, double *__restrict__ joints, uint8_t *__restrict__ reachable,
              uint8_t *__restrict__ state, uint8_t *__restrict__ emergency) {
  // one thread per list entry; the blocks past the (device-side) count leave at once.  (A persistent grid with the next
  // entry's pose row prefetched into L1 -- a third of the warp samples sit on the index -> pose row load chain -- measured
  // the same 0.22 ms: profiles/r2_experiments.md.)
  disc_wait_predecessor();
  const unsigned count = hdr->n_finish;
  const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  double prev[7];
#pragma unroll
  for (int q = 0; q < 7; ++q) prev[q] = prev_joints[q];
  const uint32_t tag = finish_idx[k];
  const int64_t i = tag & ~kDiscLiteral;
  double j[7];
  const int bits = disc_finish_listed(A, par, M + 16 * i, (tag & kDiscLiteral) != 0, finish_theta[k], prev, j);
#pragma unroll
  for (int q = 0; q < 7; ++q) joints[7 * i + q] = j[q];
  reachable[i] = 1;
  state[i] = R2IK_STATE_REACHABLE;
  if (emergency) emergency[i] = (uint8_t)bits;
}

#endif  // __CUDACC__

}  // namespace r2ik
