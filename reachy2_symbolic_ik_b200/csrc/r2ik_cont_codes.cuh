// K3 finish pass on winding codes (k_cont_raw_joints_codes + k_cont_finish_codes).
//
// The last link of ControlIK's continuous mode (ctl:393-405, utl:493-589) takes the joints of a waypoint and returns
//     nj = previous_sol + angle_diff(j, previous_sol)                 (allow_multiturn)
// clamped to +-6 pi (joints 0, 2, 6), checked for continuity against previous_sol, and keeps it as the next previous_sol.
// As a scan over the raw joints (round 1: four lanes per trajectory) this reads and rewrites 56 bytes per waypoint -- 2.9 ms
// of the 10.2 ms of cfg 4 -- although
// nj is j itself -- to one rounding -- unless a joint has wound past +-pi.  Consecutive outputs are congruent to the raw
// joints modulo 2 pi, so everything the recursion needs from a waypoint depends on the RAW joints of that waypoint and of
// its predecessor only:
//     d_q   = angle_diff(j_q(w), j_q(w-1))                            the step of joint q
//     dk_q  = rint((j_q(w-1) + d_q - j_q(w)) / 2 pi)  in {-1, 0, +1}   the change of its winding number
//     viol  = any_q |d_q| > max_step_q                                 the continuity verdict (utl:571-589)
// The joints kernel computes them in parallel (the predecessor's joints come through shared memory) and stores them as a
// 16-bit code per waypoint; the scan then walks 2 bytes per waypoint, adds integer windings and writes the ABSOLUTE winding
// of each joint back into the code (a last, fully parallel kernel adds 2 pi k to the rows that have one: done inside the
// scan, that read-modify-write is a dependent DRAM access per waypoint of every wound trajectory, and the 31 ordinary
// lanes of its warp wait for it: 0.8 ms).  The scan touches a joints row only where the waypoint is IRREGULAR -- first of its trajectory or of its
// block (no predecessor in shared memory), invalid rotation, serial get_joints, or a predecessor that is one of those --
// or the controller is not in its ordinary state (initialising, latched, a continuity violation, |k| >= 3 where the
// +-6 pi clamp can fire).  An irregular waypoint takes the reference's statements verbatim on the stored row (the
// same code as the serial kernel), after which the windings are read back off the result.
//
// Blocks of the joints kernel are aligned to trajectories and overlap by one waypoint: a block of 128 threads stores 127
// waypoints and its first thread recomputes the last waypoint of the previous block as their predecessor (0.8 % more
// arithmetic), so that only the first waypoint of a trajectory is irregular by position.  (With disjoint blocks the scan
// took one exact step -- a dependent DRAM round trip -- per 128 waypoints: 0.40 ms instead of 0.1 ms for cfg 4.)
//
// The two device functions are __host__ __device__: tests/hostsim runs them on the host against the serial form.
#pragma once

#include <string.h>

#define R2IK_CODE_BLOCK 128
#define R2IK_CODE_IRREGULAR 0x8000u
#define R2IK_CODE_VIOL 0x4000u
#define R2IK_CODE_STILL 0x1555u       // all seven winding changes zero, continuous: the ordinary waypoint

namespace r2ik {

// Code of waypoint w from its raw joints j and its predecessor's jp (both ordinary: valid rotation, straight-line get_joints).
// With r = rint((j - jp) / 2 pi) the wrapped step is d = (j - jp) - 2 pi r and the output nj = nj_prev + d sits 2 pi (-r)
// further from the raw j than nj_prev sat from jp: dk = -r.  (d = +-pi exactly, where the reference's angle_diff picks
// -pi, is a continuity violation either way and goes to the exact statements.)
R2IK_HD unsigned cont_wind_code(const double j[7], const double jp[7]) {
  unsigned code = 0;
  bool viol = false;
#pragma unroll
  for (int q = 0; q < 7; ++q) {
    const double e = j[q] - jp[q];
    const double r = rint(e * (1.0 / kTwoPi));
    const double d = fma(-r, kTwoPi, e);
    code |= (unsigned)(1 - (int)r) << (2 * q);
    viol = viol || !(fabs(d) <= (q < 4 ? 0.5 : 1.0));       // NaN-safe: anything that is not a small step is a violation
  }
  return code | (viol ? R2IK_CODE_VIOL : 0u);
}

// An irregular waypoint's code: its kind (R2IK_WP_*) and serial flag ride in the low bits.
R2IK_HD unsigned cont_irregular_code(int c) { return R2IK_CODE_IRREGULAR | (unsigned)(c & 0x7f) | ((c & R2IK_WP_SERIAL) ? 0x80u : 0u); }

// State of the scan between segments of a trajectory (beside the controller state R2ikTrajState).
struct CodeScan {
  int kq[7];        // winding of each joint: nj = raw + 2 pi kq
  int last;         // last waypoint taken on the fast path since the last exact step (-1: none)
  bool fast;        // previous_sol is the row of waypoint `last` (not materialised in the controller state)
  bool last_final;  // ... which is stored final (an exact step wrote it) rather than raw (+ 2 pi kq still to be added)
  bool any_wound;   // some kq != 0: every waypoint gets its absolute windings written until the joints unwind
};
R2IK_HD void code_scan_init(CodeScan &sc) {
  for (int q = 0; q < 7; ++q) sc.kq[q] = 0;
  sc.last = -1; sc.fast = false; sc.any_wound = false; sc.last_final = false;
}

// The finish scan of the waypoints [w0, w1) of ONE trajectory on winding codes.  `rows` = the trajectory's W x 7 raw joints
// (in / out), `thetas` its W rate-limited thetas, `reach` / `st` its flag / state bytes (reach already holds kind == TARGET
// for every waypoint; st the reference state); `seg_codes` = the codes of [w0, w1) (any memory: the kernel passes a
// shared-memory tile), in: the winding CHANGES, out: the absolute windings still to be added to the stored rows
// (R2IK_CODE_STILL = none; cont_apply_windings does it); `chunk_ok`: seg_codes + (w - w0) is 16-byte aligned whenever w is
// a multiple of 8.
// Returns true when it changed a code of the segment.
template <typename SerialFn>
R2IK_HD bool cont_finish_codes_segment(int w0, int w1, const double *current_joints, R2ikTrajState &cs, CodeScan &sc,
                                       const double *thetas, uint16_t *seg_codes, bool chunk_ok, double *rows, uint8_t *reach,
                                       uint8_t *st, SerialFn serial_joints) {
  bool changed = false;
  for (int w = w0; w < w1; ++w) {
    // eight ordinary waypoints at a time (one 128-bit load of their codes) while nothing is wound
    if (sc.fast && !sc.any_wound && chunk_ok && (w & 7) == 0 && w + 8 <= w1) {
      uint32_t c4[4];
#if defined(__CUDA_ARCH__)
      const uint4 v = *reinterpret_cast<const uint4 *>(seg_codes + (w - w0));
      c4[0] = v.x; c4[1] = v.y; c4[2] = v.z; c4[3] = v.w;
#else
      memcpy(c4, seg_codes + (w - w0), 16);
#endif
      const uint32_t still2 = R2IK_CODE_STILL | (R2IK_CODE_STILL << 16);
      if (c4[0] == still2 && c4[1] == still2 && c4[2] == still2 && c4[3] == still2) { sc.last = w + 7; sc.last_final = false; w += 7; continue; }
    }
    const unsigned code = seg_codes[w - w0];
    if (sc.fast && !sc.any_wound && code == R2IK_CODE_STILL) { sc.last = w; sc.last_final = false; continue; }   // nothing wound, nothing winds: the row stands
    bool exact = !sc.fast || (code & (R2IK_CODE_IRREGULAR | R2IK_CODE_VIOL)) != 0;
    int nk[7];
    bool wound = false;
    if (!exact) {
#pragma unroll
      for (int q = 0; q < 7; ++q) {
        nk[q] = sc.kq[q] + (int)((code >> (2 * q)) & 3u) - 1;
        wound = wound || nk[q] != 0;
      }
      // an absolute winding has two bits in the code (-1, 0, +1); the second turn of any joint goes to the exact
      // statements (|raw| <= 3 pi / 2, so the +-6 pi clamp of joints 0 / 2 / 6, utl:535-568, is far beyond that)
      unsigned abs_code = 0;
#pragma unroll
      for (int q = 0; q < 7; ++q) {
        exact = exact || abs(nk[q]) >= 2;
        abs_code |= (unsigned)(nk[q] + 1) << (2 * q);
      }
      if (!exact) {
#pragma unroll
        for (int q = 0; q < 7; ++q) sc.kq[q] = nk[q];
        sc.any_wound = wound;
        changed = changed || abs_code != code;
        seg_codes[w - w0] = (uint16_t)abs_code;          // R2IK_CODE_STILL when nothing is wound
        sc.last = w; sc.last_final = false;
        continue;
      }
    }
    double *row = rows + 7 * (size_t)w;
    // ---- the reference's statements on this waypoint (ctl:205-210, 306-313, 393-405), from a materialised state
    if (sc.fast && sc.last >= 0) {
#pragma unroll
      for (int q = 0; q < 7; ++q)
        cs.previous_sol[q] = rows[7 * (size_t)sc.last + q] + (sc.last_final ? 0.0 : kTwoPi * (double)sc.kq[q]);
      cs.previous_theta = thetas[sc.last];
      sc.last = -1;
    }
    sc.fast = false;
    changed = changed || code != R2IK_CODE_STILL;
    seg_codes[w - w0] = (uint16_t)R2IK_CODE_STILL;       // this row is final when the scan leaves it
    if (cs.emergency_stop) {
#pragma unroll
      for (int q = 0; q < 7; ++q) row[q] = cs.previous_sol[q];
      reach[w] = 0; st[w] = R2IK_STATE_EMERGENCY;
      continue;
    }
    int kind, is_serial;
    if (code & R2IK_CODE_IRREGULAR) { kind = (int)(code & 0x7fu); is_serial = (code & 0x80u) != 0; }
    else { kind = reach[w] ? R2IK_WP_TARGET : R2IK_WP_NO_SAMPLE; is_serial = 0; }     // any valid kind: only TARGET matters below
    if (kind == R2IK_WP_INVALID) { reach[w] = 0; continue; }      // joints are NaN, state is INVALID_ROTATION already
    if (!cs.has_previous_sol) {
#pragma unroll
      for (int q = 0; q < 7; ++q) cs.previous_sol[q] = current_joints[q];
      cs.has_previous_sol = 1;
      cs.init = 1;
    }
    cs.previous_theta = thetas[w];
    double raw[7], nj[7];
    if (is_serial) serial_joints(w, kind, cs.previous_theta, cs.previous_sol[0], cs.previous_sol[2], raw);
    else {
#pragma unroll
      for (int q = 0; q < 7; ++q) raw[q] = row[q];
    }
#pragma unroll
    for (int q = 0; q < 7; ++q) nj[q] = raw[q];
    cont_finish(cs, nj);
#pragma unroll
    for (int q = 0; q < 7; ++q) row[q] = nj[q];
    if (code & R2IK_CODE_IRREGULAR) reach[w] = kind == R2IK_WP_TARGET ? 1 : 0;
    // back to the fast path when the result is the raw row plus whole turns (not clamped, not held back)
    if (!cs.emergency_stop) {
      bool ok = true;
#pragma unroll
      for (int q = 0; q < 7; ++q) {
        sc.kq[q] = (int)rint((nj[q] - raw[q]) * (1.0 / kTwoPi));
        ok = ok && fabs(nj[q] - (raw[q] + kTwoPi * (double)sc.kq[q])) < 1e-9;
      }
      if (ok) {
        sc.fast = true; sc.last = w; sc.last_final = true;
        sc.any_wound = (sc.kq[0] | sc.kq[1] | sc.kq[2] | sc.kq[3] | sc.kq[4] | sc.kq[5] | sc.kq[6]) != 0;
      }
    }
  }
  return changed;
}

// ... and its end: the controller state the trajectory leaves behind.
R2IK_HD void cont_finish_codes_end(R2ikTrajState &cs, const CodeScan &sc, const double *thetas, const double *rows) {
  if (sc.fast && sc.last >= 0) {
#pragma unroll
    for (int q = 0; q < 7; ++q)
      cs.previous_sol[q] = rows[7 * (size_t)sc.last + q] + (sc.last_final ? 0.0 : kTwoPi * (double)sc.kq[q]);
    cs.previous_theta = thetas[sc.last];
  }
}

// The last step: rows whose code carries absolute windings get them (one waypoint; fully parallel).
R2IK_HD void cont_apply_windings(unsigned code, double *row) {
  if (code == R2IK_CODE_STILL) return;
#pragma unroll
  for (int q = 0; q < 7; ++q) {
    const int k = (int)((code >> (2 * q)) & 3u) - 1;
    if (k) row[q] = row[q] + kTwoPi * (double)k;
  }
}

// Raw joints of waypoint k (kind c, not INVALID) at its rate-limited theta: get_joints by the straight-line route + the
// Orbita3D limit.  Returns true (serial) when get_joints met a degenerate input -- an exact singularity needs previous_sol,
// so the finish scan redoes the waypoint in order -- or when the test hook force_serial_mod = m > 0 picks the waypoint
// (ABI parameter test_force_serial_mod: every m-th waypoint takes the serial route although it does not need it, so that
// the route is exercised on ordinary data).
R2IK_HD bool cont_raw_joints_item(const ArmConst &A, const R2ikCtlParams &par, const double *row, int c, const double *theta,
                                  size_t k, int force_serial_mod, double j[7]) {
  Solve S;
  double pos[3];
  load_pose<R2IK_POSE_MAT4>(row, true, pos, S.R);
  if (c == R2IK_WP_UNREACHABLE) is_reachable_R<true>(A, pos, S);
  else circle_of_reachable(A, pos, S);   // reachable (phase 1 decided): the elbow circle is all get_joints needs
  double st, ct, E[3];
  sincos_any(*theta, st, ct);
  bool serial = !get_joints_impl<false>(A, S, ct, st, 0.0, 0.0, j, E);
  if (force_serial_mod > 0 && k % (size_t)force_serial_mod == 0) serial = true;
  if (!serial) limit_orbita3d_wrist(j, par.orbita3d_max_angle);
  return serial;
}

// The serial get_joints of one waypoint (ctl:369-393 with previous_sol[0], [2]): the rare route.
R2IK_HD void cont_serial_joints(const ArmConst &A, const R2ikCtlParams &par, const double *row, int kind, double theta,
                                double prev0, double prev2, double j[7]) {
  Solve S;
  double pos[3];
  load_pose<R2IK_POSE_MAT4>(row, true, pos, S.R);
  if (kind != R2IK_WP_UNREACHABLE) is_reachable_R<false>(A, pos, S);
  cont_raw_joints(A, par, kind, pos, S, theta, prev0, prev2, j);
}

// A whole trajectory in one segment (tests/hostsim).
template <typename SerialFn>
R2IK_HD void cont_finish_codes_trajectory(int W, const double *current_joints, R2ikTrajState &cs, const double *thetas,
                                          uint16_t *codes, double *rows, uint8_t *reach, uint8_t *st, SerialFn serial_joints) {
  CodeScan sc;
  code_scan_init(sc);
  cont_finish_codes_segment(0, W, current_joints, cs, sc, thetas, codes, ((uintptr_t)codes & 15) == 0, rows, reach, st, serial_joints);
  cont_finish_codes_end(cs, sc, thetas, rows);
  for (int w = 0; w < W; ++w) cont_apply_windings(codes[w], rows + 7 * (size_t)w);
}

}  // namespace r2ik

#if defined(__CUDACC__)
// cont_serial_joints, out of line on the device: the rare route
__device__ __noinline__ void tile_serial_joints(const r2ik::ArmConst &A, const R2ikCtlParams &par, const double *M, int kind, double theta,
                                                double prev0, double prev2, double *j) {
  double jj[7];
  r2ik::cont_serial_joints(A, par, M, kind, theta, prev0, prev2, jj);
  for (int q = 0; q < 7; ++q) j[q] = jj[q];
}

// Joints of a waypoint for its theta + Orbita3D limit, the winding code against the predecessor
// through shared memory, row-contiguous stores of the block's 127 x 7 raw joints.  Thread 0 of a block holds the waypoint
// before the block's first one (computed again, not stored).
#define R2IK_CODE_STORED (R2IK_CODE_BLOCK - 1)     // waypoints a block stores
#ifndef R2IK_CODE_MINBLOCKS
#define R2IK_CODE_MINBLOCKS 8   // 64 registers + 136 B of spills: 4 / 5 / 6 / 7 / 8 blocks -> 7.91 / 7.91 / 7.70 / 7.74 / 7.66 ms for cfg 4 (s46)
#endif
__global__ void __launch_bounds__(R2IK_CODE_BLOCK, R2IK_CODE_MINBLOCKS)
k_cont_raw_joints_codes(const __grid_constant__ r2ik::ArmConst A, const __grid_constant__ R2ikCtlParams par, const double *__restrict__ M,
                        int W, const double *__restrict__ ws, uint8_t *__restrict__ code, const uint8_t *__restrict__ state,
                        double *__restrict__ joints, uint16_t *__restrict__ codes16, int force_serial_mod) {
  using namespace r2ik;
  __shared__ double sj[R2IK_CODE_BLOCK][7];
  __shared__ uint8_t sc[R2IK_CODE_BLOCK];
  const int tid = threadIdx.x;
  const int nblk = (W + R2IK_CODE_STORED - 1) / R2IK_CODE_STORED;    // blocks per trajectory
  const int64_t t = blockIdx.x / nblk;
  const int wb = (int)(blockIdx.x - t * nblk) * R2IK_CODE_STORED;    // first stored waypoint of this block
  const int w = wb + tid - 1;                                        // thread 0: the predecessor of the block
  const bool active = w >= 0 && w < W;
  const size_t k = (size_t)t * W + (active ? w : 0);
  int c = R2IK_WP_INVALID;
  double j[7];
#pragma unroll
  for (int q = 0; q < 7; ++q) j[q] = NAN;
  bool serial = false;
  if (active) {
    if (tid > 0) {
      c = code[k];
    } else {
      // the previous block owns this waypoint and may already have replaced its code by the reach flag: thread 0 takes the
      // kind from the state byte instead, which nobody writes here (INVALID_ROTATION; EMPTY / LIMITED_BY_SHOULDER = the
      // reachable kinds, which this kernel treats alike; anything else = unreachable)
      const int sb = state[k];
      c = sb == R2IK_STATE_INVALID_ROTATION ? R2IK_WP_INVALID
          : (sb == R2IK_STATE_EMPTY || sb == R2IK_STATE_LIMITED_BY_SHOULDER) ? R2IK_WP_TARGET : R2IK_WP_UNREACHABLE;
    }
    if (c != R2IK_WP_INVALID) serial = cont_raw_joints_item(A, par, M + 16 * k, c, ws + k, k, force_serial_mod, j);
  }
  const bool ordinary = active && c != R2IK_WP_INVALID && !serial;
#pragma unroll
  for (int q = 0; q < 7; ++q) sj[tid][q] = j[q];
  sc[tid] = ordinary ? 1 : 0;
  __syncthreads();
  if (active && tid > 0) {
    unsigned cd;
    if (ordinary && sc[tid - 1]) {
      double jp[7];
#pragma unroll
      for (int q = 0; q < 7; ++q) jp[q] = sj[tid - 1][q];
      cd = cont_wind_code(j, jp);
    } else {
      cd = cont_irregular_code(serial ? (c | R2IK_WP_SERIAL) : c);
    }
    codes16[k] = (uint16_t)cd;
    code[k] = (c == R2IK_WP_TARGET) ? 1 : 0;          // from here on this array is `reachable`
  }
  // the 127 x 7 doubles the block stores are contiguous in global memory: one row-contiguous request per instruction
  const int n_here = min(R2IK_CODE_STORED, W - wb);
  double *dst = joints + ((size_t)t * W + (size_t)wb) * 7;
  const double *src = &sj[1][0];
#pragma unroll
  for (int i = 0; i < 7; ++i) {
    const int o = tid + R2IK_CODE_BLOCK * i;
    if (o < 7 * n_here) dst[o] = src[o];
  }
}

// One thread per trajectory.  The codes move through shared memory in tiles of 64 trajectories x 128 waypoints (256 B per
// trajectory, loaded with row-contiguous 128-bit requests): read directly, every thread would wait a DRAM latency per 16
// bytes of its own row -- 125 dependent misses per trajectory, 0.8 ms for cfg 4.  Row stride 272 bytes (17 x 16): rows stay
// 16-byte aligned and the 128-bit reads of a quarter warp fall on 8 x 4 distinct banks.
#define R2IK_CODE_TILE 128
__global__ void __launch_bounds__(R2IK_K3_BLOCK, 8)
k_cont_finish_codes(const __grid_constant__ r2ik::ArmConst A, const __grid_constant__ R2ikCtlParams par, const double *__restrict__ M,
                    int64_t T, int W, const double *__restrict__ current_joints, R2ikTrajState *__restrict__ states,
                    const double *__restrict__ ws, uint16_t *__restrict__ codes16, double *__restrict__ joints,
                    uint8_t *__restrict__ reachable, uint8_t *__restrict__ state) {
  using namespace r2ik;
  __shared__ __align__(16) uint16_t s_codes[R2IK_K3_BLOCK][R2IK_CODE_TILE + 8];
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x;
  const int64_t t = t0 + threadIdx.x;
  const bool live = t < T;
  const size_t base = (size_t)(live ? t : T - 1) * W;
  R2ikTrajState cs = states[live ? t : T - 1];
  CodeScan sc;
  code_scan_init(sc);
  const double *Mt = M + 16 * base;
  auto serial = [&](int w, int kind, double theta, double p0, double p2, double *out) {
    tile_serial_joints(A, par, Mt + 16 * (size_t)w, kind, theta, p0, p2, out);
  };
  const bool vec = ((uintptr_t)codes16 & 15) == 0 && (W & 7) == 0;      // every trajectory's codes start 16-byte aligned
  for (int w0 = 0; w0 < W; w0 += R2IK_CODE_TILE) {
    const int nw = min(R2IK_CODE_TILE, W - w0);
    if (vec) {
      const int chunks = (nw + 7) >> 3;                                 // 16-byte chunks per trajectory row of this tile
      for (int f = threadIdx.x; f < R2IK_K3_BLOCK * chunks; f += R2IK_K3_BLOCK) {
        const int r = f / chunks, c = f - r * chunks;
        if (t0 + r < T)
          *reinterpret_cast<uint4 *>(&s_codes[r][8 * c]) = *reinterpret_cast<const uint4 *>(codes16 + (size_t)(t0 + r) * W + w0 + 8 * c);
      }
    } else {
      for (int f = threadIdx.x; f < R2IK_K3_BLOCK * nw; f += R2IK_K3_BLOCK) {
        const int r = f / nw, c = f - r * nw;
        if (t0 + r < T) s_codes[r][c] = codes16[(size_t)(t0 + r) * W + w0 + c];
      }
    }
    __syncthreads();
    bool changed = false;
    if (live)
      changed = cont_finish_codes_segment(w0, w0 + nw, current_joints + 7 * t, cs, sc, ws + base, &s_codes[threadIdx.x][0], true,
                                          joints + 7 * base, reachable + base, state + base, serial);
    // a tile that changed goes back with the absolute windings in it (k_cont_apply_windings reads them)
    if (!__syncthreads_or(changed ? 1 : 0)) continue;
    if (vec) {
      const int chunks = (nw + 7) >> 3;
      for (int f = threadIdx.x; f < R2IK_K3_BLOCK * chunks; f += R2IK_K3_BLOCK) {
        const int r = f / chunks, c = f - r * chunks;
        if (t0 + r < T)
          *reinterpret_cast<uint4 *>(codes16 + (size_t)(t0 + r) * W + w0 + 8 * c) = *reinterpret_cast<const uint4 *>(&s_codes[r][8 * c]);
      }
    } else {
      for (int f = threadIdx.x; f < R2IK_K3_BLOCK * nw; f += R2IK_K3_BLOCK) {
        const int r = f / nw, c = f - r * nw;
        if (t0 + r < T) codes16[(size_t)(t0 + r) * W + w0 + c] = s_codes[r][c];
      }
    }
    __syncthreads();
  }
  if (live) {
    cont_finish_codes_end(cs, sc, ws + base, joints + 7 * base);
    states[t] = cs;
  }
}

// nj = j + 2 pi k for the waypoints the scan found wound (a few per thousand): eight waypoints per thread, one 128-bit
// load of their codes (the trailing n_wp % 8 and unaligned buffers one by one).
__global__ void __launch_bounds__(256)
k_cont_apply_windings(int64_t n_wp, const uint16_t *__restrict__ codes16, double *__restrict__ joints) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t k0 = 8 * g;
  if (k0 >= n_wp) return;
  if (((uintptr_t)codes16 & 15) == 0 && k0 + 8 <= n_wp) {
    const uint4 v = *reinterpret_cast<const uint4 *>(codes16 + k0);
    const uint32_t still2 = R2IK_CODE_STILL | (R2IK_CODE_STILL << 16);
    if (v.x == still2 && v.y == still2 && v.z == still2 && v.w == still2) return;
    const uint32_t c4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) r2ik::cont_apply_windings((c4[i >> 1] >> (16 * (i & 1))) & 0xffffu, joints + 7 * (k0 + i));
    return;
  }
  for (int64_t k = k0; k < n_wp && k < k0 + 8; ++k) r2ik::cont_apply_windings(codes16[k], joints + 7 * k);
}
#endif
