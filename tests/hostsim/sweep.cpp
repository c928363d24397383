// TEST-ONLY host harness of the elbow-angle sweep (tests/test_sweep_host.py compiles it with the flags of
// tests/hostsim/Makefile): the device item functions of k_symik_sweep looped over poses and samples on the CPU.  It is
// not part of libr2ik.so and is never imported by the package.
#include <cstdint>
#include <type_traits>

#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_device.cuh"
#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_host.h"

using namespace r2ik;

// f(std::integral_constant<int, KIND>) for the pose layout `kind` (EULER6, anything else MAT4), as in hostsim.cpp
template <typename F>
static void by_kind(int kind, F f) {
  if (kind == R2IK_POSE_EULER6) f(std::integral_constant<int, R2IK_POSE_EULER6>());
  else f(std::integral_constant<int, R2IK_POSE_MAT4>());
}

extern "C" {

// r2ik_symik_sweep_f64 (k_symik_sweep): one solve per pose, then the K samples, with the kernel's item functions.
// Every output is required here.
void hs_symik_sweep(const R2ikArmConfig *cfg, int kind, const double *poses, int64_t n, const double *thetas,
                    int theta_stride, int K, int no_limits, const double *prev, uint8_t *state, double *interval,
                    double *thetas_used, double *joints, double *elbow, uint8_t *projected) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  const double prev0 = prev ? prev[0] : 0.0, prev2 = prev ? prev[2] : 0.0;
  by_kind(kind, [&](auto KI) {
    for (int64_t i = 0; i < n; ++i) {
      const double *row = poses + pose_stride(KI()) * i;
      Solve S;
      const Reach rc = no_limits ? symik_reach<KI(), true>(A, row, S) : symik_reach<KI(), false>(A, row, S);
      state[i] = (uint8_t)rc.state;
      interval[2 * i] = rc.i0; interval[2 * i + 1] = rc.i1;
      for (int k = 0; k < K; ++k) {
        const size_t o = (size_t)i * K + k;
        const double th = sweep_theta(rc, thetas ? thetas + (size_t)theta_stride * i : nullptr, K, k);
        thetas_used[o] = th;
        projected[o] = sweep_sample(A, S, rc, th, prev0, prev2, joints + 7 * o, elbow + 3 * o);
      }
    }
  });
}

// sweep_theta's sampled angles (thetas NULL) for n reachable intervals itv (n x 2): out n x K
void hs_sweep_theta(const double *itv, int64_t n, int K, double *out) {
  for (int64_t i = 0; i < n; ++i) {
    Reach rc;
    rc.state = R2IK_STATE_REACHABLE; rc.i0 = itv[2 * i]; rc.i1 = itv[2 * i + 1];
    for (int k = 0; k < K; ++k) out[(size_t)i * K + k] = sweep_theta(rc, nullptr, K, k);
  }
}

}  // extern "C"
