// TEST-ONLY host harness of the batched get_best_theta_to_current_joints (tests/test_best_theta_host.py compiles it with
// the flags of tests/hostsim/Makefile): symik_best_theta, the per-pose body of k_symik_best_theta, looped over the poses
// on the CPU.  It is not part of libr2ik.so and is never imported by the package.
#include <cstdint>
#include <type_traits>

#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_control.cuh"
#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_host.h"

using namespace r2ik;

// f(std::integral_constant<int, KIND>) for the pose layout `kind` (EULER6, anything else MAT4), as in hostsim.cpp
template <typename F>
static void by_kind(int kind, F f) {
  if (kind == R2IK_POSE_EULER6) f(std::integral_constant<int, R2IK_POSE_EULER6>());
  else f(std::integral_constant<int, R2IK_POSE_MAT4>());
}

extern "C" {

// r2ik_symik_best_theta_f64 (k_symik_best_theta) with the kernel's item function.  joints may be null.
void hs_symik_best_theta(const R2ikArmConfig *cfg, int kind, const double *poses, int64_t n, const double *current_joints,
                         int cj_stride, double preferred_theta, int no_limits, uint8_t *state, double *theta,
                         double *joints) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  by_kind(kind, [&](auto KI) {
    for (int64_t i = 0; i < n; ++i) {
      const double *row = poses + pose_stride(KI()) * i, *cj = current_joints + (size_t)cj_stride * i;
      double j[7];
      state[i] = (uint8_t)(no_limits ? symik_best_theta<KI(), true>(A, row, cj, preferred_theta, joints != nullptr, theta[i], j)
                                     : symik_best_theta<KI(), false>(A, row, cj, preferred_theta, joints != nullptr, theta[i], j));
      if (joints)
        for (int k = 0; k < 7; ++k) joints[7 * i + k] = j[k];
    }
  });
}

}  // extern "C"
