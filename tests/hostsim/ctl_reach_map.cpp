// TEST-ONLY host harness of the controller's workspace map (tests/test_ctl_reach_map_host.py compiles it with the flags
// of tests/hostsim/Makefile): the device item functions of k_ctl_reach_map looped over voxels and orientations on the
// CPU.  It is not part of libr2ik.so and is never imported by the package.
#include <cstdint>

#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_control.cuh"
#include "../../reachy2_symbolic_ik_b200/csrc/r2ik_host.h"

using namespace r2ik;

extern "C" {

// The public constants of an arm (max_arm_length: the reach cube of the map's default grid)
void hs_arm_constants(const R2ikArmConfig *cfg, R2ikArmConstants *pub) {
  ArmConst A;
  derive_constants(*cfg, A, *pub);
}

// r2ik_ctl_reach_map_u32 (k_ctl_reach_map) for the orientations ori (n_ori x 9, row-major 3x3): per-voxel counts, and
// with `pairs` non-null the verdict of every (voxel, orientation) pair, pairs[v * n_ori + o] = reachable | accepted << 1.
// Every voxel runs every pair (the kernel's block early-out skips only pairs whose pre-checks fail, which ctl_reach_pair
// rejects as its first step).
void hs_ctl_reach_map(const R2ikArmConfig *cfg, const R2ikCtlParams *par, const double *origin, const double *step,
                      const int32_t *dims, const double *ori, int32_t n_ori, uint32_t *accepted, uint32_t *reachable,
                      uint8_t *pairs) {
  ArmConst A; R2ikArmConstants pub;
  derive_constants(*cfg, A, pub);
  double R[512 * 9];
  bool ok[512];
  for (int32_t base = 0; base < n_ori; base += 512) {
    const int m = n_ori - base < 512 ? n_ori - base : 512;
    for (int o = 0; o < m; ++o) ok[o] = ctl_map_rotation(ori + 9 * (size_t)(base + o), R + 9 * o);
    int64_t v = 0;
    for (int ix = 0; ix < dims[0]; ++ix)
      for (int iy = 0; iy < dims[1]; ++iy)
        for (int iz = 0; iz < dims[2]; ++iz, ++v) {
          const double pos[3] = {grid_coord(origin[0], ix, step[0]), grid_coord(origin[1], iy, step[1]),
                                 grid_coord(origin[2], iz, step[2])};
          if (base == 0) { accepted[v] = 0; reachable[v] = 0; }
          for (int o = 0; o < m; ++o) {
            CtlPair c = {false, false};
            if (ok[o]) c = ctl_reach_pair(A, *par, pos, R + 9 * o);
            accepted[v] += c.accepted ? 1u : 0u;
            reachable[v] += c.reachable ? 1u : 0u;
            if (pairs) pairs[(size_t)v * n_ori + base + o] = (uint8_t)((c.reachable ? 1 : 0) | (c.accepted ? 2 : 0));
          }
        }
  }
}

}  // extern "C"
