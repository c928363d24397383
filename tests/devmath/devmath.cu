// TEST-ONLY device probe library: every elementary routine of the solver's math layer (r2ik_math.cuh, the
// helpers of r2ik_device.cuh and the FP32 routines of r2ik_device_f32.cuh) as its own kernel, one thread per
// element, so tests/test_gpu_math.py can compare the *device* arithmetic -- MUFU seeds, Newton steps, .approx
// instructions, FMA contraction under the shipped nvcc flags -- with high-precision references.  The host build
// of the same headers (tests/hostsim) takes the exact library operations instead, so it cannot stand in for this.
// Never linked into libr2ik.so.
//
// Every launcher takes device pointers, the element count and a stream, and returns the cudaError_t of the launch.
#include <cuda_runtime.h>
#include <stdint.h>

#include "r2ik_device_f32.cuh"

using namespace r2ik;

#define DM_KERNEL_BEGIN(name, ...)                                         \
  __global__ void k_##name(__VA_ARGS__, int64_t n) {                        \
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;      \
    if (i >= n) return;
#define DM_KERNEL_END }

static constexpr int kBlock = 256;
static inline unsigned dm_grid(int64_t n) { return (unsigned)((n + kBlock - 1) / kBlock); }

// ------------------------------------------------------------------------------------------------- FP64
DM_KERNEL_BEGIN(div_fast, const double *a, const double *b, double *out) out[i] = div_fast(a[i], b[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(rcp_fast, const double *b, double *out) out[i] = rcp_fast(b[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(rsqrt_pos, const double *x, double *out) out[i] = rsqrt_pos(x[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(sqrt_nonneg, const double *x, double *out) out[i] = sqrt_nonneg(x[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(sqrt_rsqrt_nonneg, const double *x, double *out, double *inv)
  double v;
  out[i] = sqrt_rsqrt_nonneg(x[i], v);
  inv[i] = v;
DM_KERNEL_END
DM_KERNEL_BEGIN(atan2_core, const double *y, const double *x, double *out, uint8_t *ok)
  out[i] = atan2_core(y[i], x[i]);
  ok[i] = atan2_core_ok(y[i], x[i]);
DM_KERNEL_END
DM_KERNEL_BEGIN(angle_of_unit, const double *c, const double *s, double *out) out[i] = angle_of_unit(c[i], s[i]); DM_KERNEL_END
// the fast route of cs_and_angle: (c, s) = (x, y) / |(x, y)| under the exponent window of cs_of_atan2, then angle_of_unit
DM_KERNEL_BEGIN(cs_and_angle, const double *y, const double *x, double *c, double *s, double *ang, uint8_t *degenerate)
  double cc, ss;
  bool deg = false;
  ang[i] = cs_and_angle<false>(y[i], x[i], cc, ss, deg);
  c[i] = cc; s[i] = ss; degenerate[i] = deg;
DM_KERNEL_END
DM_KERNEL_BEGIN(sincos_small, const double *x, double *sn, double *cs, uint8_t *ok)
  double a, b;
  sincos_small(x[i], a, b);
  sn[i] = a; cs[i] = b; ok[i] = sincos_small_ok(x[i]);
DM_KERNEL_END
DM_KERNEL_BEGIN(sincos_any, const double *x, double *sn, double *cs)
  double a, b;
  sincos_any(x[i], a, b);
  sn[i] = a; cs[i] = b;
DM_KERNEL_END
DM_KERNEL_BEGIN(pymod_2pi, const double *x, double *out) out[i] = pymod_2pi(x[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(angle_diff, const double *a, const double *b, double *out) out[i] = angle_diff(a[i], b[i]); DM_KERNEL_END
// element i: sample idx[i] of np.linspace(start[i], stop[i], num[i])
DM_KERNEL_BEGIN(linspace_value, const double *start, const double *stop, const int32_t *num, const int32_t *idx, double *out)
  const Linspace L = make_linspace(start[i], stop[i], num[i]);
  out[i] = linspace_value(L, idx[i]);
DM_KERNEL_END

// ------------------------------------------------------------------------------------------------- FP32
DM_KERNEL_BEGIN(rsqrt_f, const float *x, float *out) out[i] = f32::rsqrt_f(x[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(rcp_f, const float *x, float *out) out[i] = f32::rcp_f(x[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(sqrt_f, const float *x, float *out) out[i] = f32::sqrt_f(x[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(sincos_f, const float *x, float *sn, float *cs)
  float a, b;
  f32::sincos_f(x[i], a, b);
  sn[i] = a; cs[i] = b;
DM_KERNEL_END
DM_KERNEL_BEGIN(angle_of_unit_f, const float *c, const float *s, float *out) out[i] = f32::angle_of_unit_f(c[i], s[i]); DM_KERNEL_END
DM_KERNEL_BEGIN(cs_and_angle_f, const float *y, const float *x, float *c, float *s, float *ang, uint8_t *esc)
  float cc, ss;
  bool e = false;
  ang[i] = f32::cs_and_angle_f(y[i], x[i], cc, ss, e);
  c[i] = cc; s[i] = ss; esc[i] = e;
DM_KERNEL_END

#define DM_LAUNCH(name, params, args)                                                   \
  extern "C" int dm_##name params {                                                     \
    if (n <= 0) return (int)cudaSuccess;                                                \
    k_##name<<<dm_grid(n), kBlock, 0, stream>>> args;                                   \
    return (int)cudaGetLastError();                                                     \
  }

DM_LAUNCH(div_fast, (const double *a, const double *b, double *out, int64_t n, cudaStream_t stream), (a, b, out, n))
DM_LAUNCH(rcp_fast, (const double *b, double *out, int64_t n, cudaStream_t stream), (b, out, n))
DM_LAUNCH(rsqrt_pos, (const double *x, double *out, int64_t n, cudaStream_t stream), (x, out, n))
DM_LAUNCH(sqrt_nonneg, (const double *x, double *out, int64_t n, cudaStream_t stream), (x, out, n))
DM_LAUNCH(sqrt_rsqrt_nonneg, (const double *x, double *out, double *inv, int64_t n, cudaStream_t stream), (x, out, inv, n))
DM_LAUNCH(atan2_core, (const double *y, const double *x, double *out, uint8_t *ok, int64_t n, cudaStream_t stream), (y, x, out, ok, n))
DM_LAUNCH(angle_of_unit, (const double *c, const double *s, double *out, int64_t n, cudaStream_t stream), (c, s, out, n))
DM_LAUNCH(cs_and_angle, (const double *y, const double *x, double *c, double *s, double *ang, uint8_t *degenerate, int64_t n,
                         cudaStream_t stream), (y, x, c, s, ang, degenerate, n))
DM_LAUNCH(sincos_small, (const double *x, double *sn, double *cs, uint8_t *ok, int64_t n, cudaStream_t stream), (x, sn, cs, ok, n))
DM_LAUNCH(sincos_any, (const double *x, double *sn, double *cs, int64_t n, cudaStream_t stream), (x, sn, cs, n))
DM_LAUNCH(pymod_2pi, (const double *x, double *out, int64_t n, cudaStream_t stream), (x, out, n))
DM_LAUNCH(angle_diff, (const double *a, const double *b, double *out, int64_t n, cudaStream_t stream), (a, b, out, n))
DM_LAUNCH(linspace_value, (const double *start, const double *stop, const int32_t *num, const int32_t *idx, double *out, int64_t n,
                           cudaStream_t stream), (start, stop, num, idx, out, n))
DM_LAUNCH(rsqrt_f, (const float *x, float *out, int64_t n, cudaStream_t stream), (x, out, n))
DM_LAUNCH(rcp_f, (const float *x, float *out, int64_t n, cudaStream_t stream), (x, out, n))
DM_LAUNCH(sqrt_f, (const float *x, float *out, int64_t n, cudaStream_t stream), (x, out, n))
DM_LAUNCH(sincos_f, (const float *x, float *sn, float *cs, int64_t n, cudaStream_t stream), (x, sn, cs, n))
DM_LAUNCH(angle_of_unit_f, (const float *c, const float *s, float *out, int64_t n, cudaStream_t stream), (c, s, out, n))
DM_LAUNCH(cs_and_angle_f, (const float *y, const float *x, float *c, float *s, float *ang, uint8_t *esc, int64_t n,
                           cudaStream_t stream), (y, x, c, s, ang, esc, n))
