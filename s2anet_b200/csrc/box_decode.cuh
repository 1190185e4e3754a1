// box_decode.cuh -- the rotated-box decode arithmetic shared by the decode kernels (decode.cu) and the FAM-decode
// epilogue of the plain tensor-core conv (conv_tc.cu), so that both round exactly the same way.
//
// Arithmetic: models/boxes.py:82-162 (delta2bbox_rotated) and utils/general.py:925-930 (norm_angle),
// operation by operation with individually rounded fp32 operations and the same dtype promotion as
// PyTorch applies in the reference's half-precision validation (SURVEY Appendix A.7): anchors are
// fp32, deltas are T; clamp / exp / pi*dangle are evaluated in T (rounded to T), everything that
// touches an anchor value is fp32.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math.h>

#include "common.cuh"

namespace s2a {

// round a float through T (what storing a T tensor element does)
template <typename T> __device__ __forceinline__ float round_through(float v);
template <> __device__ __forceinline__ float round_through<float>(float v) { return v; }
template <> __device__ __forceinline__ float round_through<__nv_bfloat16>(float v) {
  return __bfloat162float(__float2bfloat16_rn(v));
}
template <> __device__ __forceinline__ float round_through<__half>(float v) { return __half2float(__float2half_rn(v)); }

// models/anchors.py:94-95 for one square anchor per location: centre = index * stride + 0.5 * (stride - 1),
// w = h = scale * stride, theta = angle
__device__ __forceinline__ void fam_grid_anchor(int x, int y, float stride, float scale, float angle, float a[5]) {
  const float half = __fmul_rn(0.5f, __fsub_rn(stride, 1.0f));
  a[0] = __fadd_rn(__fmul_rn((float)x, stride), half);
  a[1] = __fadd_rn(__fmul_rn((float)y, stride), half);
  a[2] = __fmul_rn(stride, scale);
  a[3] = __fmul_rn(stride, scale);
  a[4] = angle;
}

// models/boxes.py:82-162 with is_encode_relative=True; a = (x, y, w, h, theta) fp32, d = deltas already
// widened from T.  lim = max_ratio rounded to T (torch.clamp converts its bounds to the tensor dtype).
template <typename T>
__device__ __forceinline__ void delta2bbox_rotated(const float a[5], float dx, float dy, float dw, float dh, float da,
                                                   float lim, float out[5]) {
  dw = dw < -lim ? -lim : (dw > lim ? lim : dw);          // NaN stays NaN, like torch.clamp
  dh = dh < -lim ? -lim : (dh > lim ? lim : dh);
  const float cosa = cosf(a[4]), sina = sinf(a[4]);
  const float dxw = __fmul_rn(dx, a[2]), dyh = __fmul_rn(dy, a[3]);
  out[0] = __fadd_rn(__fsub_rn(__fmul_rn(dxw, cosa), __fmul_rn(dyh, sina)), a[0]);      // boxes.py:148
  out[1] = __fadd_rn(__fadd_rn(__fmul_rn(dxw, sina), __fmul_rn(dyh, cosa)), a[1]);      // boxes.py:149
  out[2] = __fmul_rn(a[2], round_through<T>(expf(dw)));                                 // boxes.py:155
  out[3] = __fmul_rn(a[3], round_through<T>(expf(dh)));
  const float kPi = 3.14159274101257324f, kQuarterPi = 0.785398185253143311f;           // float(np.pi), float(np.pi / 4)
  const float ga = __fadd_rn(round_through<T>(__fmul_rn(da, kPi)), a[4]);               // boxes.py:159
  // norm_angle (utils/general.py:925-930): (ga + pi/4) % pi - pi/4 with Python's sign convention
  float m = fmodf(__fadd_rn(ga, kQuarterPi), kPi);
  if (m != 0.0f && m < 0.0f) m = __fadd_rn(m, kPi);
  out[4] = __fsub_rn(m, kQuarterPi);
}

// The clamp bound of dw / dh: boxes.py:115 np.abs(np.log(wh_ratio_clip)), rounded to the deltas' dtype.
inline float clamp_limit(double wh_ratio_clip, int dtype) {
  const float m = (float)fabs(log(wh_ratio_clip));
  if (dtype == S2A_BF16) return __bfloat162float(__float2bfloat16_rn(m));
  if (dtype == S2A_F16) return __half2float(__float2half_rn(m));
  return m;
}

}  // namespace s2a
