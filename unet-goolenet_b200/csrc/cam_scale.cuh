// pytorch-grad-cam's scale_cam_image on one raw Grad-CAM map, shared by the Grad-CAM op (csrc/cam.cu) and the
// source-frame op (csrc/source_frame.cu), so that both normalise a stored cam to the same bits.
#pragma once
#include <cfloat>

namespace ug {

// One warp (lane = threadIdx.x & 31) normalises the hw values of v in place: v = cam - min(cam); v = v / (1e-7f + max(v))
// in fp32 (min / max are exact in any order).  raw, when not null, receives the values before scaling.
__device__ __forceinline__ void cam_scale_warp(float* v, int hw, int lane, float* raw) {
  float mn = FLT_MAX;
  for (int p = lane; p < hw; p += 32) mn = fminf(mn, v[p]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
  float mx = 0.0f;
  for (int p = lane; p < hw; p += 32) mx = fmaxf(mx, __fsub_rn(v[p], mn));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const float den = __fadd_rn(1e-7f, mx);
  for (int p = lane; p < hw; p += 32) {
    const float cam = v[p];
    if (raw) raw[p] = cam;
    v[p] = __fdiv_rn(__fsub_rn(cam, mn), den);
  }
}

}  // namespace ug
