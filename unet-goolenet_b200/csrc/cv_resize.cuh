// cv2.resize INTER_LINEAR on float32 maps, restated bit-exactly: shared by the wavelet step (csrc/wavelet.cu) and the
// Grad-CAM op (csrc/cam.cu).  The caller passes the coordinate scale: OpenCV 4.13 computes it as in / out, while the
// wavelet kernels pass 1 / (out / in) (the form they were pinned with; the two differ by 1 ulp for some sizes, see
// DESIGN.md §8).  The NumPy twins are oracle/wavelet_ref.cv_resize_linear_f32 (1 / (out / in)) and
// oracle/cam_ref.cv_resize_linear_f32 (in / out).
#pragma once

namespace ug {

// cv2.resize INTER_LINEAR coordinate (OpenCV 4.x): fx = (d + 0.5) * scale - 0.5 in double; s = floor(fx); the
// FRACTION fx - s is what gets cast to float (measured against cv2 4.13: casting fx itself is off by up to 3e-3)
__device__ __forceinline__ void cv_coord(int d, double scale, int n_in, int* s0, int* s1, float* w1) {
  const double fxd = __dadd_rn(__dmul_rn((double)d + 0.5, scale), -0.5);
  int s = (int)floor(fxd);
  float fx = (float)__dadd_rn(fxd, -(double)s);
  if (s < 0) {
    fx = 0.0f;
    s = 0;
  }
  if (s >= n_in - 1) {
    fx = 0.0f;
    s = n_in - 1;
  }
  *s0 = s;
  *s1 = min(s + 1, n_in - 1);
  *w1 = fx;
}

__device__ __forceinline__ float cv_bilinear(const float* __restrict__ m, int w2, int y0, int y1, float wy, int x0, int x1,
                                             float wx) {
  // OpenCV 4.x evaluates each pass as the fused lerp x0 + (x1 - x0) * f (bit-exact against cv2 4.13, see
  // oracle/wavelet_ref.py cv_resize_linear_f32)
  const float a00 = m[y0 * w2 + x0], a10 = m[y1 * w2 + x0];
  const float r0 = __fmaf_rn(__fsub_rn(m[y0 * w2 + x1], a00), wx, a00);  // horizontal pass
  const float r1 = __fmaf_rn(__fsub_rn(m[y1 * w2 + x1], a10), wx, a10);
  return __fmaf_rn(__fsub_rn(r1, r0), wy, r0);                           // vertical pass
}

}  // namespace ug
