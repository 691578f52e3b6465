// Grad-CAM at GoogLeNet's inception5b (ug_cam_desc): the class activation map of each image's target class and the map
// normalised and resized into the image's ROI box, as pytorch-grad-cam's GradCAM + scale_cam_image compute it.
//
// One launch over a grid of (image, band of kCamRows output rows).  Every CTA of an image recomputes the h*w dots of
// length C (49 x 1024 for the network: 100 KB of bf16 features, read from L2 after the first CTA) into shared memory,
// normalises them and writes its band of cam_map; band 0 also writes cam and status.  The work is bounded by the
// cam_map write (S*S*4 bytes per image), so the recomputation costs L2 reads only.
#include <cfloat>
#include <cstdint>
#include "cam_scale.cuh"
#include "common.cuh"
#include "cv_resize.cuh"
#include "engine.h"

namespace ug {

static constexpr int kCamThreads = 256;
static constexpr int kCamRows = 56;       // output rows per CTA: 4 bands of a 224-row map, 1024 CTAs for 256 images
static constexpr int kCamMaxSide = 32;    // h, w
static constexpr int kCamMaxC = 2048;
static constexpr int kCamMaxS = 1024;

__global__ void __launch_bounds__(kCamThreads) cam_kernel(ug_cam_desc d) {
  __shared__ __align__(16) float wc[kCamMaxC];          // fc row of the target class
  __shared__ float v[kCamMaxSide * kCamMaxSide];        // cam, then the normalised map
  __shared__ int xs0[kCamMaxS], xs1[kCamMaxS];          // cv2 x coordinates of the box columns
  __shared__ float xw[kCamMaxS];
  __shared__ int ys0[kCamRows], ys1[kCamRows];          // ... and of this band's rows
  __shared__ float yw[kCamRows];
  __shared__ int s_cls, s_box[4];
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int i = blockIdx.x, tid = threadIdx.x, S = d.S, hw = d.h * d.w;
  const int r0 = blockIdx.y * kCamRows, r1 = min(S, r0 + kCamRows);
  if (tid == 0) {
    int c = 0;
    if (d.cls) {
      c = d.cls[i];
    } else {  // first argmax; a NaN counts as the maximum (torch.argmax)
      const float* l = d.logits + (long long)i * d.ncls;
      float best = l[0];
      for (int j = 1; j < d.ncls; ++j) {
        const float x = l[j];
        if (x > best || (x != x && best == best)) {
          best = x;
          c = j;
        }
      }
    }
    int4 b = make_int4(0, 0, S, S);
    if (d.boxes) b = make_int4(d.boxes[4LL * i], d.boxes[4LL * i + 1], d.boxes[4LL * i + 2], d.boxes[4LL * i + 3]);
    const bool ok = c >= 0 && c < d.ncls && 0 <= b.x && b.x < b.z && b.z <= S && 0 <= b.y && b.y < b.w && b.w <= S;
    s_cls = ok ? c : -1;
    s_box[0] = b.x;
    s_box[1] = b.y;
    s_box[2] = b.z;
    s_box[3] = b.w;
    if (blockIdx.y == 0 && d.status) d.status[i] = ok ? 0 : 1;
  }
  __syncthreads();
  const int c = s_cls;
  float* out = d.cam_map + (long long)i * S * S + (long long)r0 * S;
  const int n_out = (r1 - r0) * S;
  if (c < 0) {  // rejected entry: zeros, nothing read through it
    for (int k = tid; k < n_out; k += kCamThreads) out[k] = 0.0f;
    if (blockIdx.y == 0)
      for (int p = tid; p < hw; p += kCamThreads) d.cam[(long long)i * hw + p] = 0.0f;
    return;
  }
  const int x0 = s_box[0], y0 = s_box[1], bw = s_box[2] - x0, bh = s_box[3] - y0;
  const float* wrow = d.fc_w + (long long)c * d.C;
  for (int k = tid; k < d.C; k += kCamThreads) wc[k] = wrow[k];
  const double sx = (double)d.w / bw, sy = (double)d.h / bh;  // cv2 4.13: scale = ssize / dsize
  for (int x = tid; x < bw; x += kCamThreads) cv_coord(x, sx, d.w, &xs0[x], &xs1[x], &xw[x]);
  for (int r = tid; r < r1 - r0; r += kCamThreads)
    if (r0 + r >= y0 && r0 + r < y0 + bh) cv_coord(r0 + r - y0, sy, d.h, &ys0[r], &ys1[r], &yw[r]);
  __syncthreads();

  // cam[p] = max(0, sum_k W[c][k] * feat[p][k] / (h*w)): one warp per pixel, 8 channels per 16-byte load
  const int warp = tid >> 5, lane = tid & 31;
  const unsigned short* f = static_cast<const unsigned short*>(d.feat) + (long long)i * hw * d.C;  // bf16
  for (int p = warp; p < hw; p += kCamThreads / 32) {
    const uint4* fp = reinterpret_cast<const uint4*>(f + (long long)p * d.C);
    float acc = 0.0f;
#pragma unroll 4
    for (int k8 = lane; k8 < d.C / 8; k8 += 32) {  // unrolled: the four 16-byte loads of C = 1024 are in flight at once
      const uint4 q = __ldg(fp + k8);
      const float4 wa = *reinterpret_cast<const float4*>(wc + 8 * k8);
      const float4 wb = *reinterpret_cast<const float4*>(wc + 8 * k8 + 4);
      acc = __fmaf_rn(__uint_as_float(q.x << 16), wa.x, acc);  // bf16 -> fp32 is exact: the high half of the word
      acc = __fmaf_rn(__uint_as_float(q.x & 0xffff0000u), wa.y, acc);
      acc = __fmaf_rn(__uint_as_float(q.y << 16), wa.z, acc);
      acc = __fmaf_rn(__uint_as_float(q.y & 0xffff0000u), wa.w, acc);
      acc = __fmaf_rn(__uint_as_float(q.z << 16), wb.x, acc);
      acc = __fmaf_rn(__uint_as_float(q.z & 0xffff0000u), wb.y, acc);
      acc = __fmaf_rn(__uint_as_float(q.w << 16), wb.z, acc);
      acc = __fmaf_rn(__uint_as_float(q.w & 0xffff0000u), wb.w, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) v[p] = fmaxf(0.0f, __fdiv_rn(acc, (float)hw));
  }
  __syncthreads();

  // scale_cam_image (band 0 also stores the raw cam)
  if (warp == 0) cam_scale_warp(v, hw, lane, blockIdx.y == 0 ? d.cam + (long long)i * hw : nullptr);
  __syncthreads();

  // this band of cam_map: cv2.resize(v, (bw, bh), INTER_LINEAR) at (x0, y0), zero elsewhere
  for (int k = tid; k < n_out; k += kCamThreads) {
    const int r = k / S, x = k - r * S, y = r0 + r;
    float val = 0.0f;
    if (y >= y0 && y < y0 + bh && x >= x0 && x < x0 + bw) {
      const int dx = x - x0;
      val = cv_bilinear(v, d.w, ys0[r], ys1[r], yw[r], xs0[dx], xs1[dx], xw[dx]);
    }
    out[k] = val;
  }
}

int launch_cam(ug_engine* h, const ug_cam_desc* d, cudaStream_t s) {
  if (!d->feat || !d->fc_w || (!d->cls && !d->logits) || !d->cam || !d->cam_map || d->B <= 0 || d->h <= 0 ||
      d->w <= 0 || d->h > kCamMaxSide || d->w > kCamMaxSide || d->C <= 0 || d->C % 8 || d->C > kCamMaxC ||
      d->ncls <= 0 || d->S <= 0 || d->S > kCamMaxS || (reinterpret_cast<uintptr_t>(d->feat) & 15))
    return set_error(h, UG_EINVAL, "cam: bad args (h, w <= %d, C %% 8 == 0, C <= %d, S <= %d, feat 16-byte aligned)",
                     kCamMaxSide, kCamMaxC, kCamMaxS);
  const dim3 grid(d->B, ceil_div(d->S, kCamRows));
  h->launches += 1;
  return check_cuda(h, launch_pdl(cam_kernel, grid, kCamThreads, 0, s, *d), "cam launch");
}

}  // namespace ug
