// Source-frame outputs (ug_source_frame_desc): each image's segmentation mask, ROI box and Grad-CAM map carried from the
// SxS UNet input frame to the image's own H x W, as a user of the reference would draw them on the image they read:
// mask = sigmoid(cv2.resize(logits, (W, H), INTER_LINEAR)) > 0.5, the box scaled outwards to source pixels, and the
// normalised cam resized straight into that box.
//
// One launch over (kSfCtas CTAs per image, image); CTA x of image i takes the bands x, x + gridDim.x, ... of kSfRows
// output rows.  The grid depends on B, S and (uniform sources) Hs only, never on the table, which a plan image's host
// fills after the program is built.  Per CTA, the cv2 column coordinates of the image's W mask columns and of its box
// columns are built once in shared memory; per band, the logits rows the band reads are staged in shared memory,
// then the mask is written as aligned 4-byte words (ragged offsets have any alignment: a byte head and tail) and the
// CAM map as coalesced floats.  The op is bound by its writes (1 byte per source pixel, 4 more with the map).
#include <cstdint>
#include "cam_scale.cuh"
#include "common.cuh"
#include "cv_resize.cuh"
#include "engine.h"

namespace ug {

static constexpr int kSfThreads = 256;
static constexpr int kSfRows = 8;           // output rows per band
static constexpr int kSfMaxS = 256;
static constexpr int kSfMaxRatio = 8;       // source sides up to 8*S, as ug_resize_ragged
static constexpr int kSfMaxSide = kSfMaxRatio * kSfMaxS;
static constexpr int kSfCamMaxSide = 32;    // h, w
static constexpr int kSfTargetCtas = 4096;  // CTAs per launch when the images are tall enough (~5.5 waves)

__global__ void __launch_bounds__(kSfThreads, 5) source_frame_kernel(ug_source_frame_desc d) {
  __shared__ __align__(16) float stage[2 * kSfRows * kSfMaxS];  // the logits rows one band reads
  __shared__ unsigned short xs[kSfMaxSide];                      // cv2 x coordinate of each mask column
  __shared__ float xw[kSfMaxSide];
  __shared__ unsigned char cxs[kSfMaxSide];                      // ... of each column of the CAM map's box
  __shared__ float cxw[kSfMaxSide];
  __shared__ float v[kSfCamMaxSide * kSfCamMaxSide];             // the normalised cam
  __shared__ int slot0[kSfRows], slot1[kSfRows], rows[2 * kSfRows];  // stage slots of each output row's rows
  __shared__ float yw[kSfRows];
  __shared__ int cys0[kSfRows], cys1[kSfRows];
  __shared__ float cyw[kSfRows];
  __shared__ long long s_off;
  __shared__ int s_ok, s_H, s_W, s_box[4];
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int i = blockIdx.y, tid = threadIdx.x, S = d.S;
  if (tid == 0) {
    long long off;
    int H, W;
    bool ok = true;
    if (d.index) {
      const ug_ragged_image e = d.index[i];
      off = e.px_offset;
      H = e.H;
      W = e.W;
      ok = off >= 0 && H >= 1 && W >= 1 && H <= kSfMaxRatio * S && W <= kSfMaxRatio * S && off <= d.capacity_px &&
           (long long)H * W <= d.capacity_px - off;
    } else {
      H = d.Hs;
      W = d.Ws;
      off = (long long)i * H * W;
    }
    const int x0 = d.boxes[4LL * i], y0 = d.boxes[4LL * i + 1], x1 = d.boxes[4LL * i + 2], y1 = d.boxes[4LL * i + 3];
    ok = ok && 0 <= x0 && x0 < x1 && x1 <= S && 0 <= y0 && y0 < y1 && y1 <= S;
    // the smallest source-pixel box covering the S-frame box, in 64-bit integers (all terms are non-negative)
    int b[4] = {0, 0, 0, 0};
    if (ok) {
      b[0] = (int)((long long)x0 * W / S);
      b[1] = (int)((long long)y0 * H / S);
      b[2] = (int)(((long long)x1 * W + S - 1) / S);
      b[3] = (int)(((long long)y1 * H + S - 1) / S);
    }
    if (blockIdx.x == 0) {
      for (int k = 0; k < 4; ++k) d.src_boxes[4LL * i + k] = b[k];
      if (d.status) d.status[i] = ok ? 0 : 1;
    }
    s_ok = ok;
    s_off = off;
    s_H = H;
    s_W = W;
    for (int k = 0; k < 4; ++k) s_box[k] = b[k];
  }
  __syncthreads();
  if (!s_ok) return;  // rejected entry: nothing is read or written through it
  const int H = s_H, W = s_W, X0 = s_box[0], Y0 = s_box[1], bw = s_box[2] - X0, bh = s_box[3] - Y0;
  const bool cam = d.cam != nullptr;
  const int warp = tid >> 5, lane = tid & 31;
  const double sx = (double)S / W, sy = (double)S / H;  // cv2 4.13: scale = ssize / dsize
  const double csx = (double)d.w / bw, csy = (double)d.h / bh;
  for (int x = tid; x < W; x += kSfThreads) {
    int a, b;
    float f;
    cv_coord(x, sx, S, &a, &b, &f);
    xs[x] = (unsigned short)a;
    xw[x] = f;
  }
  if (cam) {
    for (int x = tid; x < bw; x += kSfThreads) {
      int a, b;
      float f;
      cv_coord(x, csx, d.w, &a, &b, &f);
      cxs[x] = (unsigned char)a;
      cxw[x] = f;
    }
    const int hw = d.h * d.w;
    for (int p = tid; p < hw; p += kSfThreads) v[p] = d.cam[(long long)i * hw + p];
    __syncthreads();
    if (warp == 0) cam_scale_warp(v, hw, lane, nullptr);  // made visible by the first barrier of the band loop
  }

  unsigned char* mimg = d.mask + s_off;
  float* cimg = cam ? d.cam_map + s_off : nullptr;
  const float4* lg = reinterpret_cast<const float4*>(d.logits + (long long)i * S * S);
  const int q = S / 4;  // float4 per logits row
  const int n_bands = (H + kSfRows - 1) / kSfRows;
  for (int band = blockIdx.x; band < n_bands; band += gridDim.x) {
    const int r0 = band * kSfRows, nr = min(kSfRows, H - r0);
    // The stage holds the contiguous run of source rows the band reads when it fits (always when H >= S), else the
    // two rows of each output row.
    int lo, hi, a, b;
    float f;
    cv_coord(r0, sy, S, &lo, &b, &f);
    cv_coord(r0 + nr - 1, sy, S, &a, &hi, &f);
    const bool run = hi - lo < 2 * kSfRows;
    if (tid < nr) {
      cv_coord(r0 + tid, sy, S, &a, &b, &f);
      slot0[tid] = run ? a - lo : 2 * tid;
      slot1[tid] = run ? b - lo : 2 * tid + 1;
      rows[2 * tid] = a;
      rows[2 * tid + 1] = b;
      yw[tid] = f;
    } else if (cam && tid >= 32 && tid < 32 + nr) {
      const int y = r0 + tid - 32 - Y0;
      if (y >= 0 && y < bh) {
        cv_coord(y, csy, d.h, &a, &b, &f);
        cys0[tid - 32] = a;
        cys1[tid - 32] = b;
        cyw[tid - 32] = f;
      }
    }
    __syncthreads();
    const int n_stage = run ? hi - lo + 1 : 2 * nr;
    for (int k = tid; k < n_stage * q; k += kSfThreads) {
      const int j = k / q;
      reinterpret_cast<float4*>(stage)[k] = __ldg(lg + (long long)(run ? lo + j : rows[j]) * q + (k - j * q));
    }
    __syncthreads();

    // mask: pixel p of the band is row p / W, column p % W; the band is one contiguous byte range of the image
    const int n = nr * W;
    unsigned char* dst = mimg + (long long)r0 * W;
    const int head = min(n, (int)((4u - (unsigned)(reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u));
    const int n_words = (n - head) >> 2, tail = head + 4 * n_words;
    auto px = [&](int r, int x) -> unsigned {
      const int c = xs[x];
      const float l = cv_bilinear(stage, S, slot0[r], slot1[r], yw[r], c, min(c + 1, S - 1), xw[x]);
      // the OUTC epilogues' torch.sigmoid(seg_out) > 0.5 in fp32.  For |l| > 1e-3 the fp32 sigmoid is at least 2.5e-4
      // away from 0.5, far beyond its rounding error, so it equals l > 0 there (also for +-inf); NaN takes the full form
      if (fabsf(l) > 1e-3f) return l > 0.0f ? 1u : 0u;
      return 1.0f / (1.0f + expf(-l)) > 0.5f ? 1u : 0u;
    };
    {
      // Lane l of a warp evaluates pixels base + 32j + l (j < 4, consecutive lanes read consecutive table entries);
      // four ballots give the warp's 128 mask bits, and lane l writes the word of pixels base + 4l .. base + 4l + 3.
      const int warps = kSfThreads / 32, end = tail;
      int p = head + 128 * warp + lane, r = p / W, x = p - r * W;  // advanced 32 pixels per step
      for (int w0 = 32 * warp; w0 < n_words; w0 += 32 * warps) {
        unsigned bits[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          bits[j] = __ballot_sync(0xffffffffu, p < end && px(r, x));
          p += 32;
          x += 32;
          if (x >= W) {
            const int t = x / W;
            r += t;
            x -= t * W;
          }
        }
        const unsigned q4 = lane < 8 ? bits[0] : lane < 16 ? bits[1] : lane < 24 ? bits[2] : bits[3];
        const unsigned nib = (q4 >> ((4 * lane) & 31)) & 0xFu;
        if (w0 + lane < n_words)
          reinterpret_cast<unsigned*>(dst + head)[w0 + lane] =
              (nib & 1u) | ((nib >> 1) & 1u) << 8 | ((nib >> 2) & 1u) << 16 | (nib >> 3) << 24;
        p += 128 * (warps - 1);
        x += 128 * (warps - 1);
        if (x >= W) {
          const int t = x / W;
          r += t;
          x -= t * W;
        }
      }
    }
    if (tid < head) {
      dst[tid] = (unsigned char)px(tid / W, tid % W);
    } else if (tid >= 32 && tid - 32 < n - tail) {
      const int p = tail + tid - 32;
      dst[p] = (unsigned char)px(p / W, p % W);
    }

    // CAM map: cv2.resize(v, (bw, bh), INTER_LINEAR) at (X0, Y0), zero elsewhere
    if (cam) {
      float* cdst = cimg + (long long)r0 * W;
      int r = tid / W, x = tid - r * W;  // advanced by kSfThreads pixels per step
      for (int k = tid; k < n; k += kSfThreads) {
        const int y = r0 + r, dx = x - X0;
        float val = 0.0f;
        if (y >= Y0 && y < Y0 + bh && dx >= 0 && dx < bw) {
          const int c = cxs[dx];
          val = cv_bilinear(v, d.w, cys0[r], cys1[r], cyw[r], c, min(c + 1, d.w - 1), cxw[dx]);
        }
        cdst[k] = val;
        x += kSfThreads;
        if (x >= W) {
          const int t = x / W;
          r += t;
          x -= t * W;
        }
      }
    }
    __syncthreads();  // the next band overwrites the row tables and the stage
  }
}

int launch_source_frame(ug_engine* h, const ug_source_frame_desc* d, cudaStream_t s) {
  const bool cam = d->cam != nullptr;
  const int smax = kSfMaxRatio * d->S;
  if (!d->logits || !d->boxes || !d->mask || !d->src_boxes || cam != (d->cam_map != nullptr) || d->B <= 0 ||
      d->B > 65535 || d->S <= 0 || d->S > kSfMaxS || d->S % 4 || (reinterpret_cast<uintptr_t>(d->logits) & 15) ||
      (cam && (d->h <= 0 || d->w <= 0 || d->h > kSfCamMaxSide || d->w > kSfCamMaxSide)) ||
      (d->index ? d->capacity_px <= 0 : (d->Hs < 1 || d->Ws < 1 || d->Hs > smax || d->Ws > smax)))
    return set_error(h, UG_EINVAL,
                     "source_frame: bad args (cam and cam_map both or neither, h, w <= %d, S <= %d and a multiple of 4, "
                     "logits 16-byte aligned, Hs, Ws in [1, 8*S] or a table with capacity_px > 0)",
                     kSfCamMaxSide, kSfMaxS);
  const int h_max = d->index ? smax : d->Hs;  // the table is not read here: size the grid for the tallest image allowed
  const dim3 grid(std::min(ceil_div(h_max, kSfRows), std::max(1, ceil_div(kSfTargetCtas, d->B))), d->B);
  h->launches += 1;
  return check_cuda(h, launch_pdl(source_frame_kernel, grid, kSfThreads, 0, s, *d), "source_frame launch");
}

}  // namespace ug
