// Device restatement of the reference's `wavelet_enhance` (分类/test.py:17-63): grayscale uint8 image -> pseudo-RGB
// uint8 HWC (R = normalised image, G = normalised single-level Haar approximation resized back, B = normalised Haar
// detail magnitude resized back).  SURVEY §8f.2: the host pre-processing step in front of the stage-2 path.
//
//   K1 wavelet_dwt_kernel      Haar analysis in float32 exactly as PyWavelets orders it (axis 0 then axis 1,
//                              out = f*x[2o+1] + f*x[2o], 'symmetric' extension for odd sizes), cA and
//                              sqrt(cH^2+cV^2+cD^2) at half resolution into the workspace; min / max of the image
//   K2 wavelet_up_kernel<0>    min / max of the two bilinearly up-sampled half-resolution maps (cv2.resize
//                              INTER_LINEAR restated bit-exactly: half-pixel centres, replicated border, fused lerp)
//   K3 wavelet_up_kernel<1>    recomputes the up-sampling, applies the reference's normalize()
//                              ((x - min) / max(x - min) * 255 truncated to uint8) and writes HWC
// The wavelet_ragged_* kernels run the same per-image functions over a ragged batch (ug_wavelet_ragged_desc).
// All three are memory-light (one 8-bit image in, three out).  Non-negative floats are reduced with integer atomics
// on their bit patterns (order-preserving for x >= 0; every value here is >= 0).
#include <cfloat>
#include "common.cuh"
#include "cv_resize.cuh"
#include "engine.h"

namespace ug {

static constexpr float kHaar = 0.70710678118654752440f;  // float32(1/sqrt(2)), pywt's haar dec_lo / dec_hi

struct WvStats {  // per image, float bit patterns (all values >= 0)
  unsigned gmin, gmax, lmin, lmax, hmin, hmax, pad0, pad1;
};

__global__ void wavelet_init_kernel(WvStats* st, int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) {
    st[i].gmin = st[i].lmin = st[i].hmin = 0x7F7FFFFFu;  // FLT_MAX
    st[i].gmax = st[i].lmax = st[i].hmax = 0u;
  }
}

__device__ __forceinline__ void block_minmax(float mn, float mx, unsigned* gmn, unsigned* gmx) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(gmn, __float_as_uint(mn));
    atomicMax(gmx, __float_as_uint(mx));
  }
}

// The per-image arithmetic below is shared by the uniform kernels (one [B][H][W] batch) and the ragged ones (image n
// described by a table entry); each __global__ kernel only locates image n and calls it.

// min / max of the gray image (needed first: the reference rescales by 255 when max <= 1)
__device__ __forceinline__ void wv_gray_minmax(const unsigned char* __restrict__ g, int HW, WvStats* st) {
  float mn = FLT_MAX, mx = 0.0f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += gridDim.x * blockDim.x) {
    const float v = (float)g[i];
    mn = fminf(mn, v);
    mx = fmaxf(mx, v);
  }
  block_minmax(mn, mx, &st->gmin, &st->gmax);
}

// half-resolution pixel i of cA and of the detail magnitude
__device__ __forceinline__ void wv_dwt_px(const unsigned char* __restrict__ g, const WvStats* st, float* __restrict__ cA,
                                          float* __restrict__ hf, int H, int W, int w2, int i) {
  const int oy = i / w2, ox = i - oy * w2;
  const float sc = __uint_as_float(st->gmax) <= 1.0f ? 255.0f : 1.0f;  // `if gray_img.max() <= 1.0: *= 255`
  const int y0 = 2 * oy, y1 = min(2 * oy + 1, H - 1), x0 = 2 * ox, x1 = min(2 * ox + 1, W - 1);  // symmetric extension
  const float p00 = __fmul_rn((float)g[y0 * W + x0], sc), p01 = __fmul_rn((float)g[y0 * W + x1], sc);
  const float p10 = __fmul_rn((float)g[y1 * W + x0], sc), p11 = __fmul_rn((float)g[y1 * W + x1], sc);
  // axis 0 (rows): lo = f*x[2o+1] + f*x[2o], hi = -f*x[2o+1] + f*x[2o]   (separate fp32 multiply and add)
  const float a_x0 = __fadd_rn(__fmul_rn(kHaar, p10), __fmul_rn(kHaar, p00));
  const float a_x1 = __fadd_rn(__fmul_rn(kHaar, p11), __fmul_rn(kHaar, p01));
  const float d_x0 = __fadd_rn(__fmul_rn(-kHaar, p10), __fmul_rn(kHaar, p00));
  const float d_x1 = __fadd_rn(__fmul_rn(-kHaar, p11), __fmul_rn(kHaar, p01));
  // axis 1 (columns)
  const float aa = __fadd_rn(__fmul_rn(kHaar, a_x1), __fmul_rn(kHaar, a_x0));
  const float ad = __fadd_rn(__fmul_rn(-kHaar, a_x1), __fmul_rn(kHaar, a_x0));
  const float da = __fadd_rn(__fmul_rn(kHaar, d_x1), __fmul_rn(kHaar, d_x0));
  const float dd = __fadd_rn(__fmul_rn(-kHaar, d_x1), __fmul_rn(kHaar, d_x0));
  cA[i] = aa;
  // np.sqrt(cH**2 + cV**2 + cD**2) with cH = da, cV = ad, cD = dd
  hf[i] = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(da, da), __fmul_rn(ad, ad)), __fmul_rn(dd, dd)));
}

// kWrite = false: min / max of the two up-sampled maps into st.  kWrite = true: normalise and write HWC to out.
template <bool kWrite>
__device__ __forceinline__ void wv_up(const unsigned char* __restrict__ g, WvStats* st, const float* __restrict__ a,
                                      const float* __restrict__ hh, unsigned char* __restrict__ out, int H, int W, int h2,
                                      int w2) {
  const double sx = 1.0 / ((double)W / w2), sy = 1.0 / ((double)H / h2);  // cv2: scale = 1 / (dsize / ssize)
  float lmn = FLT_MAX, lmx = 0.0f, hmn = FLT_MAX, hmx = 0.0f;
  float gmin = 0.f, gmax = 0.f, lmin = 0.f, lmax = 0.f, hmin = 0.f, hmax = 0.f, gsc = 1.0f;
  if (kWrite) {
    gsc = __uint_as_float(st->gmax) <= 1.0f ? 255.0f : 1.0f;
    gmin = __fmul_rn(__uint_as_float(st->gmin), gsc);
    gmax = __fmul_rn(__uint_as_float(st->gmax), gsc);
    lmin = __uint_as_float(st->lmin);
    lmax = __uint_as_float(st->lmax);
    hmin = __uint_as_float(st->hmin);
    hmax = __uint_as_float(st->hmax);
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < H * W; i += gridDim.x * blockDim.x) {
    const int y = i / W, x = i - y * W;
    int x0, x1, y0, y1;
    float wx, wy;
    cv_coord(x, sx, w2, &x0, &x1, &wx);
    cv_coord(y, sy, h2, &y0, &y1, &wy);
    const float lo = cv_bilinear(a, w2, y0, y1, wy, x0, x1, wx);
    const float hi = cv_bilinear(hh, w2, y0, y1, wy, x0, x1, wx);
    if (!kWrite) {
      lmn = fminf(lmn, lo);
      lmx = fmaxf(lmx, lo);
      hmn = fminf(hmn, hi);
      hmx = fmaxf(hmx, hi);
    } else {
      // normalize(): x = x - min; if max(x) != 0: x = x / max(x); (x * 255).astype(uint8)   (fp32, truncation)
      const float gv = __fmul_rn((float)g[i], gsc);
      float v[3] = {__fadd_rn(gv, -gmin), __fadd_rn(lo, -lmin), __fadd_rn(hi, -hmin)};
      const float mx[3] = {__fadd_rn(gmax, -gmin), __fadd_rn(lmax, -lmin), __fadd_rn(hmax, -hmin)};
      unsigned char* o = out + (long long)i * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (mx[c] != 0.0f) v[c] = __fdiv_rn(v[c], mx[c]);
        o[c] = (unsigned char)(int)__fmul_rn(v[c], 255.0f);
      }
    }
  }
  if (!kWrite) {
    block_minmax(lmn, lmx, &st->lmin, &st->lmax);
    block_minmax(hmn, hmx, &st->hmin, &st->hmax);
  }
}

// ---------------------------------------------------------------- uniform batch [B][H][W]
__global__ void __launch_bounds__(256) wavelet_gray_stats_kernel(const unsigned char* __restrict__ gray, WvStats* st,
                                                                 int HW) {
  const int n = blockIdx.y;
  wv_gray_minmax(gray + (long long)n * HW, HW, &st[n]);
}

__global__ void __launch_bounds__(256) wavelet_dwt_kernel(const unsigned char* __restrict__ gray, const WvStats* st,
                                                          float* __restrict__ cA, float* __restrict__ hf, int H, int W,
                                                          int h2, int w2) {
  const int n = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= h2 * w2) return;
  const long long o = (long long)n * h2 * w2;
  wv_dwt_px(gray + (long long)n * H * W, &st[n], cA + o, hf + o, H, W, w2, i);
}

template <bool kWrite>
__global__ void __launch_bounds__(256) wavelet_up_kernel(const unsigned char* __restrict__ gray, WvStats* st,
                                                         const float* __restrict__ cA, const float* __restrict__ hf,
                                                         unsigned char* __restrict__ out, int H, int W, int h2, int w2) {
  const int n = blockIdx.y;
  const long long o = (long long)n * h2 * w2;
  wv_up<kWrite>(gray + (long long)n * H * W, &st[n], cA + o, hf + o, kWrite ? out + (long long)n * H * W * 3 : nullptr, H,
                W, h2, w2);
}

// ---------------------------------------------------------------- ragged batch (ug_wavelet_ragged_desc)
// Image n: gray + off, out + 3*off, and its cA / detail maps at workspace offset `off` (h2*w2 <= H*W, so the slices of
// disjoint images are disjoint).  The table is checked entry by entry; a bad entry is skipped by every kernel.
static constexpr int kWvMaxSide = 32768;

struct WvRagged {
  const ug_ragged_image* index;
  int* status;
  long long capacity_px;
};

__device__ __forceinline__ bool wv_entry(const WvRagged& rg, int n, ug_ragged_image* e) {
  *e = rg.index[n];
  return e->px_offset >= 0 && e->H >= 2 && e->W >= 2 && e->H <= kWvMaxSide && e->W <= kWvMaxSide &&
         e->px_offset <= rg.capacity_px && (long long)e->H * e->W <= rg.capacity_px - e->px_offset;
}

__global__ void wavelet_ragged_init_kernel(WvStats* st, WvRagged rg, int B) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) {
    st[i].gmin = st[i].lmin = st[i].hmin = 0x7F7FFFFFu;  // FLT_MAX
    st[i].gmax = st[i].lmax = st[i].hmax = 0u;
    ug_ragged_image e;
    const bool ok = wv_entry(rg, i, &e);
    if (rg.status) rg.status[i] = ok ? 0 : 1;
  }
}

__global__ void __launch_bounds__(256) wavelet_ragged_gray_stats_kernel(const unsigned char* __restrict__ gray,
                                                                        WvStats* st, WvRagged rg) {
  pdl_wait();
  pdl_launch_dependents();
  const int n = blockIdx.y;
  ug_ragged_image e;
  if (!wv_entry(rg, n, &e)) return;
  wv_gray_minmax(gray + e.px_offset, e.H * e.W, &st[n]);
}

__global__ void __launch_bounds__(256) wavelet_ragged_dwt_kernel(const unsigned char* __restrict__ gray,
                                                                 const WvStats* st, float* __restrict__ cA,
                                                                 float* __restrict__ hf, WvRagged rg) {
  pdl_wait();
  pdl_launch_dependents();
  const int n = blockIdx.y;
  ug_ragged_image e;
  if (!wv_entry(rg, n, &e)) return;
  const int h2 = (e.H + 1) / 2, w2 = (e.W + 1) / 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < h2 * w2; i += gridDim.x * blockDim.x)
    wv_dwt_px(gray + e.px_offset, &st[n], cA + e.px_offset, hf + e.px_offset, e.H, e.W, w2, i);
}

template <bool kWrite>
__global__ void __launch_bounds__(256) wavelet_ragged_up_kernel(const unsigned char* __restrict__ gray, WvStats* st,
                                                                const float* __restrict__ cA, const float* __restrict__ hf,
                                                                unsigned char* __restrict__ out, WvRagged rg) {
  pdl_wait();
  pdl_launch_dependents();
  const int n = blockIdx.y;
  ug_ragged_image e;
  if (!wv_entry(rg, n, &e)) return;
  wv_up<kWrite>(gray + e.px_offset, &st[n], cA + e.px_offset, hf + e.px_offset, kWrite ? out + 3 * e.px_offset : nullptr,
                e.H, e.W, (e.H + 1) / 2, (e.W + 1) / 2);
}

int launch_wavelet(ug_engine* h, const ug_wavelet_desc* d, cudaStream_t s) {
  if (!d->gray || !d->out_u8 || !d->workspace || d->B <= 0 || d->H < 2 || d->W < 2)
    return set_error(h, UG_EINVAL, "wavelet: bad args (H, W >= 2)");
  const int h2 = (d->H + 1) / 2, w2 = (d->W + 1) / 2;
  const size_t need = ug_wavelet_workspace_bytes(d->B, d->H, d->W);
  if (d->workspace_bytes < need) return set_error(h, UG_EINVAL, "wavelet: workspace too small (%zu < %zu)", d->workspace_bytes, need);
  WvStats* st = static_cast<WvStats*>(d->workspace);
  float* cA = reinterpret_cast<float*>(st + ((d->B + 3) / 4) * 4);
  float* hf = cA + (size_t)d->B * h2 * w2;
  const int HW = d->H * d->W;
  const dim3 gfull(std::min(ceil_div(HW, 256), 64), d->B);
  wavelet_init_kernel<<<ceil_div(d->B, 128), 128, 0, s>>>(st, d->B);
  wavelet_gray_stats_kernel<<<gfull, 256, 0, s>>>(d->gray, st, HW);
  wavelet_dwt_kernel<<<dim3(ceil_div((long long)h2 * w2, 256), d->B), 256, 0, s>>>(d->gray, st, cA, hf, d->H, d->W, h2, w2);
  wavelet_up_kernel<false><<<gfull, 256, 0, s>>>(d->gray, st, cA, hf, nullptr, d->H, d->W, h2, w2);
  wavelet_up_kernel<true><<<gfull, 256, 0, s>>>(d->gray, st, cA, hf, d->out_u8, d->H, d->W, h2, w2);
  h->launches += 5;
  return check_cuda(h, cudaGetLastError(), "wavelet launch");
}

int launch_wavelet_ragged(ug_engine* h, const ug_wavelet_ragged_desc* d, cudaStream_t s) {
  if (!d->gray || !d->index || !d->out_u8 || !d->workspace || d->B <= 0 || d->capacity_px <= 0)
    return set_error(h, UG_EINVAL, "wavelet_ragged: bad args");
  const size_t need = ug_wavelet_ragged_workspace_bytes(d->B, d->capacity_px);
  if (d->workspace_bytes < need)
    return set_error(h, UG_EINVAL, "wavelet_ragged: workspace too small (%zu < %zu)", d->workspace_bytes, need);
  WvStats* st = static_cast<WvStats*>(d->workspace);
  float* cA = reinterpret_cast<float*>(st + ((d->B + 3) / 4) * 4);
  float* hf = cA + d->capacity_px;
  const WvRagged rg{d->index, d->status, d->capacity_px};
  // The table lives on the device, so the grid is sized from the capacity (a bound on the largest image) and every
  // kernel strides over its image; blocks past an image's extent do no work.
  const dim3 grid(std::min(ceil_div(d->capacity_px, 256), 64), d->B);
  int rc = check_cuda(h, launch_pdl(wavelet_ragged_init_kernel, ceil_div(d->B, 128), 128, 0, s, st, rg, d->B), "wavelet_ragged init");
  if (rc == UG_OK)
    rc = check_cuda(h, launch_pdl(wavelet_ragged_gray_stats_kernel, grid, 256, 0, s, d->gray, st, rg), "wavelet_ragged stats");
  if (rc == UG_OK)
    rc = check_cuda(h, launch_pdl(wavelet_ragged_dwt_kernel, grid, 256, 0, s, d->gray, st, cA, hf, rg), "wavelet_ragged dwt");
  if (rc == UG_OK)
    rc = check_cuda(h, launch_pdl(wavelet_ragged_up_kernel<false>, grid, 256, 0, s, d->gray, st, cA, hf, nullptr, rg),
                    "wavelet_ragged up");
  if (rc == UG_OK)
    rc = check_cuda(h, launch_pdl(wavelet_ragged_up_kernel<true>, grid, 256, 0, s, d->gray, st, cA, hf, d->out_u8, rg),
                    "wavelet_ragged up");
  h->launches += 5;
  return rc;
}

}  // namespace ug

extern "C" size_t ug_wavelet_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  const size_t h2 = (H + 1) / 2, w2 = (W + 1) / 2;
  return (size_t)((B + 3) / 4) * 4 * sizeof(ug::WvStats) + 2 * (size_t)B * h2 * w2 * sizeof(float);
}

extern "C" size_t ug_wavelet_ragged_workspace_bytes(int B, long long capacity_px) {
  if (B <= 0 || capacity_px <= 0) return 0;
  return (size_t)((B + 3) / 4) * 4 * sizeof(ug::WvStats) + 2 * (size_t)capacity_px * sizeof(float);
}
