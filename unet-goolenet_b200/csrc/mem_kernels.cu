// Memory-bound kernels of the hot path (NHWC bf16 activations, 16-byte vector accesses, coalesced along C):
// max pooling, LayerNorm, attention, CoordAtt3 statistics + gate, mask -> bbox,
// PIL-exact crop/resize and the GoogLeNet head.  Reference lines are cited on the descriptors in ugnet.h.
#include <cfloat>
#include <cmath>
#include <algorithm>
#include "common.cuh"
#include "engine.h"

namespace ug {

// ------------------------------------------------------------------------------------------------
// max pooling: one thread per (output pixel, 8-channel group); channel groups vary fastest.
__global__ void __launch_bounds__(256) pool_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                   ug_pool_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int cg = d.C / 8;
  const long long total = (long long)d.B * d.OH * d.OW * cg;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int g = (int)(t % cg);
  long long pp = t / cg;
  const int ox = (int)(pp % d.OW);
  pp /= d.OW;
  const int oy = (int)(pp % d.OH);
  const int n = (int)(pp / d.OH);
  const uint32_t ninf = 0xFF80FF80u;  // (-inf, -inf) in bf16
  uint4 m = make_uint4(ninf, ninf, ninf, ninf);
  for (int r = 0; r < d.k; ++r) {
    const int iy = oy * d.stride + r - d.pad;
    if (iy < 0 || iy >= d.H) continue;
    for (int s = 0; s < d.k; ++s) {
      const int ix = ox * d.stride + s - d.pad;
      if (ix < 0 || ix >= d.W) continue;
      const uint4 v =
          *reinterpret_cast<const uint4*>(in + (((long long)n * d.H + iy) * d.W + ix) * d.in_cstride + g * 8);
      m.x = bf16x2_max(m.x, v.x);
      m.y = bf16x2_max(m.y, v.y);
      m.z = bf16x2_max(m.z, v.z);
      m.w = bf16x2_max(m.w, v.w);
    }
  }
  *reinterpret_cast<uint4*>(out + (((long long)n * d.OH + oy) * d.OW + ox) * d.out_cstride + g * 8) = m;
}

// 3x3 stride-1 pad-1 max pooling (the Inception branch4 pools): one thread per (image, output row, 8-channel group)
// slides along the row keeping the last three column maxima, so every input pixel is loaded three times instead of
// nine (these maps are L2 resident and the generic kernel was bound by the 9x re-read).
__global__ void __launch_bounds__(256) pool3x3s1_kernel(const __nv_bfloat16* __restrict__ in,
                                                        __nv_bfloat16* __restrict__ out, ug_pool_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int cg = d.C / 8;
  const long long total = (long long)d.B * d.H * cg;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int g = (int)(t % cg);
  const long long pp = t / cg;
  const int oy = (int)(pp % d.H);
  const int n = (int)(pp / d.H);
  const uint32_t ninf = 0xFF80FF80u;  // (-inf, -inf) in bf16
  const uint4 vinf = make_uint4(ninf, ninf, ninf, ninf);
  const int r0 = oy > 0 ? oy - 1 : oy, r1 = oy + 1 < d.H ? oy + 1 : oy;   // valid input rows r0..r1
  const __nv_bfloat16* base = in + ((long long)n * d.H * d.W) * d.in_cstride + g * 8;
  auto colmax = [&](int x) {
    uint4 m = vinf;
    for (int r = r0; r <= r1; ++r) {
      const uint4 v = *reinterpret_cast<const uint4*>(base + ((long long)r * d.W + x) * d.in_cstride);
      m.x = bf16x2_max(m.x, v.x);
      m.y = bf16x2_max(m.y, v.y);
      m.z = bf16x2_max(m.z, v.z);
      m.w = bf16x2_max(m.w, v.w);
    }
    return m;
  };
  uint4 a = vinf, b = colmax(0);  // column maxima at x-1 and x
  __nv_bfloat16* orow = out + (((long long)n * d.H + oy) * d.W) * d.out_cstride + g * 8;
  for (int x = 0; x < d.W; ++x) {
    const uint4 c = x + 1 < d.W ? colmax(x + 1) : vinf;
    uint4 m;
    m.x = bf16x2_max(bf16x2_max(a.x, b.x), c.x);
    m.y = bf16x2_max(bf16x2_max(a.y, b.y), c.y);
    m.z = bf16x2_max(bf16x2_max(a.z, b.z), c.z);
    m.w = bf16x2_max(bf16x2_max(a.w, b.w), c.w);
    *reinterpret_cast<uint4*>(orow + (long long)x * d.out_cstride) = m;
    a = b;
    b = c;
  }
}

// 3x3 stride-2 pad-0 ceil-mode max pooling (GoogLeNet maxpool1-4): one thread per (image, 2x2 block of output pixels,
// 8-channel group).  The four windows of a block cover 5x5 input pixels: 25 independent loads for four outputs (6.25
// per output instead of 9; the generic kernel ran at 52-55 % of the HBM peak with the L2 -> SM path at ~7 TB/s).
// A sliding-window form (one thread per output row, 6 loads per output) was slower: too few, too serial threads
// (profiles/r02_pool_s2.txt).  Columns / rows past the map (ceil mode) are skipped = -inf padding.
__global__ void __launch_bounds__(256) pool3x3s2_kernel(const __nv_bfloat16* __restrict__ in,
                                                        __nv_bfloat16* __restrict__ out, ug_pool_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int cg = d.C / 8;
  const int bw = (d.OW + 1) >> 1, bh = (d.OH + 1) >> 1;
  const int total = d.B * bh * bw * cg;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int g = t % cg;
  int pp = t / cg;
  const int bx = pp % bw;
  pp /= bw;
  const int by = pp % bh;
  const int n = pp / bh;
  const uint32_t ninf = 0xFF80FF80u;  // (-inf, -inf) in bf16
  const uint4 vinf = make_uint4(ninf, ninf, ninf, ninf);
  auto vmax = [](const uint4& a, const uint4& b) {
    return make_uint4(bf16x2_max(a.x, b.x), bf16x2_max(a.y, b.y), bf16x2_max(a.z, b.z), bf16x2_max(a.w, b.w));
  };
  const int y0 = 4 * by, x0 = 4 * bx;
  const __nv_bfloat16* base = in + ((long long)n * d.H * d.W) * d.in_cstride + g * 8;
  uint4 o[2][2] = {{vinf, vinf}, {vinf, vinf}};
#pragma unroll
  for (int c = 0; c < 5; ++c) {
    uint4 v[5];
#pragma unroll
    for (int r = 0; r < 5; ++r)
      v[r] = (y0 + r < d.H && x0 + c < d.W)
                 ? *reinterpret_cast<const uint4*>(base + ((long long)(y0 + r) * d.W + x0 + c) * d.in_cstride)
                 : vinf;
    const uint4 top = vmax(vmax(v[0], v[1]), v[2]), bot = vmax(vmax(v[2], v[3]), v[4]);
    if (c <= 2) {
      o[0][0] = vmax(o[0][0], top);
      o[1][0] = vmax(o[1][0], bot);
    }
    if (c >= 2) {
      o[0][1] = vmax(o[0][1], top);
      o[1][1] = vmax(o[1][1], bot);
    }
  }
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int oy = 2 * by + dy, ox = 2 * bx + dx;
      if (oy < d.OH && ox < d.OW)
        *reinterpret_cast<uint4*>(out + (((long long)n * d.OH + oy) * d.OW + ox) * d.out_cstride + g * 8) = o[dy][dx];
    }
}

// 3x3 stride-1 pad-1 max pooling, block form: one thread per (image, 2x2 block of output pixels, 8-channel group): the four
// windows cover 4x4 input pixels, 16 independent loads for four outputs.
__global__ void __launch_bounds__(256) pool3x3s1_block_kernel(const __nv_bfloat16* __restrict__ in,
                                                              __nv_bfloat16* __restrict__ out, ug_pool_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int cg = d.C / 8;
  const int bw = (d.W + 1) >> 1, bh = (d.H + 1) >> 1;
  const int total = d.B * bh * bw * cg;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int g = t % cg;
  int pp = t / cg;
  const int bx = pp % bw;
  pp /= bw;
  const int by = pp % bh;
  const int n = pp / bh;
  const uint32_t ninf = 0xFF80FF80u;  // (-inf, -inf) in bf16
  const uint4 vinf = make_uint4(ninf, ninf, ninf, ninf);
  auto vmax = [](const uint4& a, const uint4& b) {
    return make_uint4(bf16x2_max(a.x, b.x), bf16x2_max(a.y, b.y), bf16x2_max(a.z, b.z), bf16x2_max(a.w, b.w));
  };
  const int y0 = 2 * by - 1, x0 = 2 * bx - 1;
  const __nv_bfloat16* base = in + ((long long)n * d.H * d.W) * d.in_cstride + g * 8;
  uint4 o[2][2] = {{vinf, vinf}, {vinf, vinf}};
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint4 v[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int y = y0 + r, x = x0 + c;
      v[r] = (y >= 0 && y < d.H && x >= 0 && x < d.W)
                 ? *reinterpret_cast<const uint4*>(base + ((long long)y * d.W + x) * d.in_cstride)
                 : vinf;
    }
    const uint4 mid = vmax(v[1], v[2]);
    const uint4 top = vmax(v[0], mid), bot = vmax(mid, v[3]);
    if (c <= 2) {
      o[0][0] = vmax(o[0][0], top);
      o[1][0] = vmax(o[1][0], bot);
    }
    if (c >= 1) {
      o[0][1] = vmax(o[0][1], top);
      o[1][1] = vmax(o[1][1], bot);
    }
  }
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int oy = 2 * by + dy, ox = 2 * bx + dx;
      if (oy < d.H && ox < d.W)
        *reinterpret_cast<uint4*>(out + (((long long)n * d.H + oy) * d.W + ox) * d.out_cstride + g * 8) = o[dy][dx];
    }
}

static bool misaligned(const void* p, uintptr_t bytes) { return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) != 0; }

static void plan_grid(MemLaunch* L, MemKernel k, dim3 grid, unsigned block, int variant = -1, size_t smem = 0) {
  L->kernel = k;
  L->variant = variant;
  L->grid = grid;
  L->block = block;
  L->smem = smem;
  L->max_rows = 0;
}

int plan_pool(ug_engine* h, const ug_pool_desc* d, MemLaunch* L) {
  if (!d->in || !d->out || d->C % 8 || d->in_cstride % 8 || d->out_cstride % 8 || d->k <= 0 || d->stride <= 0)
    return set_error(h, UG_EINVAL, "pool: bad args (C and strides must be multiples of 8)");
  if (misaligned(d->in, 16) || misaligned(d->out, 16))
    return set_error(h, UG_EINVAL, "pool: in / out must be 16-byte aligned");
  if ((d->OH - 1) * d->stride - d->pad >= d->H || (d->OW - 1) * d->stride - d->pad >= d->W)
    return set_error(h, UG_EINVAL, "pool: last window starts outside the input");
  // Block forms for 3x3 windows (profiles/r02_pool_s2.txt, against the generic kernel for stride 2 and sliding rows for
  // stride 1): maxpool1 0.1505 -> 0.107 ms per 256 images (4.8 TB/s of DRAM traffic), maxpool2 0.118 ->
  // 0.086, the branch-4 pools on 28x28 / 14x14 maps 0.074 / 0.042 -> 0.058 / 0.033; the 7x7 maps stay on sliding rows
  // (0.015 against 0.0195 ms).
  const long long cg = d->C / 8;
  if (d->k == 3 && d->stride == 1 && d->pad == 1 && d->OH == d->H && d->OW == d->W && d->H * d->W >= 196)
    plan_grid(L, MemKernel::Pool3x3s1Block, ceil_div((long long)d->B * ((d->H + 1) / 2) * ((d->W + 1) / 2) * cg, 256), 256);
  else if (d->k == 3 && d->stride == 1 && d->pad == 1 && d->OH == d->H && d->OW == d->W)
    plan_grid(L, MemKernel::Pool3x3s1, ceil_div((long long)d->B * d->H * cg, 256), 256);
  else if (d->k == 3 && d->stride == 2 && d->pad == 0 && 2 * (d->OH - 1) < d->H && 2 * (d->OW - 1) < d->W)
    plan_grid(L, MemKernel::Pool3x3s2, ceil_div((long long)d->B * ((d->OH + 1) / 2) * ((d->OW + 1) / 2) * cg, 256), 256);
  else
    plan_grid(L, MemKernel::Pool, ceil_div((long long)d->B * d->OH * d->OW * cg, 256), 256);
  return UG_OK;
}

int launch_pool(ug_engine* h, const ug_pool_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_pool(h, d, &L);
  if (rc != UG_OK) return rc;
  const __nv_bfloat16* in = reinterpret_cast<const __nv_bfloat16*>(d->in);
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(d->out);
  switch (L.kernel) {
    case MemKernel::Pool3x3s1Block: launch_pdl(pool3x3s1_block_kernel, L.grid, L.block, 0, s, in, out, *d); break;
    case MemKernel::Pool3x3s1: launch_pdl(pool3x3s1_kernel, L.grid, L.block, 0, s, in, out, *d); break;
    case MemKernel::Pool3x3s2: launch_pdl(pool3x3s2_kernel, L.grid, L.block, 0, s, in, out, *d); break;
    default: launch_pdl(pool_kernel, L.grid, L.block, 0, s, in, out, *d); break;
  }
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "pool launch");
}

// ------------------------------------------------------------------------------------------------
// LayerNorm: one warp per kLnTok consecutive tokens, C = 256 * kNV in {256, 512, 768, 1024}.  All rows of the warp are
// fetched before any arithmetic (the 196-token x 512 maps are tiny: with one token per warp and two loads per lane the
// kernel ran at 12 % of the HBM peak, bound by load latency), gamma / beta are read once per warp; two-pass statistics
// in fp32 registers (kNV is a template parameter so that the rows stay in registers).
static constexpr int kLnTok = 4;

template <int kNV>
__global__ void __launch_bounds__(256) layernorm_kernel(const __nv_bfloat16* __restrict__ in,
                                                        __nv_bfloat16* __restrict__ out,
                                                        const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, int M, int C, float eps) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int t0 = warp * kLnTok;
  if (t0 >= M) return;
  uint4 raw[kLnTok][kNV];
#pragma unroll
  for (int t = 0; t < kLnTok; ++t) {
    const __nv_bfloat16* row = in + (long long)min(t0 + t, M - 1) * C;
#pragma unroll
    for (int i = 0; i < kNV; ++i) raw[t][i] = __ldg(reinterpret_cast<const uint4*>(row + (i * 32 + lane) * 8));
  }
  float4 ga[kNV][2], be[kNV][2];
#pragma unroll
  for (int i = 0; i < kNV; ++i) {
    const int c0 = (i * 32 + lane) * 8;
    ga[i][0] = __ldg(reinterpret_cast<const float4*>(gamma + c0));
    ga[i][1] = __ldg(reinterpret_cast<const float4*>(gamma + c0 + 4));
    be[i][0] = __ldg(reinterpret_cast<const float4*>(beta + c0));
    be[i][1] = __ldg(reinterpret_cast<const float4*>(beta + c0 + 4));
  }
#pragma unroll
  for (int t = 0; t < kLnTok; ++t) {
    float v[kNV * 8];
    float sum = 0.0f;
#pragma unroll
    for (int i = 0; i < kNV; ++i) {
      const uint32_t w[4] = {raw[t][i].x, raw[t][i].y, raw[t][i].z, raw[t][i].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[i * 8 + 2 * j] = bf16_lo(w[j]);
        v[i * 8 + 2 * j + 1] = bf16_hi(w[j]);
        sum += v[i * 8 + 2 * j] + v[i * 8 + 2 * j + 1];
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum / C;
    float sq = 0.0f;
#pragma unroll
    for (int i = 0; i < kNV * 8; ++i) {
      const float dlt = v[i] - mean;
      sq += dlt * dlt;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = rsqrtf(sq / C + eps);
    if (t0 + t < M) {
      __nv_bfloat16* orow = out + (long long)(t0 + t) * C;
#pragma unroll
      for (int i = 0; i < kNV; ++i) {
        const float g8[8] = {ga[i][0].x, ga[i][0].y, ga[i][0].z, ga[i][0].w, ga[i][1].x, ga[i][1].y, ga[i][1].z, ga[i][1].w};
        const float b8[8] = {be[i][0].x, be[i][0].y, be[i][0].z, be[i][0].w, be[i][1].x, be[i][1].y, be[i][1].z, be[i][1].w};
        float r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = (v[i * 8 + j] - mean) * rstd * g8[j] + b8[j];
        uint4 o;
        o.x = pack_bf16x2(r[0], r[1]);
        o.y = pack_bf16x2(r[2], r[3]);
        o.z = pack_bf16x2(r[4], r[5]);
        o.w = pack_bf16x2(r[6], r[7]);
        *reinterpret_cast<uint4*>(orow + (i * 32 + lane) * 8) = o;
      }
    }
  }
}

int plan_layernorm(ug_engine* h, const ug_layernorm_desc* d, MemLaunch* L) {
  if (!d->in || !d->out || !d->gamma || !d->beta || d->M <= 0 || d->C % 256 || d->C > 1024 || d->C <= 0)
    return set_error(h, UG_EINVAL, "layernorm: C must be a multiple of 256 up to 1024");
  if (misaligned(d->gamma, 16) || misaligned(d->beta, 16) || misaligned(d->in, 16) || misaligned(d->out, 16))
    return set_error(h, UG_EINVAL, "layernorm: in / out / gamma / beta must be 16-byte aligned");
  const long long warps = ((long long)d->M + kLnTok - 1) / kLnTok;
  plan_grid(L, MemKernel::LayerNorm, ceil_div(warps * 32, 256), 256, d->C / 256);
  return UG_OK;
}

int launch_layernorm(ug_engine* h, const ug_layernorm_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_layernorm(h, d, &L);
  if (rc != UG_OK) return rc;
  const __nv_bfloat16* in = reinterpret_cast<const __nv_bfloat16*>(d->in);
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(d->out);
  switch (L.variant) {
    case 1: launch_pdl(layernorm_kernel<1>, L.grid, L.block, 0, s, in, out, d->gamma, d->beta, d->M, d->C, d->eps); break;
    case 2: launch_pdl(layernorm_kernel<2>, L.grid, L.block, 0, s, in, out, d->gamma, d->beta, d->M, d->C, d->eps); break;
    case 3: launch_pdl(layernorm_kernel<3>, L.grid, L.block, 0, s, in, out, d->gamma, d->beta, d->M, d->C, d->eps); break;
    default: launch_pdl(layernorm_kernel<4>, L.grid, L.block, 0, s, in, out, d->gamma, d->beta, d->M, d->C, d->eps); break;
  }
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "layernorm launch");
}

// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// Tensor-core attention for S <= 208 tokens (the 14x14 bottleneck: S = 196), dim_head = 64.
// One CTA (4 warps) per (image, head).  K (row-major, padded pitch) and V^T are staged in shared memory; each warp
// owns 16-query slabs: S = Q K^T with mma.sync m16n8k16 (bf16 in, fp32 accumulate; the matrices are far too
// small for tcgen05 tiles), fp32 softmax on the accumulator fragments, P re-used in registers as the A operand
// of O = P V (accumulator layout of the first MMA == A-fragment layout of the second).
static constexpr int kAttnSP = 208;           // padded sequence length (multiple of 16)
static constexpr int kAttnKPitch = 72;        // bf16 elements per sK row  (144 B: conflict-free fragment loads)
static constexpr int kAttnVPitch = 72;        // bf16 elements per sV row (row-major [key][dim]; fragments via ldmatrix.trans)

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(128, 3) attention_mma_kernel(ug_attn_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  extern __shared__ uint4 attn_smem[];
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(attn_smem);   // [kAttnSP][kAttnKPitch]
  __nv_bfloat16* sV = sK + kAttnSP * kAttnKPitch;                     // [kAttnSP][kAttnVPitch]
  const int b = blockIdx.x / d.heads;
  const int hd = blockIdx.x % d.heads;
  const __nv_bfloat16* q = reinterpret_cast<const __nv_bfloat16*>(d.q);
  const __nv_bfloat16* k = reinterpret_cast<const __nv_bfloat16*>(d.k);
  const __nv_bfloat16* v = reinterpret_cast<const __nv_bfloat16*>(d.v);
  // K and V of this (image, head) -> smem with cp.async (all 26 16-byte copies of a thread in flight at once; the
  // load -> store loop this replaces exposed one global-load latency per iteration, a third of the kernel time).
  // Rows beyond S are zero-filled (src-size 0).
  for (int i = threadIdx.x; i < kAttnSP * 8; i += blockDim.x) {
    const int row = i >> 3, part = i & 7;
    const long long tok = (long long)b * d.S + (row < d.S ? row : 0);
    const unsigned nbytes = row < d.S ? 16u : 0u;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(sK + row * kAttnKPitch + part * 8)),
                 "l"(k + tok * d.k_stride + hd * 64 + part * 8), "r"(nbytes)
                 : "memory");
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(sV + row * kAttnVPitch + part * 8)),
                 "l"(v + tok * d.v_stride + hd * 64 + part * 8), "r"(nbytes)
                 : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const float sl2 = d.scale * 1.4426950408889634f;
  const int nslabs = (d.S + 15) / 16;
  for (int slab = warp; slab < nslabs; slab += 4) {
    const int r0 = slab * 16 + g, r1 = r0 + 8;
    const long long tok0 = (long long)b * d.S + r0, tok1 = (long long)b * d.S + r1;
    uint32_t qa[4][4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const int c = hd * 64 + kk * 16 + 2 * t;
      qa[kk][0] = r0 < d.S ? __ldg(reinterpret_cast<const uint32_t*>(q + tok0 * d.q_stride + c)) : 0u;
      qa[kk][1] = r1 < d.S ? __ldg(reinterpret_cast<const uint32_t*>(q + tok1 * d.q_stride + c)) : 0u;
      qa[kk][2] = r0 < d.S ? __ldg(reinterpret_cast<const uint32_t*>(q + tok0 * d.q_stride + c + 8)) : 0u;
      qa[kk][3] = r1 < d.S ? __ldg(reinterpret_cast<const uint32_t*>(q + tok1 * d.q_stride + c + 8)) : 0u;
    }
    float sc[kAttnSP / 8][4];
#pragma unroll
    for (int nt = 0; nt < kAttnSP / 8; ++nt) {
      sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.0f;
      const __nv_bfloat16* krow = sK + (nt * 8 + g) * kAttnKPitch + 2 * t;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(krow + kk * 16);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(krow + kk * 16 + 8);
        mma_bf16_16816(sc[nt], qa[kk], b0, b1);
      }
    }
    // fp32 softmax over the key axis (columns nt*8 + 2t, +1); rows g (c0,c1) and g+8 (c2,c3)
    float m0 = -FLT_MAX, m1 = -FLT_MAX;
#pragma unroll
    for (int nt = 0; nt < kAttnSP / 8; ++nt) {
      const int col = nt * 8 + 2 * t;
      if (col >= d.S) sc[nt][0] = sc[nt][2] = -FLT_MAX;
      if (col + 1 >= d.S) sc[nt][1] = sc[nt][3] = -FLT_MAX;
      m0 = fmaxf(m0, fmaxf(sc[nt][0], sc[nt][1]));
      m1 = fmaxf(m1, fmaxf(sc[nt][2], sc[nt][3]));
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float l0 = 0.0f, l1 = 0.0f;
#pragma unroll
    for (int nt = 0; nt < kAttnSP / 8; ++nt) {
      sc[nt][0] = exp2f((sc[nt][0] - m0) * sl2);
      sc[nt][1] = exp2f((sc[nt][1] - m0) * sl2);
      sc[nt][2] = exp2f((sc[nt][2] - m1) * sl2);
      sc[nt][3] = exp2f((sc[nt][3] - m1) * sl2);
      l0 += sc[nt][0] + sc[nt][1];
      l1 += sc[nt][2] + sc[nt][3];
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    float o[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.0f;
#pragma unroll
    for (int kk = 0; kk < kAttnSP / 16; ++kk) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(sc[2 * kk][0], sc[2 * kk][1]);
      pa[1] = pack_bf16x2(sc[2 * kk][2], sc[2 * kk][3]);
      pa[2] = pack_bf16x2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
      pa[3] = pack_bf16x2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
      // B fragments of V[16 keys][8 dims] blocks: V is row-major in smem (key-major), the mma wants it key-contiguous
      // per dim, i.e. transposed: ldmatrix.trans (lanes 0-15 address the 16 key rows, lanes 16-31 those of the next
      // 8-dim block).  The element-wise transposed staging this replaces cost 12.5k conflicted 2-byte stores per block.
#pragma unroll
      for (int nt = 0; nt < 8; nt += 2) {
        const __nv_bfloat16* vp = sV + (kk * 16 + (lane & 15)) * kAttnVPitch + (nt + (lane >> 4)) * 8;
        uint32_t b0, b1, b2, b3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3)
                     : "r"(smem_u32(vp)));
        mma_bf16_16816(o[nt], pa, b0, b1);
        mma_bf16_16816(o[nt + 1], pa, b2, b3);
      }
    }
    const float i0 = 1.0f / l0, i1 = 1.0f / l1;
    __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(d.out);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int c = hd * 64 + nt * 8 + 2 * t;
      if (r0 < d.S) *reinterpret_cast<uint32_t*>(out + tok0 * d.out_stride + c) = pack_bf16x2(o[nt][0] * i0, o[nt][1] * i0);
      if (r1 < d.S) *reinterpret_cast<uint32_t*>(out + tok1 * d.out_stride + c) = pack_bf16x2(o[nt][2] * i1, o[nt][3] * i1);
    }
  }
}

int plan_attention(ug_engine* h, const ug_attn_desc* d, MemLaunch* L) {
  if (!d->q || !d->k || !d->v || !d->out || d->S <= 0 || d->heads <= 0 || d->B <= 0 || d->variant != 0)
    return set_error(h, UG_EINVAL, "attention: bad args");
  if (d->S > kAttnSP) return set_error(h, UG_EUNSUPPORTED, "attention: S <= %d tokens (the 14x14 bottleneck has 196)", kAttnSP);
  if (d->q_stride % 8 || d->k_stride % 8 || d->v_stride % 8 || d->out_stride % 8)
    return set_error(h, UG_EINVAL, "attention: row strides must be multiples of 8");
  const long long cols = 64LL * d->heads;
  if (cols > d->q_stride || cols > d->k_stride || cols > d->v_stride || cols > d->out_stride)
    return set_error(h, UG_EINVAL, "attention: 64 * heads = %lld columns must fit in every row stride", cols);
  // K and V rows are staged with 16-byte cp.async, q is read and out written as bf16 pairs
  if (misaligned(d->k, 16) || misaligned(d->v, 16) || misaligned(d->q, 4) || misaligned(d->out, 4))
    return set_error(h, UG_EINVAL, "attention: k / v must be 16-byte aligned, q / out 4-byte aligned");
  plan_grid(L, MemKernel::Attention, d->B * d->heads, 128, -1,
            (size_t)(kAttnSP * kAttnKPitch + kAttnSP * kAttnVPitch) * sizeof(__nv_bfloat16));
  return UG_OK;
}

int launch_attention(ug_engine* h, const ug_attn_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_attention(h, d, &L);
  if (rc != UG_OK) return rc;
  if (!h->attr_attn) {
    const cudaError_t e = cudaFuncSetAttribute(attention_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(attention_mma_kernel)");
    h->attr_attn = true;
  }
  launch_pdl(attention_mma_kernel, L.grid, L.block, L.smem, s, *d);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "attention launch");
}

// ------------------------------------------------------------------------------------------------
// CoordAtt3 statistics, stage 1: block (split, image) reduces its pixel range; threads are laid out as
// (C/8 channel groups) x (256/(C/8) pixel lanes), partial results combined through shared memory.
__global__ void __launch_bounds__(256) chanstats_kernel(ug_chanstats_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  __shared__ float s_sum[256 * 8];
  __shared__ float s_max[256 * 8];
  const int cg = d.C / 8;       // channel groups (<= 64)
  const int lanes = 256 / cg;   // pixel lanes per group
  const int g = threadIdx.x % cg;
  const int pl = threadIdx.x / cg;
  const int split = blockIdx.x, n = blockIdx.y;
  const int per = (d.HW + d.splits - 1) / d.splits;
  const int p0 = split * per;
  const int p1 = min(d.HW, p0 + per);
  const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(d.in) + (long long)n * d.HW * d.in_cstride + g * 8;
  float sum[8], mx[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sum[j] = 0.0f;
    mx[j] = -FLT_MAX;
  }
  for (int p = p0 + pl; p < p1; p += lanes) {
    const uint4 u = *reinterpret_cast<const uint4*>(base + (long long)p * d.in_cstride);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a = bf16_lo(w[j]), b = bf16_hi(w[j]);
      sum[2 * j] += a;
      sum[2 * j + 1] += b;
      mx[2 * j] = fmaxf(mx[2 * j], a);
      mx[2 * j + 1] = fmaxf(mx[2 * j + 1], b);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    s_sum[threadIdx.x * 8 + j] = sum[j];
    s_max[threadIdx.x * 8 + j] = mx[j];
  }
  __syncthreads();
  // thread c (< C) folds the pixel lanes of channel c in a fixed order
  for (int c = threadIdx.x; c < d.C; c += 256) {
    const int gg = c / 8, j = c % 8;
    float a = 0.0f, b = -FLT_MAX;
    for (int l = 0; l < lanes; ++l) {
      a += s_sum[(l * cg + gg) * 8 + j];
      b = fmaxf(b, s_max[(l * cg + gg) * 8 + j]);
    }
    const long long o = ((long long)n * d.splits + split) * d.C + c;
    d.psum[o] = a;
    d.pmax[o] = b;
  }
}

int plan_chanstats(ug_engine* h, const ug_chanstats_desc* d, MemLaunch* L) {
  if (!d->in || !d->psum || !d->pmax || d->C % 8 || d->C > 512 || d->C < 8 || (256 % (d->C / 8)) || d->splits <= 0 ||
      d->in_cstride % 8)
    return set_error(h, UG_EINVAL, "chanstats: C must be 8*2^k <= 512");
  if (misaligned(d->in, 16)) return set_error(h, UG_EINVAL, "chanstats: in must be 16-byte aligned");
  plan_grid(L, MemKernel::ChanStats, dim3(d->splits, d->B), 256);
  return UG_OK;
}

int launch_chanstats(ug_engine* h, const ug_chanstats_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_chanstats(h, d, &L);
  if (rc != UG_OK) return rc;
  launch_pdl(chanstats_kernel, L.grid, L.block, 0, s, *d);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "chanstats launch");
}

// stage 2 + gate MLP.  Two launches so that each image is spread over kGateSplit blocks:
//   gate_hidden_kernel: fold the partial sums/maxima, hid = relu(W1 avg + b1) + relu(W2 max + b2)   (slice of hid)
//   gate_out_kernel:    g = sigmoid(W3 hid + b3)                                                     (slice of g)
static constexpr int kGateSplit = 8;

__global__ void __launch_bounds__(256) gate_hidden_kernel(ug_gate_desc d, float* __restrict__ hid_out) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  __shared__ float s_avg[512], s_max[512];
  const int n = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int c = threadIdx.x; c < d.C; c += blockDim.x) {
    float a = 0.0f, b = -FLT_MAX;
    for (int sp = 0; sp < d.splits; ++sp) {
      const long long o = ((long long)n * d.splits + sp) * d.C + c;
      a += d.psum[o];
      b = fmaxf(b, d.pmax[o]);
    }
    s_avg[c] = a / (float)d.HW;
    s_max[c] = b;
  }
  __syncthreads();
  const int hid = d.C / 2;
  const int per = (hid + kGateSplit - 1) / kGateSplit;
  const int j0 = blockIdx.x * per, j1 = min(hid, j0 + per);
  for (int j = j0 + warp; j < j1; j += 8) {
    float a = 0.0f, b = 0.0f;
    for (int c = lane; c < d.C; c += 32) {
      a += __ldg(d.w1 + (long long)j * d.C + c) * s_avg[c];
      b += __ldg(d.w2 + (long long)j * d.C + c) * s_max[c];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane == 0) hid_out[(long long)n * hid + j] = fmaxf(a + d.b1[j], 0.0f) + fmaxf(b + d.b2[j], 0.0f);
  }
}

__global__ void __launch_bounds__(256) gate_out_kernel(ug_gate_desc d, const float* __restrict__ hid_in) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  __shared__ float s_hid[256];
  const int n = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int hid = d.C / 2;
  for (int j = threadIdx.x; j < hid; j += blockDim.x) s_hid[j] = hid_in[(long long)n * hid + j];
  __syncthreads();
  const int per = (d.C + kGateSplit - 1) / kGateSplit;
  const int c0 = blockIdx.x * per, c1 = min(d.C, c0 + per);
  for (int c = c0 + warp; c < c1; c += 8) {
    float a = 0.0f;
    for (int j = lane; j < hid; j += 32) a += __ldg(d.w3 + (long long)c * hid + j) * s_hid[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) d.g[(long long)n * d.C + c] = 1.0f / (1.0f + expf(-(a + d.b3[c])));
  }
}

int plan_gate(ug_engine* h, const ug_gate_desc* d, MemLaunch* L) {
  if (!d->psum || !d->pmax || !d->w1 || !d->w2 || !d->w3 || !d->b1 || !d->b2 || !d->b3 || !d->g || !d->hid ||
      d->C > 512 || d->C % 2 || d->HW <= 0 || d->splits <= 0)
    return set_error(h, UG_EINVAL, "gate: bad args (C <= 512, hid scratch required)");
  plan_grid(L, MemKernel::Gate, dim3(kGateSplit, d->B), 256);
  return UG_OK;
}

int launch_gate(ug_engine* h, const ug_gate_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_gate(h, d, &L);
  if (rc != UG_OK) return rc;
  launch_pdl(gate_hidden_kernel, L.grid, L.block, 0, s, *d, d->hid);
  launch_pdl(gate_out_kernel, L.grid, L.block, 0, s, *d, d->hid);
  h->launches += 2;
  return check_cuda(h, cudaGetLastError(), "gate launch");
}

// ------------------------------------------------------------------------------------------------
// mask -> bbox: one block per image; warp-shuffle min/max, then one thread applies roi.py:25-36.
__global__ void __launch_bounds__(1024) bbox_kernel(const unsigned char* __restrict__ mask, int* __restrict__ boxes, int H,
                                                    int W, int padding) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  __shared__ int s_red[4][32];
  const int n = blockIdx.x;
  const unsigned char* m = mask + (long long)n * H * W;
  int xmin = INT_MAX, ymin = INT_MAX, xmax = -1, ymax = -1;
  const int total = H * W;
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    if (m[i] == 1) {
      const int y = i / W, x = i - y * W;
      xmin = min(xmin, x);
      xmax = max(xmax, x);
      ymin = min(ymin, y);
      ymax = max(ymax, y);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    xmin = min(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
    ymin = min(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
    xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
    ymax = max(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    s_red[0][warp] = xmin;
    s_red[1][warp] = ymin;
    s_red[2][warp] = xmax;
    s_red[3][warp] = ymax;
  }
  __syncthreads();
  if (warp == 0) {
    const int nw = blockDim.x >> 5;
    xmin = lane < nw ? s_red[0][lane] : INT_MAX;
    ymin = lane < nw ? s_red[1][lane] : INT_MAX;
    xmax = lane < nw ? s_red[2][lane] : -1;
    ymax = lane < nw ? s_red[3][lane] : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      xmin = min(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
      ymin = min(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
      xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
      ymax = max(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
    }
    if (lane == 0) {
      int x0, y0, x1, y1;
      if (xmax < 0) {  // empty mask: centred square of side min(h,w)//2 (roi.py:26-31)
        const int cx = W / 2, cy = H / 2, size = min(H, W) / 2;
        x0 = cx - size / 2;
        x1 = cx + size / 2;
        y0 = cy - size / 2;
        y1 = cy + size / 2;
      } else {  // roi.py:33-36 (max is an exclusive slice end)
        x0 = max(xmin - padding, 0);
        x1 = min(xmax + padding, W);
        y0 = max(ymin - padding, 0);
        y1 = min(ymax + padding, H);
      }
      boxes[n * 4 + 0] = x0;
      boxes[n * 4 + 1] = y0;
      boxes[n * 4 + 2] = x1;
      boxes[n * 4 + 3] = y1;
    }
  }
}

int plan_bbox(ug_engine* h, const ug_bbox_desc* d, MemLaunch* L) {
  if (!d->mask || !d->boxes || d->B <= 0 || d->H <= 0 || d->W <= 0) return set_error(h, UG_EINVAL, "bbox: bad args");
  plan_grid(L, MemKernel::BBox, d->B, 1024);
  return UG_OK;
}

int launch_bbox(ug_engine* h, const ug_bbox_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_bbox(h, d, &L);
  if (rc != UG_OK) return rc;
  launch_pdl(bbox_kernel, L.grid, L.block, 0, s, d->mask, d->boxes, d->H, d->W, d->padding);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "bbox launch");
}

// ------------------------------------------------------------------------------------------------
// PIL-exact crop + bilinear resize (Pillow ImagingResample, 8 bits per channel):
//   coefficient tables per axis are computed in fp64 exactly as precompute_coeffs() does, then quantised to
//   22-bit fixed point; horizontal pass first (uint8 result), vertical pass second.
static constexpr int kPrecBits = 22;  // 32 - 8 - 2

__device__ __forceinline__ int clip8(int v) {
  v >>= kPrecBits;
  return v < 0 ? 0 : (v > 255 ? 255 : v);
}

// ------------------------------------------------------------------------------------------------
// Device front-end: PIL-exact bilinear resize of uint8 HWC source images of ANY size to SxS (the reference's
// CDDataAugmentation.transform: F.resize(..., BILINEAR) on a PIL image + to_tensor; Pillow's antialiased
// resample: support = max(in/out, 1), up to 2*ceil(support)+1 taps per axis), written as fp32 NCHW / 255.
// One block per (group of R output rows, image): the horizontal pass of the source rows those output rows need is
// kept in shared memory as uint8 (exactly Pillow's intermediate image), the vertical pass reads it from there.
static constexpr int kRsMaxTaps = 17;   // support <= 8: source side up to 8 * S
static constexpr int kRsMaxSide = 8;    // (kRsMaxTaps - 1) / 2
static constexpr int kRsRows = 8;       // output rows per block

struct RsCoef {
  int xmin, n;
  int kk[kRsMaxTaps];
};

__device__ void pil_coef_general(int in_size, int out_size, int xx, RsCoef* c) {
  const double scale = __ddiv_rn((double)in_size, (double)out_size);
  const double filterscale = scale < 1.0 ? 1.0 : scale;
  const double support = filterscale;  // bilinear: support 1.0 * filterscale
  const double ss = __ddiv_rn(1.0, filterscale);
  const double center = __dmul_rn(__dadd_rn((double)xx, 0.5), scale);
  int xmin = (int)__dadd_rn(__dadd_rn(center, -support), 0.5);
  if (xmin < 0) xmin = 0;
  int xmax = (int)__dadd_rn(__dadd_rn(center, support), 0.5);
  if (xmax > in_size) xmax = in_size;
  int n = xmax - xmin;
  if (n > kRsMaxTaps) n = kRsMaxTaps;
  double k[kRsMaxTaps];
  double ww = 0.0;
  for (int x = 0; x < n; ++x) {
    double a = __dmul_rn(__dadd_rn(__dadd_rn((double)(x + xmin), -center), 0.5), ss);
    if (a < 0.0) a = -a;
    const double w = a < 1.0 ? __dadd_rn(1.0, -a) : 0.0;
    k[x] = w;
    ww = __dadd_rn(ww, w);
  }
  c->xmin = xmin;
  c->n = n;
  for (int x = 0; x < n; ++x) {
    double kv = k[x];
    if (ww != 0.0) kv = __ddiv_rn(kv, ww);
    const double scaled = __dmul_rn(kv, (double)(1 << kPrecBits));
    c->kk[x] = kv < 0.0 ? (int)__dadd_rn(-0.5, scaled) : (int)__dadd_rn(0.5, scaled);
  }
}

// Source modes.  kUniform: uint8 HWC images of one size (ug_resize_desc).  kCrop: the box (x0,y0,x1,y1) of an fp32
// NCHW image in [0,1], quantised as (x*255).astype(uint8) with the channel order reversed (roi.py:39-44), i.e. the
// ROI stage (ug_cropresize_desc); d.src is unused, `img` / `boxes` / `IH` / `IW` describe the float image.  kRagged:
// uint8 HWC images of different sizes (ug_resize_ragged_desc); image n's size and offset come from rg.index[n].
enum { kUniform = 0, kCrop = 1, kRagged = 2 };
struct RaggedSrc {
  const ug_ragged_image* index;
  int* status;
  long long src_bytes;
};

template <int kMode>
__global__ void __launch_bounds__(256) resize_u8_kernel(ug_resize_desc d, int max_src_rows, const float* __restrict__ img,
                                                        const int* __restrict__ boxes, int IH, int IW, RaggedSrc rg) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  extern __shared__ unsigned char rs_smem[];
  RsCoef* s_h = reinterpret_cast<RsCoef*>(rs_smem);                   // [S] horizontal coefficients
  RsCoef* s_v = s_h + d.S;                                             // [kRsRows] vertical coefficients
  unsigned char* s_tmp = reinterpret_cast<unsigned char*>(s_v + kRsRows);  // [max_src_rows][S*3] after the h-pass
  const int n = blockIdx.y;
  const int oy0 = blockIdx.x * kRsRows;
  const int rows = min(kRsRows, d.S - oy0);
  int bx0 = 0, by0 = 0;
  long long src_off = (long long)n * d.Hs * d.Ws * 3;
  if (kMode == kCrop) {
    bx0 = boxes[n * 4 + 0];
    by0 = boxes[n * 4 + 1];
    d.Ws = boxes[n * 4 + 2] - bx0;
    d.Hs = boxes[n * 4 + 3] - by0;
  }
  if (kMode == kRagged) {
    // the table comes from outside the library: check the entry before reading a byte of the image
    const ug_ragged_image e = rg.index[n];
    const int smax = kRsMaxSide * d.S;
    const bool ok = e.px_offset >= 0 && e.H >= 1 && e.W >= 1 && e.H <= smax && e.W <= smax &&
                    e.px_offset <= rg.src_bytes / 3 && (long long)e.H * e.W * 3 <= rg.src_bytes - 3 * e.px_offset;
    if (rg.status && blockIdx.x == 0 && threadIdx.x == 0) rg.status[n] = ok ? 0 : 1;
    if (!ok) {  // this block's output rows of a rejected image are zeros
      for (int t = threadIdx.x; t < rows * d.S; t += blockDim.x) {
        const int oy = oy0 + t / d.S, ox = t % d.S;
        if (d.out_u8) {
          unsigned char* o = d.out_u8 + (((long long)n * d.S + oy) * d.S + ox) * 3;
          o[0] = o[1] = o[2] = 0;
        }
        if (d.out_f32)
          for (int c = 0; c < 3; ++c) d.out_f32[(((long long)n * 3 + c) * d.S + oy) * d.S + ox] = 0.0f;
      }
      return;
    }
    d.Hs = e.H;
    d.Ws = e.W;
    src_off = 3 * e.px_offset;
  }
  for (int i = threadIdx.x; i < d.S; i += blockDim.x) pil_coef_general(d.Ws, d.S, i, &s_h[i]);
  if (threadIdx.x < rows) pil_coef_general(d.Hs, d.S, oy0 + threadIdx.x, &s_v[threadIdx.x]);
  __syncthreads();
  const int sy0 = s_v[0].xmin;                                          // first / one-past-last source row needed
  const int sy1 = s_v[rows - 1].xmin + s_v[rows - 1].n;
  const unsigned char* src = kMode == kCrop ? nullptr : d.src + src_off;
  const float* fimg = kMode == kCrop ? img + (long long)n * 3 * IH * IW : nullptr;
  const int row_elems = d.S * 3;
  for (int t = threadIdx.x; t < (sy1 - sy0) * d.S; t += blockDim.x) {   // horizontal pass (one output pixel, 3 ch)
    const int r = t / d.S, ox = t - r * d.S;
    const RsCoef& hc = s_h[ox];
    int a0 = 1 << (kPrecBits - 1), a1 = a0, a2 = a0;
    if (kMode == kCrop) {
      // (roi*255).astype(uint8): fp32 multiply, truncate; output channel c reads plane 2-c (cv2.COLOR_BGR2RGB)
      const float* p0 = fimg + ((long long)(by0 + sy0 + r)) * IW + bx0 + hc.xmin;
      const long long plane = (long long)IH * IW;
      for (int i = 0; i < hc.n; ++i) {
        const int k = hc.kk[i];
        a0 += (((int)__fmul_rn(__ldg(p0 + 2 * plane + i), 255.0f)) & 255) * k;
        a1 += (((int)__fmul_rn(__ldg(p0 + plane + i), 255.0f)) & 255) * k;
        a2 += (((int)__fmul_rn(__ldg(p0 + i), 255.0f)) & 255) * k;
      }
    } else {
      const unsigned char* sp = src + ((long long)(sy0 + r) * d.Ws + hc.xmin) * 3;
      for (int i = 0; i < hc.n; ++i) {
        const int k = hc.kk[i];
        a0 += (int)__ldg(sp + 3 * i) * k;
        a1 += (int)__ldg(sp + 3 * i + 1) * k;
        a2 += (int)__ldg(sp + 3 * i + 2) * k;
      }
    }
    unsigned char* tp = s_tmp + r * row_elems + ox * 3;
    tp[0] = (unsigned char)clip8(a0);
    tp[1] = (unsigned char)clip8(a1);
    tp[2] = (unsigned char)clip8(a2);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < rows * d.S; t += blockDim.x) {          // vertical pass + to_tensor
    const int ry = t / d.S, ox = t - ry * d.S;
    const RsCoef& vc = s_v[ry];
    const unsigned char* tp = s_tmp + (vc.xmin - sy0) * row_elems + ox * 3;
    int a0 = 1 << (kPrecBits - 1), a1 = a0, a2 = a0;
    for (int j = 0; j < vc.n; ++j) {
      const int k = vc.kk[j];
      a0 += (int)tp[j * row_elems] * k;
      a1 += (int)tp[j * row_elems + 1] * k;
      a2 += (int)tp[j * row_elems + 2] * k;
    }
    const int v[3] = {clip8(a0), clip8(a1), clip8(a2)};
    const int oy = oy0 + ry;
    if (d.out_u8) {
      unsigned char* o = d.out_u8 + (((long long)n * d.S + oy) * d.S + ox) * 3;
      o[0] = (unsigned char)v[0];
      o[1] = (unsigned char)v[1];
      o[2] = (unsigned char)v[2];
    }
    if (d.out_f32) {
#pragma unroll
      for (int c = 0; c < 3; ++c)  // F.to_tensor: uint8 -> float32, divided by 255
        d.out_f32[(((long long)n * 3 + c) * d.S + oy) * d.S + ox] = (float)v[c] / 255.0f;
    }
  }
}

int launch_resize_u8(ug_engine* h, const ug_resize_desc* d, cudaStream_t s) {
  if (!d->src || (!d->out_f32 && !d->out_u8) || d->B <= 0 || d->Hs <= 0 || d->Ws <= 0 || d->S <= 0 || d->S > 512)
    return set_error(h, UG_EINVAL, "resize: bad args (S <= 512)");
  const double sc = std::max((double)d->Hs / d->S, (double)d->Ws / d->S);
  if (2 * (int)ceil(std::max(sc, 1.0)) + 1 > kRsMaxTaps)
    return set_error(h, UG_EUNSUPPORTED, "resize: source more than 8x larger than the output");
  // source rows needed by kRsRows output rows: (kRsRows - 1) * scale + 2 * support + 2
  const double scy = std::max((double)d->Hs / d->S, 1.0);
  const int max_rows = std::min(d->Hs, (int)ceil((kRsRows - 1) * ((double)d->Hs / d->S) + 2.0 * scy + 3.0));
  const size_t smem = (size_t)(d->S + kRsRows) * sizeof(RsCoef) + (size_t)max_rows * d->S * 3;
  if (smem > h->attr_resize) {
    if (smem > 200 * 1024) return set_error(h, UG_EUNSUPPORTED, "resize: shared memory request %zu too large", smem);
    cudaError_t e = cudaFuncSetAttribute((const void*)resize_u8_kernel<kUniform>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(resize_u8_kernel)");
    h->attr_resize = smem;
  }
  launch_pdl(resize_u8_kernel<kUniform>, dim3(ceil_div(d->S, kRsRows), d->B), 256, smem, s, *d, max_rows, nullptr, nullptr,
             0, 0, RaggedSrc{});
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "resize_u8 launch");
}

// Ragged front-end: the uniform kernel with per-image sizes from the table.  Shared memory and grid are sized for the
// largest source the descriptor admits (sides up to kRsMaxSide * S), so the launch does not depend on the table.
int launch_resize_ragged(ug_engine* h, const ug_resize_ragged_desc* d, cudaStream_t s) {
  if (!d->src || !d->index || (!d->out_f32 && !d->out_u8) || d->B <= 0 || d->S <= 0 || d->S > 512 || d->src_bytes < 0)
    return set_error(h, UG_EINVAL, "resize_ragged: bad args (S <= 512)");
  const double sc = kRsMaxSide;
  const int max_rows = (int)ceil((kRsRows - 1) * sc + 2.0 * sc + 3.0);
  const size_t smem = (size_t)(d->S + kRsRows) * sizeof(RsCoef) + (size_t)max_rows * d->S * 3;
  if (smem > h->attr_ragged) {
    if (smem > 200 * 1024) return set_error(h, UG_EUNSUPPORTED, "resize_ragged: shared memory request %zu too large", smem);
    cudaError_t e = cudaFuncSetAttribute((const void*)resize_u8_kernel<kRagged>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(resize_u8_kernel<ragged>)");
    h->attr_ragged = smem;
  }
  ug_resize_desc r;
  r.src = d->src; r.out_f32 = d->out_f32; r.out_u8 = d->out_u8; r.B = d->B; r.Hs = 0; r.Ws = 0; r.S = d->S;
  launch_pdl(resize_u8_kernel<kRagged>, dim3(ceil_div(d->S, kRsRows), d->B), 256, smem, s, r, max_rows, nullptr, nullptr,
             0, 0, RaggedSrc{d->index, d->status, d->src_bytes});
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "resize_ragged launch");
}

// ROI stage (roi.py:39-44 + data_utils.py:102,146-147): the same two-pass kernel reading the box of the float image.
// Crops are at most HxW with S >= both sides in the pipeline (224 -> 224: up-sampling, <= 3 taps), but any ratio up
// to 8x is handled.
int plan_cropresize(ug_engine* h, const ug_cropresize_desc* d, MemLaunch* L) {
  if (!d->img || !d->boxes || !d->out_u8 || d->S <= 0 || d->S > 512 || d->B <= 0 || d->H <= 0 || d->W <= 0)
    return set_error(h, UG_EINVAL, "cropresize: bad args (S <= 512)");
  const double sc = std::max(std::max((double)d->H / d->S, (double)d->W / d->S), 1.0);
  if (2 * (int)ceil(sc) + 1 > kRsMaxTaps) return set_error(h, UG_EUNSUPPORTED, "cropresize: image more than 8x the output");
  const int max_rows = std::min(d->H, (int)ceil((kRsRows - 1) * sc + 2.0 * sc + 3.0));
  const size_t smem = (size_t)(d->S + kRsRows) * sizeof(RsCoef) + (size_t)max_rows * d->S * 3;
  if (smem > 200 * 1024) return set_error(h, UG_EUNSUPPORTED, "cropresize: shared memory request %zu too large", smem);
  plan_grid(L, MemKernel::CropResize, dim3(ceil_div(d->S, kRsRows), d->B), 256, kCrop, smem);
  L->max_rows = max_rows;
  return UG_OK;
}

int launch_cropresize(ug_engine* h, const ug_cropresize_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_cropresize(h, d, &L);
  if (rc != UG_OK) return rc;
  if (L.smem > h->attr_crop) {
    cudaError_t e = cudaFuncSetAttribute((const void*)resize_u8_kernel<kCrop>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem);
    if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(resize_u8_kernel<crop>)");
    h->attr_crop = L.smem;
  }
  ug_resize_desc r;
  r.src = nullptr; r.out_f32 = nullptr; r.out_u8 = d->out_u8; r.B = d->B; r.Hs = d->H; r.Ws = d->W; r.S = d->S;
  launch_pdl(resize_u8_kernel<kCrop>, L.grid, L.block, L.smem, s, r, L.max_rows, d->img, d->boxes, d->H, d->W,
             RaggedSrc{});
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "cropresize launch");
}

// ------------------------------------------------------------------------------------------------
// Space-to-depth pack for GoogLeNet conv1 (ug_s2d_desc): one thread per packed pixel (n, Y, X) writes its 16 bf16
// channels (32 contiguous bytes): the 2x2 block of source pixels (2Y+dy-3, 2X+dx-3) x 3 channels, to_tensor and
// _transform_input applied, zero outside the image and in channels 12..15.
__global__ void __launch_bounds__(256) s2d_pack_kernel(ug_s2d_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  const int Q = d.S / 2 + 3;
  const long long total = (long long)d.B * Q * Q;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int X = (int)(t % Q);
  const int Y = (int)((t / Q) % Q);
  const int n = (int)(t / ((long long)Q * Q));
  // torchvision GoogLeNet._transform_input: x_c * (std_c / 0.5) + (mean_c - 0.5) / 0.5, the constants evaluated in
  // double and rounded once, as torch applies those Python scalars to a float tensor (evaluated from the float-rounded
  // means, the shifts of channels 0 and 2 were 15 and 2 float ulps off)
  const float sc[3] = {(float)(0.229 / 0.5), (float)(0.224 / 0.5), (float)(0.225 / 0.5)};
  const float sh[3] = {(float)((0.485 - 0.5) / 0.5), (float)((0.456 - 0.5) / 0.5), (float)((0.406 - 0.5) / 0.5)};
  float v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = 0.0f;
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) {
    const int iy = 2 * Y + dy - 3;
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int ix = 2 * X + dx - 3;
      if (iy < 0 || iy >= d.S || ix < 0 || ix >= d.S) continue;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float x = d.in_f32 ? __ldg(d.in_f32 + (((long long)n * 3 + c) * d.S + iy) * d.S + ix)
                                 : (float)__ldg(d.in_u8 + (((long long)n * d.S + iy) * d.S + ix) * 3 + c) / 255.0f;
        v[(dy * 2 + dx) * 3 + c] = x * sc[c] + sh[c];
      }
    }
  }
  uint4 o0, o1;
  o0.x = pack_bf16x2(v[0], v[1]);
  o0.y = pack_bf16x2(v[2], v[3]);
  o0.z = pack_bf16x2(v[4], v[5]);
  o0.w = pack_bf16x2(v[6], v[7]);
  o1.x = pack_bf16x2(v[8], v[9]);
  o1.y = pack_bf16x2(v[10], v[11]);
  o1.z = pack_bf16x2(v[12], v[13]);
  o1.w = pack_bf16x2(v[14], v[15]);
  uint4* out = reinterpret_cast<uint4*>(d.out) + t * 2;
  out[0] = o0;
  out[1] = o1;
}

int plan_s2d_pack(ug_engine* h, const ug_s2d_desc* d, MemLaunch* L) {
  if ((!d->in_u8 && !d->in_f32) || !d->out || d->B <= 0 || d->S <= 0 || (d->S & 1) || misaligned(d->out, 16))
    return set_error(h, UG_EINVAL, "s2d_pack: bad args (even image side, 16-byte aligned output)");
  const int Q = d->S / 2 + 3;
  plan_grid(L, MemKernel::S2d, ceil_div((long long)d->B * Q * Q, 256), 256);
  return UG_OK;
}

int launch_s2d_pack(ug_engine* h, const ug_s2d_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_s2d_pack(h, d, &L);
  if (rc != UG_OK) return rc;
  launch_pdl(s2d_pack_kernel, L.grid, L.block, 0, s, *d);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "s2d_pack launch");
}

// ------------------------------------------------------------------------------------------------
// GoogLeNet head: global average pool + fc, one block per image.
__global__ void __launch_bounds__(256) head_kernel(ug_head_desc d) {
  pdl_wait();  // programmatic dependent launch: see common.cuh
  pdl_launch_dependents();
  __shared__ float s_avg[1024];
  const int n = blockIdx.x;
  const __nv_bfloat16* in = reinterpret_cast<const __nv_bfloat16*>(d.in) + (long long)n * d.HW * d.C;
  for (int c2 = threadIdx.x; c2 < d.C / 2; c2 += blockDim.x) {
    float a = 0.0f, b = 0.0f;
    for (int p = 0; p < d.HW; ++p) {
      const uint32_t w = *reinterpret_cast<const uint32_t*>(in + (long long)p * d.C + c2 * 2);
      a += bf16_lo(w);
      b += bf16_hi(w);
    }
    s_avg[c2 * 2] = a / (float)d.HW;
    s_avg[c2 * 2 + 1] = b / (float)d.HW;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int k = warp; k < d.ncls; k += 8) {
    float a = 0.0f;
    for (int c = lane; c < d.C; c += 32) a += d.w[(long long)k * d.C + c] * s_avg[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) d.logits[(long long)n * d.ncls + k] = a + d.b[k];
  }
}

int plan_head(ug_engine* h, const ug_head_desc* d, MemLaunch* L) {
  if (!d->in || !d->w || !d->b || !d->logits || d->C > 1024 || d->C % 2 || d->HW <= 0 || d->ncls <= 0)
    return set_error(h, UG_EINVAL, "head: bad args (C <= 1024)");
  if (misaligned(d->in, 4)) return set_error(h, UG_EINVAL, "head: in must be 4-byte aligned (read as bf16 pairs)");
  plan_grid(L, MemKernel::Head, d->B, 256);
  return UG_OK;
}

int launch_head(ug_engine* h, const ug_head_desc* d, cudaStream_t s) {
  MemLaunch L;
  const int rc = plan_head(h, d, &L);
  if (rc != UG_OK) return rc;
  launch_pdl(head_kernel, L.grid, L.block, 0, s, *d);
  h->launches++;
  return check_cuda(h, cudaGetLastError(), "head launch");
}

}  // namespace ug
