// Stem convolution (the UNet's 3-input-channel layer) as a fused implicit GEMM on tcgen05: the im2col tile is built
// directly in shared memory from the source image, so no im2col matrix ever reaches HBM.
//
//   kind 0  UNet `inc`  (basicUnet.py:409, ConvBatchNorm :25-40): 3x3, stride 1, pad 1 on fp32 NCHW [B,3,H,W]
//           K index = (r*3+s)*3+c, 27 real columns, two K=16 MMAs (columns 27..31 are written as zeros).
// (GoogLeNet's conv1 runs as ug_s2d_pack + a row-tap implicit GEMM on the multi-issuer kernel, see lower.py.)
//
// One warpgroup (128 threads) = one 16x8 tile of output pixels (thread t <-> pixel row t of the MMA <-> TMEM lane t),
// N = 64 output channels.  A CTA holds kGroups = 6 independent warpgroups (own A tile, patch, accumulator and named
// barrier, one shared copy of the weights) at 80 registers per thread: 0.296 -> 0.263 ms per 128 images against five
// single-warpgroup CTAs per SM.  Per tile: every thread writes its im2col row into the 128B-swizzled K-major A tile ->
// one thread issues the MMAs -> all threads read their accumulator row from TMEM, apply folded BN + ReLU, stage the
// bf16 tile in swizzled smem -> TMA store.  The phases of one warpgroup are serial; the co-resident warpgroups of an SM
// overlap them.  The layer is bound by the 64-channel output write (128 B per pixel), not by the tensor pipe.
#include <cstring>
#include "conv_common.cuh"

namespace ug {

static constexpr int kStemTW = 16, kStemTH = 8;          // output tile
static constexpr int kStemGroups = 6;                    // warpgroups per CTA
static constexpr int kIncPatchH = kStemTH + 2, kIncPatchW = kStemTW + 2;   // 10 x 18 source pixels per channel
static constexpr int kIncPatchPitch = 48;                // floats per patch row: the two tile rows of a warp (ty, ty+1)
                                                         // then read banks [tx+s, ..] and [16+tx+s, ..]: no conflicts
static constexpr int kStemPoolBytes = 4096;  // pooled tile staging: 8 x 4 pixels x 64 channels bf16

// (instantiated as stem_conv_kernel<0, kStemGroups> only: kind 0 = inc)
template <int kKind, int kGroups>
__global__ void __launch_bounds__(128 * kGroups) stem_conv_kernel(const __grid_constant__ CUtensorMap tmB,
                                                        const __grid_constant__ CUtensorMap tmO,
                                                        const __grid_constant__ CUtensorMap tmP, const StemParams p) {
  static_assert(kKind == 0, "stem kind 0 (inc) only");
  constexpr int kAtoms = 1;                              // 64-column swizzle atoms of the A / B tiles
  constexpr int kKSteps = 2;                             // K=16 MMAs per tile
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  constexpr int kPatchBytes = 3 * kIncPatchH * kIncPatchPitch * 4;
  constexpr int kPatchAlloc = (kPatchBytes + 1023) / 1024 * 1024;
  constexpr uint32_t kTmemCols = kGroups == 1 ? 64 : (kGroups == 2 ? 128 : (kGroups <= 4 ? 256 : 512));
  const int grp = threadIdx.x >> 7;                      // warpgroup: an independent tile pipeline
  const int tid = threadIdx.x & 127;                     // thread within the warpgroup = pixel row of the tile
  const int warp = tid >> 5;                             // warp within the warpgroup = TMEM lane quarter
  const int group_bytes = kAtoms * kABytesPerStage + (p.pool ? kStemPoolBytes : 0) + kPatchAlloc;
  uint8_t* sB = smem;                                    // kAtoms x [64 rows][128 B], shared by the warpgroups
  uint8_t* sA = sB + kAtoms * 64 * 128 + grp * group_bytes;   // kAtoms x [128 rows][128 B]
  uint8_t* sO = sA;                                      // output staging [128 rows][128 B] reuses the first A atom:
                                                         // the A tile is dead once the MMAs of the tile completed
  uint8_t* sPool = sA + kAtoms * kABytesPerStage;        // pooled tile staging (4 KB, 1024-aligned) when p.pool
  float* sPatchF = reinterpret_cast<float*>(sPool + (p.pool ? kStemPoolBytes : 0));   // fp32 source patch
  uint8_t* tail = sB + kAtoms * 64 * 128 + kGroups * group_bytes;
  float* sScale = reinterpret_cast<float*>(tail);       // 16-byte aligned: read as float4
  float* sBias = sScale + 64;
  uint64_t* b_full = reinterpret_cast<uint64_t*>(sBias + 64);
  uint64_t* acc_full = b_full + 1 + grp;                 // one accumulator barrier per warpgroup
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_full + 1 + kGroups);
  auto group_sync = [&]() {
    if constexpr (kGroups == 1) __syncthreads();
    else named_bar_sync(1 + grp, 128);
  };

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmO);
    if (p.pool) prefetch_tmap(&tmP);
    mbar_init(b_full, 1);
    for (int g = 0; g < kGroups; ++g) mbar_init(b_full + 1 + g, 1);
    fence_mbar_init();
  }
  if (threadIdx.x < 32) {
    tmem_alloc(tmem_ptr, kTmemCols);
    tmem_relinquish();
  }
  if (threadIdx.x < 64) {
    sScale[threadIdx.x] = p.scale ? p.scale[threadIdx.x] : 1.0f;
    sBias[threadIdx.x] = p.bias ? p.bias[threadIdx.x] : 0.0f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_alloc_base = *tmem_ptr;
  const uint32_t tmem_base = tmem_alloc_base + grp * 64;   // this warpgroup's 64 accumulator columns
  if (threadIdx.x == 0) {  // the whole weight matrix, once per CTA
    mbar_arrive_expect_tx(b_full, (uint32_t)(kAtoms * 64 * 128));
    for (int a = 0; a < kAtoms; ++a) tma_load_2d(sB + a * 64 * 128, &tmB, b_full, a * 64, 0);
  }
  pdl_wait();                 // the prologue and the (constant) weight load overlap the previous kernel's tail
  pdl_launch_dependents();

  const int tx = tid & (kStemTW - 1);
  const int ty = tid >> 4;
  uint8_t* a_row = sA + tid * 128;
  uint8_t* o_row = sO + tid * 128;
  const int sw = tid & 7;
  const uint32_t idesc = umma_idesc_bf16(128, 64);
  uint32_t acc_phase = 0;
  bool b_ready = false;

  // inc: the fp32 source patch (3 x 10 x 18, zero outside the image) of a tile is fetched with coalesced loads ONE TILE
  // AHEAD into registers: fetched in the same iteration, every tile exposed one HBM latency (20 % of the samples)
  constexpr int kIncElems = 3 * kIncPatchH * kIncPatchW;  // 540
  constexpr int kIncSteps = (kIncElems + 127) / 128;
  float inc_raw[kIncSteps];
  auto load_inc_patch = [&](int t2) {
    const int px0 = (t2 % p.tiles_x) * kStemTW, py0 = ((t2 / p.tiles_x) % p.tiles_y) * kStemTH;
    const float* xn = p.in_f32 + (long long)(t2 / (p.tiles_x * p.tiles_y)) * 3 * p.H * p.W;
#pragma unroll
    for (int k = 0; k < kIncSteps; ++k) {
      const int idx = tid + k * 128;
      const int c = idx / (kIncPatchH * kIncPatchW), rem = idx - c * (kIncPatchH * kIncPatchW);
      const int r = rem / kIncPatchW, xx = rem - r * kIncPatchW;
      const int iy = py0 - 1 + r, ix = px0 - 1 + xx;
      const bool inb = idx < kIncElems && iy >= 0 && iy < p.H && ix >= 0 && ix < p.W;
      inc_raw[k] = inb ? __ldg(xn + ((long long)c * p.H + iy) * p.W + ix) : 0.0f;
    }
  };
  const int t_first = blockIdx.x * kGroups + grp, t_stride = gridDim.x * kGroups;
  if (t_first < p.total_tiles) load_inc_patch(t_first);

  for (int t = t_first; t < p.total_tiles; t += t_stride) {
    const int x0 = (t % p.tiles_x) * kStemTW;
    const int y0 = ((t / p.tiles_x) % p.tiles_y) * kStemTH;
    const int n = t / (p.tiles_x * p.tiles_y);

    // ---- inc: stage the 3 x 10 x 18 fp32 source patch (zero outside the image) with coalesced loads, then every
    // thread gathers its 27 taps from shared memory
    // (the patch values of THIS tile were fetched into inc_raw one tile ahead, see load_inc_patch below)
#pragma unroll
    for (int k = 0; k < kIncSteps; ++k) {
      const int idx = tid + k * 128;
      const int c = idx / (kIncPatchH * kIncPatchW), rem = idx - c * (kIncPatchH * kIncPatchW);
      const int r = rem / kIncPatchW, xx = rem - r * kIncPatchW;
      if (idx < kIncElems) sPatchF[(c * kIncPatchH + r) * kIncPatchPitch + xx] = inc_raw[k];
    }
    if (tid == 0) bulk_wait_group_read<0>();  // previous tile's TMA store has finished reading sO (= sA)
    group_sync();
    if (t + t_stride < p.total_tiles) load_inc_patch(t + t_stride);         // next tile's patch: in flight during
                                                                            // the gather, the MMA and the epilogue
    const float* pt = sPatchF + ty * kIncPatchPitch + tx;
    float v[32];
#pragma unroll
    for (int i = 27; i < 32; ++i) v[i] = 0.0f;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int sx = 0; sx < 3; ++sx)
#pragma unroll
        for (int c = 0; c < 3; ++c)
          v[(r * 3 + sx) * 3 + c] = pt[(c * kIncPatchH + r) * kIncPatchPitch + sx];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      uint4 o;
      o.x = pack_bf16x2(v[g * 8 + 0], v[g * 8 + 1]);
      o.y = pack_bf16x2(v[g * 8 + 2], v[g * 8 + 3]);
      o.z = pack_bf16x2(v[g * 8 + 4], v[g * 8 + 5]);
      o.w = pack_bf16x2(v[g * 8 + 6], v[g * 8 + 7]);
      *reinterpret_cast<uint4*>(a_row + ((g ^ sw) << 4)) = o;
    }
    fence_proxy_async_smem();  // generic-proxy writes of the A tile -> visible to the tensor core (async proxy)
    tc_fence_before();
    group_sync();
    if (tid == 0) {
      tc_fence_after();
      if (!b_ready) {
        mbar_wait(b_full, 0);
        b_ready = true;
      }
#pragma unroll
      for (int k = 0; k < kKSteps; ++k) {
        const uint64_t ad = umma_desc_sw128(smem_u32(sA + (k >> 2) * kABytesPerStage)) + 2 * (k & 3);
        const uint64_t bd = umma_desc_sw128(smem_u32(sB + (k >> 2) * 64 * 128)) + 2 * (k & 3);
        umma_bf16(tmem_base, ad, bd, idesc, k != 0 ? 1u : 0u);
      }
      umma_commit(acc_full);
    }
    mbar_wait(acc_full, acc_phase);
    acc_phase ^= 1;
    tc_fence_after();
    // ---- epilogue: folded BN + ReLU, bf16, swizzled staging, TMA store of the 16x8x64 tile
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 16) {
      uint32_t v[16];
      tmem_ld16(taddr + c0, v);
      tmem_ld_wait();
      float f[16];
      epi_math16<UG_ACT_NONE>(v, f, sScale, sBias, c0);   // ReLU folded into the bf16 conversion
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        uint4 o;
        o.x = pack_bf16x2_relu(f[g * 8 + 0], f[g * 8 + 1]);
        o.y = pack_bf16x2_relu(f[g * 8 + 2], f[g * 8 + 3]);
        o.z = pack_bf16x2_relu(f[g * 8 + 4], f[g * 8 + 5]);
        o.w = pack_bf16x2_relu(f[g * 8 + 6], f[g * 8 + 7]);
        *reinterpret_cast<uint4*>(o_row + ((((c0 >> 3) + g) ^ sw) << 4)) = o;
        if (p.pool) {
          // fused nn.MaxPool2d(2): pixel (tx, ty) = row ty*16 + tx; its 2x2 window lives in lanes ^1 (x) and ^16 (y)
          uint4 m = o;
          m.x = bf16x2_max(m.x, __shfl_xor_sync(0xffffffffu, m.x, 1));
          m.y = bf16x2_max(m.y, __shfl_xor_sync(0xffffffffu, m.y, 1));
          m.z = bf16x2_max(m.z, __shfl_xor_sync(0xffffffffu, m.z, 1));
          m.w = bf16x2_max(m.w, __shfl_xor_sync(0xffffffffu, m.w, 1));
          m.x = bf16x2_max(m.x, __shfl_xor_sync(0xffffffffu, m.x, 16));
          m.y = bf16x2_max(m.y, __shfl_xor_sync(0xffffffffu, m.y, 16));
          m.z = bf16x2_max(m.z, __shfl_xor_sync(0xffffffffu, m.z, 16));
          m.w = bf16x2_max(m.w, __shfl_xor_sync(0xffffffffu, m.w, 16));
          if (((tx | ty) & 1) == 0) {
            const int pr = (ty >> 1) * 8 + (tx >> 1);  // pooled pixel row of the 8 x 4 tile
            *reinterpret_cast<uint4*>(sPool + pr * 128 + ((((c0 >> 3) + g) ^ (pr & 7)) << 4)) = m;
          }
        }
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    group_sync();     // staging complete; every TMEM read of this accumulator is done
    if (tid == 0) {
      tma_store_4d(&tmO, sO, 0, x0, y0, n);
      if (p.pool) tma_store_4d(&tmP, sPool, 0, x0 >> 1, y0 >> 1, n);
      bulk_commit_group();
    }
  }
  if (tid == 0) bulk_wait_group_all();
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc(tmem_alloc_base, kTmemCols);
}

// ------------------------------------------------------------------------------------------ host side
int stem_prepare(ug_engine* h, const ug_stem_desc* d, StemLaunch* L) {
  if (!get_encode_fn()) return set_error(h, UG_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
  if (d->kind != 0) return set_error(h, UG_EINVAL, "stem: kind must be 0 (inc)");
  if (!d->w || !d->out || d->B <= 0 || d->H <= 0 || d->W <= 0) return set_error(h, UG_EINVAL, "stem: bad args");
  if (!d->in_f32) return set_error(h, UG_EINVAL, "stem(inc): fp32 NCHW input required");
  if (d->out_cstride % 8 || d->out_cstride < 64 || (reinterpret_cast<uintptr_t>(d->out) & 15) ||
      (reinterpret_cast<uintptr_t>(d->w) & 15))
    return set_error(h, UG_EINVAL, "stem: out/w must be 16B aligned, channel stride a multiple of 8 (>= 64)");
  const int OH = d->H, OW = d->W;
  memset(L, 0, sizeof(*L));
  StemParams& p = L->p;
  p.in_f32 = d->in_f32; p.scale = d->scale; p.bias = d->bias;
  p.B = d->B; p.H = d->H; p.W = d->W; p.OH = OH; p.OW = OW;
  p.tiles_x = (OW + kStemTW - 1) / kStemTW;
  p.tiles_y = (OH + kStemTH - 1) / kStemTH;
  p.total_tiles = p.tiles_x * p.tiles_y * d->B;
  p.pool = d->pool_out != nullptr;
  if (p.pool && ((d->H & 1) || (d->W & 1) || d->pool_cstride % 8 || d->pool_cstride < 64 ||
                 (reinterpret_cast<uintptr_t>(d->pool_out) & 15)))
    return set_error(h, UG_EINVAL, "stem: fused max-pool needs an even image, 16B-aligned pooled output");
  {
    cuuint64_t dims[2] = {64, 64};
    cuuint64_t strides[1] = {64 * 2};
    cuuint32_t box[2] = {64, 64};
    const int r = encode_bf16_sw128(&L->tmB, d->w, 2, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
    if (r) return set_error(h, UG_ECUDA, "stem: weight tensor map encode failed (%d)", r);
  }
  {
    cuuint64_t dims[4] = {64, (cuuint64_t)OW, (cuuint64_t)OH, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->out_cstride * 2, (cuuint64_t)OW * d->out_cstride * 2,
                             (cuuint64_t)OH * OW * d->out_cstride * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)kStemTW, (cuuint32_t)kStemTH, 1};
    const int r = encode_bf16_sw128(&L->tmO, d->out, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_NONE);
    if (r) return set_error(h, UG_ECUDA, "stem: output tensor map encode failed (%d)", r);
  }
  if (p.pool) {
    const long long pcs = d->pool_cstride;
    cuuint64_t dims[4] = {64, (cuuint64_t)(OW / 2), (cuuint64_t)(OH / 2), (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)(pcs * 2), (cuuint64_t)((OW / 2) * pcs * 2),
                             (cuuint64_t)((long long)(OH / 2) * (OW / 2) * pcs * 2)};
    cuuint32_t box[4] = {64, (cuuint32_t)(kStemTW / 2), (cuuint32_t)(kStemTH / 2), 1};
    const int r = encode_bf16_sw128(&L->tmP, d->pool_out, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_NONE);
    if (r) return set_error(h, UG_ECUDA, "stem: pooled output tensor map encode failed (%d)", r);
  }
  // one CTA per SM: its warpgroups share the weights (see the header comment)
  L->grid = (unsigned)std::min<long long>((p.total_tiles + kStemGroups - 1) / kStemGroups, (long long)h->num_sms);
  L->block = 128 * kStemGroups;
  const size_t patch = 3 * kIncPatchH * kIncPatchPitch * 4;
  L->smem = 1024 + (size_t)64 * 128 +
            kStemGroups * ((size_t)kABytesPerStage + (p.pool ? kStemPoolBytes : 0) + (patch + 1023) / 1024 * 1024) +
            2 * 64 * sizeof(float) + 8 * (1 + kStemGroups) + 16;
  return UG_OK;
}

int stem_launch(ug_engine* h, const StemLaunch* L, cudaStream_t s) {
  if (!h->attr_stem) {
    const cudaError_t e = cudaFuncSetAttribute((const void*)stem_conv_kernel<0, kStemGroups>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, 210 * 1024);
    if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(stem_conv_kernel)");
    h->attr_stem = true;
  }
  const cudaError_t le = launch_pdl(stem_conv_kernel<0, kStemGroups>, L->grid, L->block, L->smem, s, L->tmB,
                                    L->tmO, L->tmP, L->p);
  h->launches++;
  return check_cuda(h, le != cudaSuccess ? le : cudaGetLastError(), "stem_conv_kernel launch");
}

}  // namespace ug
