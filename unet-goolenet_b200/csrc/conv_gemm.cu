// Implicit-GEMM convolution / linear kernel for sm_100a.
//
//   D[pixels, Cout] = sum over taps (r,s) and 64-channel chunks of  A_tap[pixels, 64] * W[Cout, 64]^T
//
// * A tiles are rectangles of TW x TH x TN output pixels of the NHWC bf16 input, fetched by TMA as 4-D boxes
//   {64 channels, TW, TH, TN} whose (x,y) origin is shifted by the filter tap; out-of-bounds coordinates
//   (including negative ones) are zero-filled by TMA, which is exactly the conv zero padding.
// * B tiles are {64, BN} boxes of the packed weight matrix [Npad][R*S*Cin_pad] (K-major).
// * Both land in shared memory in the 128B-swizzled K-major layout that tcgen05.mma consumes directly.
// * One elected thread issues tcgen05.mma (M=128, N=BN, K=16) into a TMEM accumulator; four epilogue warps
//   read it back with tcgen05.ld (one output pixel per thread) and apply folded BN / bias, activation and the
//   fused epilogue (residual add, CoordAtt3 gate combine, ConvTranspose pixel shuffle, outc+sigmoid+threshold).
// * Warp roles: warps 0..3 = epilogue, warp 4 = TMA producer, warp 5 = TMEM allocator + MMA issuer.
//
// Reference ops this kernel replaces are listed on ug_conv_desc in include/ugnet.h.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include "conv_common.cuh"

namespace ug {


template <int kAct>
__global__ void __launch_bounds__(kThreads) conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA,
                                                             const __grid_constant__ CUtensorMap tmB,
                                                             const ConvKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  const int b_stage_bytes = p.BN * 128;
  uint8_t* sA = smem;
  uint8_t* sB = sA + p.stages * kABytesPerStage;
  float* sScale = reinterpret_cast<float*>(sB + p.stages * b_stage_bytes);  // 16-byte aligned: read as float4
  float* sBias = sScale + p.BN;
  uint64_t* full = reinterpret_cast<uint64_t*>(sBias + p.BN);
  uint64_t* empty = full + p.stages;
  uint64_t* tmem_full = empty + p.stages;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  // tile coordinates
  const int mt = blockIdx.x;
  const int x0 = (mt % p.tiles_x) * p.TW;
  const int y0 = ((mt / p.tiles_x) % p.tiles_y) * p.TH;
  const int n0 = (mt / (p.tiles_x * p.tiles_y)) * p.TN;
  const int ncol0 = blockIdx.y * p.BN;

  if (warp == kProducerWarp && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(tmem_ptr, p.tmem_cols);
    tmem_relinquish();
  }
  if (warp < 4) {
    for (int i = threadIdx.x; i < p.BN; i += 128) {
      const int n = ncol0 + i;
      sScale[i] = (n < p.N) ? (p.scale ? p.scale[n] : 1.0f) : 0.0f;
      sBias[i] = (n < p.N && p.bias) ? p.bias[n] : 0.0f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();                 // prologue above overlaps the previous kernel's tail (common.cuh)
  pdl_launch_dependents();

  if (warp == kProducerWarp) {
    // ------------------------------------------------------------------ TMA producer (whole warp, elected lane issues)
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx_bytes = p.a_bytes + p.b_bytes;
    int it = 0;
    for (int tap = 0; tap < p.R * p.S; ++tap) {
      const int r = tap / p.S, s = tap % p.S;
      for (int kc = 0; kc < p.kchunks; ++kc, ++it) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one_sync()) {
          mbar_arrive_expect_tx(&full[stage], tx_bytes);
          tma_load_4d(sA + stage * kABytesPerStage, &tmA, &full[stage], kc * 64, x0 + s - p.pad, y0 + r - p.pad, n0);
          tma_load_2d(sB + stage * b_stage_bytes, &tmB, &full[stage], it * 64, ncol0);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer (whole warp, elected lane issues)
    const uint32_t idesc = umma_idesc_bf16(128, p.BN);
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < p.num_k; ++it) {
      mbar_wait(&full[stage], phase);
      tc_fence_after();
      const uint64_t ad = umma_desc_sw128(smem_u32(sA + stage * kABytesPerStage));
      const uint64_t bd = umma_desc_sw128(smem_u32(sB + stage * b_stage_bytes));
      const uint32_t acc = it != 0 ? 1u : 0u;
      if (elect_one_sync()) {
        // +32 bytes (= 16 bf16) along K inside the 128B swizzle atom: +2 in the encoded start address
        umma_bf16(tmem_base, ad, bd, idesc, acc);
        umma_bf16(tmem_base, ad + 2, bd + 2, idesc, 1u);
        umma_bf16(tmem_base, ad + 4, bd + 4, idesc, 1u);
        umma_bf16(tmem_base, ad + 6, bd + 6, idesc, 1u);
        umma_commit(&empty[stage]);  // frees the smem slot once these MMAs have read it
        if (it == p.num_k - 1) umma_commit(tmem_full);  // accumulator complete
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (4 warps, 1 pixel / thread)
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const int tx = row % p.TW;
    const int trest = row / p.TW;
    const int ty = trest % p.TH;
    const int tn = trest / p.TH;
    const int x = x0 + tx, y = y0 + ty, n = n0 + tn;
    const bool valid = (row < p.TW * p.TH * p.TN) && (x < p.W) && (y < p.H) && (n < p.B);

    int dy = 0, dx = 0, cbase = ncol0;
    if (p.up == 2) {
      const int qd = ncol0 / p.convt_cout;
      dy = qd >> 1;
      dx = qd & 1;
      cbase = ncol0 % p.convt_cout;
    }
    const int oy = y * p.up + dy, ox = x * p.up + dx;
    const long long pix = (long long)oy * p.OW + ox;
    __nv_bfloat16* out_row =
        reinterpret_cast<__nv_bfloat16*>(p.out) + ((long long)n * p.OH * p.OW + pix) * p.out_cstride + cbase;
    int ncols = min(p.BN, p.N - ncol0);
    if (p.n_split) {  // split 1x1 GEMM: this n-tile lies entirely in one of the two column groups (BN divides n_split)
      if (ncol0 >= p.n_split)
        out_row = reinterpret_cast<__nv_bfloat16*>(p.out2) + ((long long)n * p.OH * p.OW + pix) * p.out2_cstride + (ncol0 - p.n_split);
      else
        ncols = min(p.BN, p.n1 - ncol0);  // (<= 0 for a tile of padding columns: nothing is stored)
    }
    const __nv_bfloat16* add_row =
        reinterpret_cast<const __nv_bfloat16*>(p.add) + (long long)n * p.add_bstride + pix * p.add_cstride + cbase;
    const float* gate_row = p.gate + (long long)n * p.N + ncol0;

    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    float dot = 0.0f;

    for (int c0 = 0; c0 < ncols; c0 += 16) {
      __syncwarp();  // tcgen05.ld is .sync.aligned: reconverge after the guarded stores
      uint32_t v[16];
      tmem_ld16(taddr + c0, v);
      tmem_ld_wait();
      float f[16];
      epi_math16<kAct>(v, f, sScale, sBias, c0);
      if (p.mode == UG_EPI_OUTC) {
#pragma unroll
        for (int j = 0; j < 16; ++j) dot += f[j] * __ldg(p.outc_w + ncol0 + c0 + j);
        continue;
      }
      const int groups = (c0 + 16 <= ncols) ? 2 : 1;  // N is a multiple of 8
      if ((p.mode == UG_EPI_ADD || p.mode == UG_EPI_GATE) && valid) {
        for (int g = 0; g < groups; ++g) epi_add_gate8(p, f + g * 8, add_row + c0 + g * 8, gate_row + c0 + g * 8);
      }
      for (int g = 0; g < groups; ++g) {
        uint4 o;
        o.x = pack_bf16x2(f[g * 8 + 0], f[g * 8 + 1]);
        o.y = pack_bf16x2(f[g * 8 + 2], f[g * 8 + 3]);
        o.z = pack_bf16x2(f[g * 8 + 4], f[g * 8 + 5]);
        o.w = pack_bf16x2(f[g * 8 + 6], f[g * 8 + 7]);
        // direct stores: each thread writes 16-byte pieces of its own pixel row.  A smem-staged, coalesced
        // copy-out was measured slower here (profiles/r01_notes.md): L2 merges the partial-line writes.
        if (valid) *reinterpret_cast<uint4*>(out_row + c0 + g * 8) = o;
      }
    }
    if (p.mode == UG_EPI_OUTC && valid) {
      const float logit = dot + p.outc_b;
      const long long o = ((long long)n * p.H + y) * p.W + x;
      p.logits[o] = logit;
      // torch.sigmoid(seg_out) > 0.5 evaluated in fp32 (roi.py:22-23, predict.py:26-27)
      const float sg = 1.0f / (1.0f + expf(-logit));
      p.mask[o] = sg > 0.5f ? 1 : 0;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, p.tmem_cols);
}


// ------------------------------------------------------------------------------------------------
// Persistent variant: one CTA per SM loops over (n-tile, pixel-tile) pairs.  The TMA producer and the MMA
// issuer run ahead across tile boundaries; accumulators are multi-buffered in TMEM (acc_stages x BN columns)
// so the epilogue of tile i overlaps the main loop of tile i+1; plain/ADD/GATE epilogues stage the bf16 tile
// in 128B-swizzled smem and write it with one TMA store per 64 channels (clipping handles ragged edges).
template <int kAct>
__global__ void __launch_bounds__(kThreads, 1) conv_gemm_persistent_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                           const __grid_constant__ CUtensorMap tmB,
                                                                           const __grid_constant__ CUtensorMap tmO,
                                                                           const __grid_constant__ CUtensorMap tmO2,
                                                                           const ConvKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  const int b_stage_bytes = p.BN * 128;
  const int n_sub = (p.BN + 63) / 64;
  const int obuf_bytes = (p.tma_store || p.stage_copy) ? n_sub * kABytesPerStage : 0;
  uint8_t* sA = smem;
  uint8_t* sB = sA + p.stages * kABytesPerStage;
  uint8_t* sO = sB + p.stages * b_stage_bytes;
  float* sScale = reinterpret_cast<float*>(sO + p.obufs * obuf_bytes);  // 16-byte aligned: read as float4
  float* sBias = sScale + p.npad;
  uint64_t* full = reinterpret_cast<uint64_t*>(sBias + p.npad);
  uint64_t* empty = full + p.stages;
  uint64_t* acc_full = empty + p.stages;
  uint64_t* acc_empty = acc_full + p.acc_stages;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + p.acc_stages);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.m_tiles * p.n_tiles;

  if (warp == kProducerWarp && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (p.tma_store) prefetch_tmap(&tmO);
    if (p.tma_store && p.n_split) prefetch_tmap(&tmO2);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < p.acc_stages; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4);  // one arrival per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(tmem_ptr, p.tmem_cols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < p.npad; i += kThreads) {
    sScale[i] = (i < p.N) ? (p.scale ? p.scale[i] : 1.0f) : 0.0f;
    sBias[i] = (i < p.N && p.bias) ? p.bias[i] : 0.0f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();                 // prologue above overlaps the previous kernel's tail (common.cuh)
  pdl_launch_dependents();

  if (warp == kProducerWarp) {
    // ------------------------------------------------------------------ TMA producer (whole warp, elected lane issues)
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx_bytes = p.a_bytes + p.b_bytes;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      // (m-major order: the n-tiles of a pixel tile run on neighbouring CTAs at the same time and share its HBM read)
      const int mt = p.m_major ? t / p.n_tiles : t % p.m_tiles, nt = p.m_major ? t % p.n_tiles : t / p.m_tiles;
      const int x0 = (mt % p.tiles_x) * p.TW;
      const int y0 = ((mt / p.tiles_x) % p.tiles_y) * p.TH;
      const int n0 = (mt / (p.tiles_x * p.tiles_y)) * p.TN;
      int it = 0;
      for (int tap = 0; tap < p.R * p.S; ++tap) {
        const int r = tap / p.S, s = tap % p.S;
        for (int kc = 0; kc < p.kchunks; ++kc, ++it) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (elect_one_sync()) {
            mbar_arrive_expect_tx(&full[stage], tx_bytes);
            tma_load_4d(sA + stage * kABytesPerStage, &tmA, &full[stage], kc * 64, x0 + s - p.pad, y0 + r - p.pad, n0);
            tma_load_2d(sB + stage * b_stage_bytes, &tmB, &full[stage], it * 64, nt * p.BN);
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer (whole warp, elected lane issues)
    const uint32_t idesc = umma_idesc_bf16(128, p.BN);
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      mbar_wait(&acc_empty[acc], acc_phase ^ 1);  // epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * p.BN;
      for (int it = 0; it < p.num_k; ++it) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint64_t ad = umma_desc_sw128(smem_u32(sA + stage * kABytesPerStage));
        const uint64_t bd = umma_desc_sw128(smem_u32(sB + stage * b_stage_bytes));
        const uint32_t accum = it != 0 ? 1u : 0u;
        if (elect_one_sync()) {
          umma_bf16(d_tmem, ad, bd, idesc, accum);
          umma_bf16(d_tmem, ad + 2, bd + 2, idesc, 1u);
          umma_bf16(d_tmem, ad + 4, bd + 4, idesc, 1u);
          umma_bf16(d_tmem, ad + 6, bd + 6, idesc, 1u);
          umma_commit(&empty[stage]);
          if (it == p.num_k - 1) umma_commit(&acc_full[acc]);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (++acc == p.acc_stages) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (4 warps, 1 pixel / thread)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int etid = threadIdx.x;  // 0..127
    const int tx = row % p.TW;
    const int trest = row / p.TW;
    const int ty = trest % p.TH;
    const int tn = trest / p.TH;
    const bool row_in_tile = row < p.TW * p.TH * p.TN;
    int acc = 0, obuf = 0;
    uint32_t acc_phase = 0;

    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      // (m-major order: the n-tiles of a pixel tile run on neighbouring CTAs at the same time and share its HBM read)
      const int mt = p.m_major ? t / p.n_tiles : t % p.m_tiles, nt = p.m_major ? t % p.n_tiles : t / p.m_tiles;
      const int x0 = (mt % p.tiles_x) * p.TW;
      const int y0 = ((mt / p.tiles_x) % p.tiles_y) * p.TH;
      const int n0 = (mt / (p.tiles_x * p.tiles_y)) * p.TN;
      const int ncol0 = nt * p.BN;
      const int x = x0 + tx, y = y0 + ty, n = n0 + tn;
      const bool valid = row_in_tile && (x < p.W) && (y < p.H) && (n < p.B);

      int dy = 0, dx = 0, cbase = ncol0;
      if (p.up == 2) {
        const int qd = ncol0 / p.convt_cout;
        dy = qd >> 1;
        dx = qd & 1;
        cbase = ncol0 % p.convt_cout;
      }
      const int oy = y * p.up + dy, ox = x * p.up + dx;
      const long long pix = (long long)oy * p.OW + ox;
      __nv_bfloat16* out_row =
          reinterpret_cast<__nv_bfloat16*>(p.out) + ((long long)n * p.OH * p.OW + pix) * p.out_cstride + cbase;
      const __nv_bfloat16* add_row =
          reinterpret_cast<const __nv_bfloat16*>(p.add) + (long long)n * p.add_bstride + pix * p.add_cstride + cbase;
      const float* gate_row = p.gate + (long long)n * p.N + ncol0;
      uint8_t* so_row = sO + obuf * obuf_bytes + row * 128;

      mbar_wait(&acc_full[acc], acc_phase);
      tc_fence_after();
      if (p.tma_store) {
        // the TMA store that last read this staging buffer must have finished reading it
        if (etid == 0) {
          if (p.obufs == 2) bulk_wait_group_read<1>();
          else bulk_wait_group_read<0>();
        }
        named_bar_sync(1, 128);
      }
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * p.BN;
      float dot = 0.0f;
      const int ncols = min(p.BN, p.N - ncol0);  // valid columns of this n-tile (multiple of 8)

      uint32_t v[16];
      __syncwarp();
      tmem_ld16(taddr, v);
      for (int c0 = 0; c0 < ncols; c0 += 16) {
        tmem_ld_wait();
        float f[16];
        epi_math16<kAct>(v, f, sScale, sBias, ncol0 + c0);
        __syncwarp();
        if (c0 + 16 < ncols) tmem_ld16(taddr + c0 + 16, v);  // next chunk in flight while this one is processed
        if (p.mode == UG_EPI_OUTC) {
#pragma unroll
          for (int j = 0; j < 16; ++j) dot += f[j] * __ldg(p.outc_w + ncol0 + c0 + j);
          continue;
        }
        const int groups = (c0 + 16 <= ncols) ? 2 : 1;
        if ((p.mode == UG_EPI_ADD || p.mode == UG_EPI_GATE) && valid) {
          for (int g = 0; g < groups; ++g) epi_add_gate8(p, f + g * 8, add_row + c0 + g * 8, gate_row + c0 + g * 8);
        }
        for (int g = 0; g < groups; ++g) {
          uint4 o;
          o.x = pack_bf16x2(f[g * 8 + 0], f[g * 8 + 1]);
          o.y = pack_bf16x2(f[g * 8 + 2], f[g * 8 + 3]);
          o.z = pack_bf16x2(f[g * 8 + 4], f[g * 8 + 5]);
          o.w = pack_bf16x2(f[g * 8 + 6], f[g * 8 + 7]);
          if (p.tma_store || p.stage_copy) {
            const int col = c0 + g * 8;
            const int sub = col >> 6, chunk = (col & 63) >> 3;
            *reinterpret_cast<uint4*>(so_row + sub * kABytesPerStage + ((chunk ^ (row & 7)) << 4)) = o;
          } else if (valid) {
            *reinterpret_cast<uint4*>(out_row + c0 + g * 8) = o;
          }
        }
      }
      // all TMEM reads of this accumulator are complete: hand it back to the MMA issuer
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[acc]);
      if (++acc == p.acc_stages) {
        acc = 0;
        acc_phase ^= 1;
      }
      if (p.mode == UG_EPI_OUTC) {
        if (valid) {
          const float logit = dot + p.outc_b;
          const long long o = ((long long)n * p.H + y) * p.W + x;
          p.logits[o] = logit;
          const float sg = 1.0f / (1.0f + expf(-logit));  // torch.sigmoid(seg_out) > 0.5 in fp32
          p.mask[o] = sg > 0.5f ? 1 : 0;
        }
      } else if (p.tma_store) {
        fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
        named_bar_sync(1, 128);
        if (etid == 0) {
          for (int sub = 0; sub * 64 < ncols; ++sub) {
            // split 1x1 GEMM: 64-column blocks at or beyond n_split belong to the second destination (the map of the
            // first one ends at n1, so its padding columns are clipped)
            const int col = ncol0 + sub * 64;
            if (p.n_split && col >= p.n_split)
              tma_store_4d(&tmO2, sO + obuf * obuf_bytes + sub * kABytesPerStage, col - p.n_split, x0, y0, n0);
            else
              tma_store_4d(&tmO, sO + obuf * obuf_bytes + sub * kABytesPerStage, col, x0, y0, n0);
          }
          bulk_commit_group();
        }
        if (p.obufs == 2) obuf ^= 1;
      } else if (p.stage_copy) {
        // ConvTranspose pixel shuffle: every output pixel owns a contiguous run of `ncols` channels, so the
        // staged tile is copied out with 16-byte stores that are contiguous across neighbouring threads.
        named_bar_sync(1, 128);
        const int cpr = ncols >> 3;  // 16-byte chunks per row
        const int nrows = p.TW * p.TH * p.TN;
        const uint8_t* sbuf = sO + obuf * obuf_bytes;
        for (int idx = etid; idx < nrows * cpr; idx += 128) {
          const int r2 = idx / cpr, ch = idx - r2 * cpr;
          const int tx2 = r2 % p.TW, rest = r2 / p.TW;
          const int x2 = x0 + tx2, y2 = y0 + rest % p.TH, n2 = n0 + rest / p.TH;
          if (x2 >= p.W || y2 >= p.H || n2 >= p.B) continue;
          const long long opix = (long long)(y2 * p.up + dy) * p.OW + (x2 * p.up + dx);
          __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) +
                               ((long long)n2 * p.OH * p.OW + opix) * p.out_cstride + cbase + ch * 8;
          const uint4 val = *reinterpret_cast<const uint4*>(sbuf + (ch >> 3) * kABytesPerStage + r2 * 128 +
                                                            (((ch & 7) ^ (r2 & 7)) << 4));
          *reinterpret_cast<uint4*>(dst) = val;
        }
        obuf ^= 1;  // two staging buffers: the barrier of the next tile orders reuse
      }
    }
    if (p.tma_store && etid == 0) bulk_wait_group_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, p.tmem_cols);
}

// ------------------------------------------------------------------------------------------ host side

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int encode_bf16_sw128(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                      const cuuint32_t* box, CUtensorMapL2promotion promo) {
  const cuuint32_t es[4] = {1, 1, 1, 1};
  return (int)get_encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides,
                              box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// Pick the pixel-tile rectangle with the best fill of the 128 MMA rows.
void choose_tile(int B, int H, int W, int* TW, int* TH, int* TN) {
  double best = -1.0;
  int bw = 1, bh = 1, bn = 1;
  for (int tw = 1; tw <= W && tw <= 128; ++tw) {
    for (int th = 1; th <= H && tw * th <= 128; ++th) {
      int tn = 1;
      if (tw == W && th == H) tn = std::max(1, std::min(B, 128 / (tw * th)));
      const double tiles = (double)ceil_div(W, tw) * ceil_div(H, th) * ceil_div(B, tn);
      const double eff = (double)W * H * B / (tiles * 128.0);
      // prefer higher efficiency; on ties prefer wider rows (longer contiguous TMA runs)
      if (eff > best + 1e-9 || (eff > best - 1e-9 && tw > bw)) {
        best = eff;
        bw = tw;
        bh = th;
        bn = tn;
      }
    }
  }
  *TW = bw;
  *TH = bh;
  *TN = bn;
}

int conv_prepare(ug_engine* h, const ug_conv_desc* d, ConvLaunch* L) {
  if (!get_encode_fn()) return set_error(h, UG_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
  if (!d->in || !d->w) return set_error(h, UG_EINVAL, "conv: null in/w pointer");
  if (d->B <= 0 || d->H <= 0 || d->W <= 0 || d->Cin <= 0 || d->N <= 0)
    return set_error(h, UG_EINVAL, "conv: non-positive shape");
  if (d->act < UG_ACT_NONE || d->act > UG_ACT_GELU) return set_error(h, UG_EINVAL, "conv: unknown activation");
  if (!(d->variant == 0 || d->variant == 1 || d->variant == 2 || (d->variant >= 5 && d->variant <= 7)))
    return set_error(h, UG_EINVAL, "conv: unknown variant %d (0, 1, 2, 5, 6 or 7)", d->variant);
  const bool rowtaps = d->R > 1 && d->S == 1 && d->pad == 0 && d->up != 2 && d->Cin <= 64;   // ug_conv_desc.in_rstride
  if (!rowtaps && (d->R <= 0 || d->S <= 0 || 2 * d->pad != d->R - 1 || d->R != d->S))
    return set_error(h, UG_EINVAL, "conv: only square stride-1 'same' filters (2*pad == R-1) or R x 1 row taps are supported");
  if ((d->in_rstride || d->in_bstride) && !(rowtaps || (d->R == 1 && d->variant == 5)))
    return set_error(h, UG_EINVAL, "conv: explicit input strides are for row-tap layers (multi-issuer kernel)");
  if (d->in_cstride % 8 || (reinterpret_cast<uintptr_t>(d->in) & 15))
    return set_error(h, UG_EINVAL, "conv: input channel stride must be a multiple of 8 and base 16B aligned");
  if (d->N % 8) return set_error(h, UG_EINVAL, "conv: N must be a multiple of 8");
  if (reinterpret_cast<uintptr_t>(d->w) & 15) return set_error(h, UG_EINVAL, "conv: weights must be 16B aligned");
  const int up = d->up == 2 ? 2 : 1;

  int BN = d->BN;
  if (BN <= 0) {
    if (d->N >= 128) BN = 128;
    else BN = ceil_div(d->N, 16) * 16;
    if (up == 2) BN = std::min(128, d->convt_cout);
  }
  if (BN % 16 || BN < 16 || BN > 256) return set_error(h, UG_EINVAL, "conv: BN must be a multiple of 16 in [16,256]");
  if (up == 2) {
    if (d->convt_cout <= 0 || d->N != 4 * d->convt_cout || (d->convt_cout % BN && d->variant != 5))
      return set_error(h, UG_EINVAL, "conv: ConvTranspose mode needs N == 4*cout and BN | cout");
    if (d->R != 1) return set_error(h, UG_EINVAL, "conv: ConvTranspose mode is a 1x1 GEMM");
  }
  if (d->mode == UG_EPI_OUTC) {
    if (d->N > BN || !d->outc_w || !d->logits || !d->mask)
      return set_error(h, UG_EINVAL, "conv: OUTC epilogue needs N <= BN and outc_w/logits/mask");
  } else {
    if (!d->out || d->out_cstride % 8 || (reinterpret_cast<uintptr_t>(d->out) & 15))
      return set_error(h, UG_EINVAL, "conv: output must be 16B aligned with channel stride multiple of 8");
  }
  if (d->mode == UG_EPI_ADD || d->mode == UG_EPI_GATE) {
    if (!d->add || d->add_cstride % 8 || d->add_bstride % 8 || (reinterpret_cast<uintptr_t>(d->add) & 15))
      return set_error(h, UG_EINVAL, "conv: add tensor must be 16B aligned with strides multiple of 8");
    if (d->mode == UG_EPI_GATE && !d->gate) return set_error(h, UG_EINVAL, "conv: GATE epilogue needs gate");
  }

  const bool split = d->out2 != nullptr || d->n_split != 0;
  if (split) {
    if (d->R != 1 || up != 1 || d->mode != UG_EPI_STORE || !d->out2 || d->n_split % 64 || d->n_split <= 0 ||
        d->n_split >= d->N || d->n1 <= 0 || d->n1 > d->n_split || d->n1 % 8 || d->out2_cstride % 8 ||
        (reinterpret_cast<uintptr_t>(d->out2) & 15) || d->variant == 5 || d->pool_out || d->stats_sum)
      return set_error(h, UG_EINVAL, "conv: a split GEMM is a 1x1 STORE layer with n_split %% 64 == 0 and 0 < n1 <= n_split < N");
    if (BN % 64) return set_error(h, UG_EINVAL, "conv: a split GEMM needs BN %% 64 == 0");
  }
  if (rowtaps) {
    if (split || d->variant == 1 || d->variant == 2) return set_error(h, UG_EINVAL, "conv: row-tap layers run on the multi-issuer kernel");
    return conv_multi_prepare(h, d, BN, L);
  }
  if (d->variant == 5) return conv_multi_prepare(h, d, d->R == 3 ? std::min(BN, 128) : BN, L);
  if (d->variant == 6) return conv_pair_prepare(h, d, L);
  if (d->variant == 7) return conv_multi_prepare(h, d, 128, L, 1);
  // 3x3 layers with <= 64 output channels on maps of at least 112x112 (the UNet's two finest levels): CTA-pair kernel
  // (conv_pair.cu, tcgen05.mma.cta_group::2) — profiles/r02_pair_kernel.txt: 64->64 0.221 -> 0.201 ms, + outc 0.208 ->
  // 0.176, 128->64 0.451 -> 0.359, 256->64 at 112x112 0.218 -> 0.188 per 64 images.  The CoordAtt3 combine on 64 input
  // channels is bound by its epilogue, not by the MMA, and stays on the multi-issuer kernel (0.277 against 0.291 ms).
  if (d->variant == 0 && d->R == 3 && up == 1 && d->N <= 64 && d->H * d->W >= 112 * 112 &&
      !(d->mode == UG_EPI_GATE && d->Cin <= 64)) {
    const int rc = conv_pair_prepare(h, d, L);
    if (rc == UG_OK) return rc;
    if (rc != UG_EUNSUPPORTED) return rc;
  }
  if (d->variant == 0 && up == 2 && d->H * d->W >= 196 && d->convt_cout % 64 == 0) {
    // ConvTranspose 2x2 s2 on maps of at least 14x14 (profiles/r02_convt_variants.txt): multi-issuer kernel (two epilogue warpgroups, pixel shuffle as
    // four strided TMA-store views); one 256-wide n-tile when that covers all four quadrants
    const int rc = conv_multi_prepare(h, d, d->N == 256 ? 256 : 128, L);
    if (rc == UG_OK) return rc;
    if (rc != UG_EUNSUPPORTED) return rc;
  }
  // 3x3 layers with 128-column n-tiles and streamed weights: clusters of two CTAs on the multi-issuer kernel (each CTA
  // streams half of every weight tile; conv_multi.cu header).  profiles/r02_pair128.txt, per 64 images: 112x112 128->128
  // 0.172 -> 0.148 ms (1600 TFLOP/s), 56x56 256->256 0.185 -> 0.164, 28x28 512->512 0.182 -> 0.169, 1024->256 0.204 ->
  // 0.186; the 256-image step +4.9 %.  Not routed: 64 input channels (resident weights, bound by the epilogue: 0.094 ->
  // 0.112 ms; GoogLeNet conv3 64->192 neutral).  The CoordAtt3 combine runs in pair mode with its residual sub-tiles
  // TMA-loaded by an extra warp (profiles/r02_resid_tma128.txt): 112x112 128->128 0.197 -> 0.165 ms.
  // GoogLeNet's 3x3 layers with N >= 128 (ragged last n-tile) gain 8-13 % each, the stage 2.151 -> 2.124 ms.
  if (d->variant == 0 && d->R == 3 && up == 1 && d->H * d->W >= 196 && !d->stats_sum && d->N >= 128 &&
      ((d->mode == UG_EPI_STORE && d->Cin > 64) || (d->mode == UG_EPI_GATE && d->Cin >= 128))) {
    const int rc = conv_multi_prepare(h, d, 128, L, 1);
    if (rc == UG_OK) return rc;
    if (rc != UG_EUNSUPPORTED) return rc;
  }
  if (d->variant == 0 && d->R == 3 && up == 1 && d->H * d->W >= 196) {
    // maps of at least 14x14: one CTA per SM, two MMA issuers sharing resident / streamed weights
    // (conv_multi.cu); measured against the other variants in profiles/r01_conv_sweep_multi_issuer.txt
    if (BN > 128 && BN < 256) {  // a single fitted n-tile (pack.choose_bn: N = 192 ... 224)
      const int rc = conv_multi_prepare(h, d, BN, L);
      if (rc == UG_OK) return rc;
      if (rc != UG_EUNSUPPORTED) return rc;
    }
    const int rc = conv_multi_prepare(h, d, std::min(BN, 128), L);
    if (rc == UG_OK) return rc;
    if (rc != UG_EUNSUPPORTED) return rc;
  }

  if (d->pool_out || d->stats_sum)
    return set_error(h, UG_EUNSUPPORTED, "conv: fused max-pool / channel statistics need the 3x3 multi-issuer kernel");
  int TW = d->TW, TH = d->TH, TN = d->TN;
  if (TW <= 0 || TH <= 0 || TN <= 0) choose_tile(d->B, d->H, d->W, &TW, &TH, &TN);
  if (TW * TH * TN > 128 || TW > 256 || TH > 256 || TN > 256)
    return set_error(h, UG_EINVAL, "conv: tile %dx%dx%d exceeds 128 rows", TW, TH, TN);

  const int cin_pad = ceil_div(d->Cin, 64) * 64;
  const int kchunks = cin_pad / 64;
  const int num_k = d->R * d->S * kchunks;
  const int n_tiles = ceil_div(d->N, BN);
  const long long ktot = (long long)d->R * d->S * cin_pad;

  // variant: 0 = auto, 1 = one tile per CTA, 2 = persistent.  Auto (measured, profiles/r01_conv_sweep.txt and
  // profiles/r01_gemm_sweep_1x1.txt): persistent for BN == 256; for 1x1 layers with many pixel tiles the one-tile
  // kernel (two CTAs per SM, 2-4 stages) is latency-bound: >= 1024 m-tiles -> multi-issuer kernel when K = 64
  // (one chunk), persistent otherwise; >= 296 m-tiles with BN > 64 -> persistent; else one tile per CTA.
  const int m_tiles_total = ceil_div(d->W, TW) * ceil_div(d->H, TH) * ceil_div(d->B, TN);
  int auto_persistent = BN == 256;
  if (d->variant == 0 && d->R == 1 && d->S == 1 && up == 1 && d->mode != UG_EPI_OUTC) {
    if (m_tiles_total >= 1024 && kchunks == 1 && (n_tiles == 1 || BN % 64 == 0) && !split) {
      const int rc = conv_multi_prepare(h, d, BN, L);
      if (rc == UG_OK) return rc;
      if (rc != UG_EUNSUPPORTED) return rc;
    }
    // (the persistent kernel stores 64-column TMA boxes: several n-tiles must then be multiples of 64 wide)
    const bool boxes_ok = n_tiles == 1 || BN % 64 == 0;
    if (boxes_ok && (m_tiles_total >= 1024 || (m_tiles_total >= 296 && BN > 64))) auto_persistent = 1;
  }
  if (split && d->n_split % BN) auto_persistent = 1;  // the one-tile kernel needs whole n-tiles on either side of n_split
  const bool persistent = d->variant == 2 || (d->variant != 1 && auto_persistent);
  if (split && !persistent && d->n_split % BN)
    return set_error(h, UG_EINVAL, "conv: split GEMM on the one-tile kernel needs BN to divide n_split (BN = 64)");
  const int tma_store = (persistent && up == 1 && d->mode != UG_EPI_OUTC) ? 1 : 0;
  const int stage_copy = (persistent && up == 2) ? 1 : 0;
  const int n_sub = ceil_div(BN, 64);
  const int obuf_bytes = (tma_store || stage_copy) ? n_sub * kABytesPerStage : 0;
  const int acc_stages = std::max(1, std::min(4, 512 / BN));
  const int npad = n_tiles * BN;
  int obufs = (persistent && (tma_store || stage_copy)) ? 2 : 0;
  int stages = d->stages;
  const int per_stage = kABytesPerStage + BN * 128;
  if (!persistent) {
    if (stages <= 0) {
      stages = (108 * 1024) / per_stage;  // two CTAs per SM
      stages = std::max(2, std::min(stages, 8));
    }
    stages = std::min(stages, std::max(2, num_k));
  } else {
    const int fixed = 1024 + 8 * (2 * 8 + 2 * acc_stages) + 16 + 2 * npad * (int)sizeof(float);
    const int budget = 227 * 1024 - fixed;
    int fit = (budget - obufs * obuf_bytes) / per_stage;
    if (tma_store && fit < 4) {
      obufs = 1;
      fit = (budget - obuf_bytes) / per_stage;
    }
    if (stages <= 0 || stages > fit) stages = fit;
    stages = std::max(2, std::min(stages, 8));
  }

  ConvKParams& p = L->p;
  memset(&p, 0, sizeof(p));
  p.H = d->H; p.W = d->W; p.B = d->B;
  p.TW = TW; p.TH = TH; p.TN = TN;
  p.tiles_x = ceil_div(d->W, TW);
  p.tiles_y = ceil_div(d->H, TH);
  const int tiles_n = ceil_div(d->B, TN);
  p.R = d->R; p.S = d->S; p.pad = d->pad;
  p.kchunks = kchunks; p.num_k = num_k;
  p.N = d->N; p.BN = BN; p.stages = stages;
  int tc = 32;
  while (tc < BN) tc <<= 1;
  p.tmem_cols = tc;
  p.a_bytes = (unsigned)(TW * TH * TN) * 128u;
  p.b_bytes = (unsigned)BN * 128u;
  p.scale = d->scale; p.bias = d->bias;
  p.act = d->act; p.mode = d->mode;
  p.out = d->out; p.out_cstride = d->out_cstride;
  p.up = up; p.convt_cout = d->convt_cout;
  p.OH = d->H * up; p.OW = d->W * up;
  p.add = d->add; p.add_bstride = d->add_bstride; p.add_cstride = d->add_cstride;
  p.gate = d->gate; p.outc_w = d->outc_w; p.outc_b = d->outc_b;
  p.logits = d->logits; p.mask = d->mask;
  p.m_tiles = m_tiles_total; p.n_tiles = n_tiles; p.acc_stages = acc_stages;
  p.m_major = n_tiles > 1 ? 1 : 0;
  p.tma_store = tma_store; p.obufs = obufs; p.npad = npad; p.stage_copy = stage_copy;
  p.out2 = d->out2; p.out2_cstride = d->out2_cstride; p.n_split = split ? d->n_split : 0; p.n1 = d->n1;
  L->kernel = persistent ? ConvKernel::Persistent : ConvKernel::OneTile;
  L->instance = d->act;   // conv_gemm_kernel / conv_gemm_persistent_kernel<UG_ACT_NONE, RELU, GELU>
  L->item_tiles = 1;
  L->block = kThreads;
  if (persistent) {
    int tcols = 32;
    while (tcols < acc_stages * BN) tcols <<= 1;
    p.tmem_cols = tcols;
  }
  if (tma_store) {
    cuuint64_t dims[4] = {(cuuint64_t)(split ? d->n1 : d->N), (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->out_cstride * 2, (cuuint64_t)d->W * d->out_cstride * 2,
                             (cuuint64_t)d->H * d->W * d->out_cstride * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TN};
    int r = encode_bf16_sw128(&L->tmO, d->out, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_NONE);
    if (r) return set_error(h, UG_ECUDA, "conv: output tensor map encode failed (%d)", r);
    memset(&L->tmO2, 0, sizeof(L->tmO2));
    if (split) {
      cuuint64_t dims2[4] = {(cuuint64_t)(d->N - d->n_split), (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
      cuuint64_t strides2[3] = {(cuuint64_t)d->out2_cstride * 2, (cuuint64_t)d->W * d->out2_cstride * 2,
                                (cuuint64_t)d->H * d->W * d->out2_cstride * 2};
      r = encode_bf16_sw128(&L->tmO2, d->out2, 4, dims2, strides2, box, CU_TENSOR_MAP_L2_PROMOTION_NONE);
      if (r) return set_error(h, UG_ECUDA, "conv: second output tensor map encode failed (%d)", r);
    }
  } else {
    memset(&L->tmO, 0, sizeof(L->tmO));
    memset(&L->tmO2, 0, sizeof(L->tmO2));
  }

  {
    cuuint64_t dims[4] = {(cuuint64_t)d->Cin, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->in_cstride * 2, (cuuint64_t)d->W * d->in_cstride * 2,
                             (cuuint64_t)d->H * d->W * d->in_cstride * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TN};
    const int r = encode_bf16_sw128(&L->tmA, d->in, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
    if (r) return set_error(h, UG_ECUDA, "conv: activation tensor map encode failed (%d)", r);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)n_tiles * BN};
    cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)BN};
    const int r = encode_bf16_sw128(&L->tmB, d->w, 2, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
    if (r) return set_error(h, UG_ECUDA, "conv: weight tensor map encode failed (%d)", r);
  }
  if (!persistent) {
    L->grid = dim3((unsigned)(p.tiles_x * p.tiles_y * tiles_n), (unsigned)n_tiles, 1);
    L->smem = 1024 + (size_t)stages * per_stage + 8 * (2 * stages + 1) + 8 + 2 * BN * sizeof(float);
  } else {
    const long long total = (long long)m_tiles_total * n_tiles;
    L->grid = dim3((unsigned)std::min<long long>(total, h->num_sms), 1, 1);
    L->smem = 1024 + (size_t)stages * per_stage + (size_t)obufs * obuf_bytes + 8 * (2 * stages + 2 * acc_stages) + 16 +
              2 * (size_t)npad * sizeof(float);
  }
  if (L->smem > 227 * 1024) return set_error(h, UG_EINVAL, "conv: shared memory request %zu too large", L->smem);
  return UG_OK;
}

int conv_launch(ug_engine* h, const ConvLaunch* L, cudaStream_t s) {
  if (!h->attr_gemm) {
    cudaError_t e = cudaSuccess;
    const int kMax = 227 * 1024;
    const void* fns[] = {(const void*)conv_gemm_kernel<UG_ACT_NONE>,
                         (const void*)conv_gemm_kernel<UG_ACT_RELU>,
                         (const void*)conv_gemm_kernel<UG_ACT_GELU>,
                         (const void*)conv_gemm_persistent_kernel<UG_ACT_NONE>,
                         (const void*)conv_gemm_persistent_kernel<UG_ACT_RELU>,
                         (const void*)conv_gemm_persistent_kernel<UG_ACT_GELU>};
    for (const void* f : fns)
      if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax);
    if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(conv_gemm kernels)");
    h->attr_gemm = true;
  }
  const int act = L->p.act;
  cudaError_t le = cudaErrorInvalidValue;
  switch (L->kernel) {
    case ConvKernel::Multi:
    case ConvKernel::MultiPair: return conv_multi_launch(h, L, s);
    case ConvKernel::Pair: return conv_pair_launch(h, L, s);
    case ConvKernel::OneTile: {
      auto fn = act == UG_ACT_RELU ? conv_gemm_kernel<UG_ACT_RELU>
                : act == UG_ACT_GELU ? conv_gemm_kernel<UG_ACT_GELU> : conv_gemm_kernel<UG_ACT_NONE>;
      le = launch_pdl(fn, L->grid, L->block, L->smem, s, L->tmA, L->tmB, L->p);
      break;
    }
    case ConvKernel::Persistent: {
      auto fn = act == UG_ACT_RELU ? conv_gemm_persistent_kernel<UG_ACT_RELU>
                : act == UG_ACT_GELU ? conv_gemm_persistent_kernel<UG_ACT_GELU> : conv_gemm_persistent_kernel<UG_ACT_NONE>;
      le = launch_pdl(fn, L->grid, L->block, L->smem, s, L->tmA, L->tmB, L->tmO, L->tmO2, L->p);
      break;
    }
  }
  h->launches++;
  return check_cuda(h, le != cudaSuccess ? le : cudaGetLastError(), "conv_gemm kernel launch");
}

}  // namespace ug
