// 3x3 convolution (stride 1, pad 1) with <= 64 output channels on CTA PAIRS: tcgen05.mma.cta_group::2.
//
// The 64-channel layers of the two finest UNet levels (224x224: conv1_e, nConvs.0 128->64, nConvs.1 + outc; 112x112:
// nConvs.1) are bounded by the shared-memory operand bandwidth of the MMA: an M=128 x N=64 x K=16 MMA reads A 4 KB +
// B 2 KB for 32 cycles of math (profiles/r01_mma_multi_issuer.txt: 53-55 cycles per MMA per SM with four chains, the
// K-split kernel of conv_multi.cu).  A CTA pair issues ONE M=256 MMA for both SMs: each CTA supplies its own 128 pixel
// rows (its own halo tile) and HALF of the weight rows (N/2 = 32), the hardware exchanges the weight halves — 5 KB
// instead of 6 KB of operand reads per SM per MMA, half the resident weight footprint (128->64 becomes resident:
// 72 KB per CTA), and one instruction issue for two SMs.  ug_mma_microbench_pair (profiles/r02_mma_pair.txt): one M=256
// N=64 MMA per 47 cycles per pair with 2-4 issuing warps.
//
// Structure = conv_multi_kernel<RELU, 9, mode, K-split> per CTA (two pixel-tile streams, two epilogue warpgroups, halo
// activation tiles, weights resident, two issuing warps per stream taking alternate (chunk, tap) items into their own
// accumulators), with the pair protocol on top:
//   * the LEADER CTA (cluster rank 0) issues every MMA; its a_full / b_full barriers collect the TMA bytes of BOTH
//     CTAs (the peer's loads use the .cta_group::2 form, which may signal the leader's barrier);
//   * tcgen05.commit ... multicast::cluster arrives on the a_empty / acc_full barriers of BOTH CTAs;
//   * the peer's epilogue warps hand accumulators back with remote arrives on the leader's acc_empty;
//   * TMEM: each CTA allocates all 512 columns with cta_group::2, so accumulator addresses coincide in both CTAs;
//   * tiles are handed out in groups of four (2 streams x 2 CTAs); a tile index past the end maps to an image index
//     >= B: TMA zero-fills its loads and clips its stores, so every role runs the same number of rounds;
//   * layers whose resident weight halves leave no room for two streams (192 / 256 input channels: 108 / 144 KB per
//     CTA) run ONE stream per CTA (hp.streams = 1; its two K-split issuers still keep the pair's tensor pipes at the
//     two-chain rate of profiles/r02_mma_pair.txt, and the epilogue of such a layer is 1/4 of its MMA time);
//   * the CoordAtt3 combine (GATE epilogue, kRT) uses the residual-by-TMA protocol of conv_multi.cu: the weight warp
//     loads the residual tile of the NEXT tile into the free staging buffer, the epilogue combines in place.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "conv_common.cuh"

namespace ug {

static constexpr int kPThreads = 448;   // warps 0-3 / 4-7 epilogue of stream 0 / 1, 8 alloc + weights, 9 activations, 10-13 issuers
static constexpr int kPI = 2;           // tile streams per CTA
static constexpr int kPKS = 2;          // issuing warps per stream (K-split)
static constexpr int kPPitch = 10;      // halo pitch: 8 output pixels + one border pixel on each side
static constexpr int kPAllocWarp = 8, kPProducerWarp = 9, kPIssuerWarp0 = 10;
static constexpr int kPAcc = 2;         // accumulator stages per (stream, K-half): 2 x 2 x 2 x 64 = 512 TMEM columns
static constexpr int kPPoolBytes = 4096;

template <int kMode, int kRT>
__global__ void __launch_bounds__(kPThreads, 1) conv_pair_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                 const __grid_constant__ CUtensorMap tmB,
                                                                 const __grid_constant__ PairMaps tmO, const ConvKParams p,
                                                                 const PairParams hp) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr int kBTile = 32 * 128;                       // this CTA's half of a 64-row weight tile
  const int nb_tiles = 9 * p.kchunks;
  const int obuf_bytes = p.tma_store ? kABytesPerStage : 0;
  const int nstr = hp.streams;
  uint8_t* sA = smem;                                    // [streams][sa] activation stages
  uint8_t* sB = sA + nstr * hp.sa * hp.a_stage_bytes;    // [kchunks][9] weight half-tiles (resident)
  uint8_t* sO = sB + nb_tiles * kBTile;                  // [streams][obufs] output staging
  uint8_t* sP = sO + nstr * p.obufs * obuf_bytes;        // [streams][obufs] pooled staging when p.pool
  float* sScale = reinterpret_cast<float*>(sP + (p.pool ? nstr * p.obufs * kPPoolBytes : 0));
  float* sBias = sScale + 64;
  float* sGate = sBias + 64;                                    // [kPI][64]: 1 + gate of the tile's image (GATE epilogue)
  uint64_t* a_full = reinterpret_cast<uint64_t*>(sGate + kPI * 64);   // [kPI][sa]   (leader's instance is the live one)
  uint64_t* a_empty = a_full + kPI * hp.sa;                     // [kPI][sa]   (own instance, multicast commits)
  uint64_t* b_full = a_empty + kPI * hp.sa;                     // [1]         (leader's)
  uint64_t* acc_full = b_full + 1;                              // [kPI][kPAcc] (own instance, multicast commits)
  uint64_t* acc_empty = acc_full + kPI * kPAcc;                 // [kPI][kPAcc] (leader's, 8 arrivals)
  uint64_t* r_full = acc_empty + kPI * kPAcc;                   // [kPI][2] residual tile landed in staging buffer b (kRT, own)
  uint64_t* r_free = r_full + kPI * 2;                          // [kPI][2] staging buffer b may be overwritten (kRT, own)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(r_free + kPI * 2);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (warp == kPProducerWarp && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (p.tma_store) {
      prefetch_tmap(&tmO.out);
      if (p.pool) prefetch_tmap(&tmO.pool);
    }
    for (int i = 0; i < kPI * hp.sa; ++i) {
      mbar_init(&a_full[i], 1);        // the leader's arrive.expect_tx for the bytes of both CTAs
      mbar_init(&a_empty[i], kPKS);    // both issuers of the stream have finished reading the stage (multicast commits)
    }
    mbar_init(b_full, 1);
    for (int i = 0; i < kPI * kPAcc; ++i) {
      mbar_init(&acc_full[i], kPKS);   // both K-halves of the tile are complete (multicast commits)
      mbar_init(&acc_empty[i], 8);     // the four epilogue warps of the stream in BOTH CTAs
    }
    for (int i = 0; i < kPI * 2; ++i) {
      mbar_init(&r_full[i], 1);
      mbar_init(&r_free[i], 1);
    }
    if (kRT) prefetch_tmap(&tmO.resid);
    fence_mbar_init();
  }
  if (warp == kPAllocWarp) {
    tmem_alloc_pair(tmem_ptr, 512);
  }
  for (int i = threadIdx.x; i < 64; i += kPThreads) {
    sScale[i] = (i < p.N) ? (p.scale ? p.scale[i] : 1.0f) : 0.0f;
    sBias[i] = (i < p.N && p.bias) ? p.bias[i] : 0.0f;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync();              // barriers of both CTAs are initialised before any remote arrive / TMA signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  if (warp != kPAllocWarp) pdl_wait();
  pdl_launch_dependents();

  // tile (quad s, stream i) of this CTA: tiles are numbered quad-major, then stream, then CTA rank
  auto tile_of = [&](int s, int i) { return (s * nstr + i) * 2 + (int)rank; };

  if (warp == kPProducerWarp) {
    // ------------------------------------------------------------------ activation producer (both CTAs, own tiles)
    int as[kPI] = {0, 0};
    uint32_t aph[kPI] = {0, 0};
    const uint32_t a_tx = (uint32_t)(kPPitch * (hp.TH + 2) * 128);
    for (int s = pair; s < hp.n_quads; s += npairs) {
      int cx[kPI], cy[kPI], cn[kPI];
#pragma unroll
      for (int i = 0; i < kPI; ++i) {
        const int mt = tile_of(s, i);   // (unused for i >= streams)
        const int t1 = hp.d_tx.div(mt), t2 = hp.d_ty.div(t1);
        cx[i] = (mt - t1 * p.tiles_x) * 8;
        cy[i] = (t1 - t2 * p.tiles_y) * hp.TH;
        cn[i] = t2;                 // >= B past the last tile: TMA zero-fills
      }
      for (int kc = 0; kc < p.kchunks; ++kc) {
#pragma unroll
        for (int i = 0; i < kPI; ++i) {
          if (i >= nstr) continue;
          const int slot = i * hp.sa + as[i];
          mbar_wait(&a_empty[slot], aph[i] ^ 1);
          if (elect_one_sync()) {
            if (rank == 0) mbar_arrive_expect_tx(&a_full[slot], 2 * a_tx);
            tma_load_4d_pair(sA + slot * hp.a_stage_bytes, &tmA, leader_addr(&a_full[slot]), kc * 64, cx[i] - 1, cy[i] - 1, cn[i]);
          }
          __syncwarp();
          if (++as[i] == hp.sa) {
            as[i] = 0;
            aph[i] ^= 1;
          }
        }
      }
    }
  } else if (warp == kPAllocWarp) {
    // ------------------------------------------------------------------ weights: this CTA's 32 rows of every (chunk, tap) tile
    if (elect_one_sync()) {
      if (rank == 0) mbar_arrive_expect_tx(b_full, (uint32_t)(2 * nb_tiles * kBTile));
      const uint32_t bar = leader_addr(b_full);
      for (int kc = 0; kc < p.kchunks; ++kc)
        for (int tap = 0; tap < 9; ++tap)
          tma_load_2d_pair(sB + (kc * 9 + tap) * kBTile, &tmB, bar, (tap * p.kchunks + kc) * 64, (int)rank * 32);
    }
    __syncwarp();
    if constexpr (kRT) {
      // residual producer: this CTA's tile sequence, one tile ahead of the epilogue (the residual is an activation
      // written by an earlier kernel of the stream); plain loads into this CTA's staging buffers and barriers
      pdl_wait();
      const uint32_t r_tx = (uint32_t)(8 * hp.TH * 128);
      int rb[kPI] = {0, 0};
      uint32_t rph[kPI] = {0, 0};
      for (int s = pair; s < hp.n_quads; s += npairs) {
#pragma unroll
        for (int i = 0; i < kPI; ++i) {
          if (i >= nstr) continue;
          const int mt = tile_of(s, i);
          const int t1 = hp.d_tx.div(mt), t2 = hp.d_ty.div(t1);
          const int x0 = (mt - t1 * p.tiles_x) * 8, y0 = (t1 - t2 * p.tiles_y) * hp.TH;
          mbar_wait(&r_free[i * 2 + rb[i]], rph[i] ^ 1);
          if (elect_one_sync()) {
            mbar_arrive_expect_tx(&r_full[i * 2 + rb[i]], r_tx);
            tma_load_4d(sO + (i * p.obufs + rb[i]) * kABytesPerStage, &tmO.resid, &r_full[i * 2 + rb[i]], 0, x0, y0, t2);
          }
          __syncwarp();
          if (++rb[i] == 2) {
            rb[i] = 0;
            rph[i] ^= 1;
          }
        }
      }
    }
  } else if (warp >= kPIssuerWarp0) {
    // ------------------------------------------------------------------ MMA issuers (leader CTA only)
    const int iw = warp - kPIssuerWarp0;
    if (rank == 0 && iw / kPKS < nstr) {
      const int i = iw / kPKS, h = iw - i * kPKS;
      const uint32_t idesc = umma_idesc_bf16(256, 64);
      int as = 0, acc = 0;
      uint32_t aph = 0, acc_phase = 0;
      mbar_wait(b_full, 0);
      tc_fence_after();
      const uint32_t sB_u32 = smem_u32(sB);
      for (int s = pair; s < hp.n_quads; s += npairs) {
        mbar_wait(&acc_empty[i * kPAcc + acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + ((i * kPAcc + acc) * kPKS + h) * 64;
        for (int kc = 0; kc < p.kchunks; ++kc) {
          mbar_wait(&a_full[i * hp.sa + as], aph);
          tc_fence_after();
          const uint64_t ad0 = umma_desc_sw128_sbo(smem_u32(sA + (i * hp.sa + as) * hp.a_stage_bytes), kPPitch * 128);
#pragma unroll 3
          for (int tap = 0; tap < 9; ++tap) {
            const int item = kc * 9 + tap;
            if ((item % kPKS) != h) continue;
            const int r = tap / 3, sx = tap - r * 3;
            const uint64_t ad = ad0 + (uint64_t)((r * kPPitch + sx) * 8);
            const uint64_t bd = umma_desc_sw128(sB_u32 + item * kBTile);
            const uint32_t first = item >= kPKS ? 1u : 0u;
            if (elect_one_sync()) {
              umma_bf16_pair(d_tmem, ad, bd, idesc, first);
              umma_bf16_pair(d_tmem, ad + 2, bd + 2, idesc, 1u);
              umma_bf16_pair(d_tmem, ad + 4, bd + 4, idesc, 1u);
              umma_bf16_pair(d_tmem, ad + 6, bd + 6, idesc, 1u);
            }
            __syncwarp();
          }
          if (elect_one_sync()) umma_commit_pair(&a_empty[i * hp.sa + as]);
          __syncwarp();
          if (++as == hp.sa) {
            as = 0;
            aph ^= 1;
          }
        }
        if (elect_one_sync()) umma_commit_pair(&acc_full[i * kPAcc + acc]);
        __syncwarp();
        if (++acc == kPAcc) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (both CTAs, own tiles)
    const int i = warp >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int etid = threadIdx.x - i * 128;
    const int tx = row & 7, ty = row >> 3;
    const bool row_in_tile = ty < hp.TH;
    uint8_t* sOi = sO + i * p.obufs * obuf_bytes;
    int acc = 0, obuf = 0;
    uint32_t acc_phase = 0;
    uint32_t r_uses = 0;   // kRT: tiles processed so far by this group (buffer = r_uses & 1, phase = (r_uses >> 1) & 1)
    for (int s = pair; s < (i < nstr ? hp.n_quads : 0); s += npairs) {
      const int mt = tile_of(s, i);
      const int t1 = hp.d_tx.div(mt), t2 = hp.d_ty.div(t1);
      const int x0 = (mt - t1 * p.tiles_x) * 8;
      const int y0 = (t1 - t2 * p.tiles_y) * hp.TH;
      const int n = t2;
      const int x = x0 + tx, y = y0 + ty;
      const bool valid = row_in_tile && (x < p.W) && (y < p.H) && (n < p.B);
      if (kMode == UG_EPI_GATE && etid < p.N && n < p.B) sGate[i * 64 + etid] = 1.0f + __ldg(p.gate + (long long)n * p.N + etid);
      mbar_wait(&acc_full[i * kPAcc + acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (i * kPAcc + acc) * kPKS * 64;
      float dot = 0.0f;
      uint32_t v[16], v2[16];
      __syncwarp();
      tmem_ld16(taddr, v);
      tmem_ld16(taddr + 64, v2);
      if (p.tma_store) {
        // staging buffer `obuf` must no longer be read by the TMA store issued obufs tiles ago
        // (the barrier also publishes sGate of this tile)
        if constexpr (kRT) {
          // the store of the previous tile (other buffer) has finished reading: hand that buffer to the residual
          // producer for the NEXT tile, then wait for this tile's residual (loaded one tile ago)
          if (etid == 0 && r_uses > 0) {
            bulk_wait_group_read<0>();
            mbar_arrive(&r_free[i * 2 + (obuf ^ 1)]);
          }
          mbar_wait(&r_full[i * 2 + obuf], (r_uses >> 1) & 1);
          ++r_uses;
        } else if (etid == 0) {
          if (p.obufs == 2) bulk_wait_group_read<1>();
          else bulk_wait_group_read<0>();
        }
        named_bar_sync(1 + i, 128);
      }
      uint8_t* so_row = sOi + obuf * obuf_bytes + row * 128;
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int c0 = cc * 16;
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(v2[j]));
        float f[16];
        epi_math16_linear<UG_ACT_RELU>(v, f, sScale, sBias, c0);   // ReLU deferred (see conv_common.cuh)
        __syncwarp();
        if (cc < 3) {
          tmem_ld16(taddr + c0 + 16, v);
          tmem_ld16(taddr + 64 + c0 + 16, v2);
        }
        if constexpr (kMode == UG_EPI_OUTC) {
          epi_relu16<UG_ACT_RELU>(f);
          const float4* ow = reinterpret_cast<const float4*>(p.outc_w + c0);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 w4 = __ldg(ow + j);
            dot += f[4 * j] * w4.x + f[4 * j + 1] * w4.y + f[4 * j + 2] * w4.z + f[4 * j + 3] * w4.w;
          }
        } else {
        if constexpr (kMode == UG_EPI_GATE) {   // e1 + d * (1 + g): the residual pieces sit where the result will be written
          epi_relu16<UG_ACT_RELU>(f);
          const uint4 a0 = *reinterpret_cast<const uint4*>(so_row + (((cc * 2) ^ (row & 7)) << 4));
          const uint4 a1 = *reinterpret_cast<const uint4*>(so_row + (((cc * 2 + 1) ^ (row & 7)) << 4));
          const float4* gp = reinterpret_cast<const float4*>(sGate + i * 64 + c0);
          epi_gate8(f, a0, gp[0], gp[1]);
          epi_gate8(f + 8, a1, gp[2], gp[3]);
        }
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          uint4 o;
          if constexpr (kMode == UG_EPI_GATE) {   // the combined value may be negative: plain conversion
            o.x = pack_bf16x2(f[g * 8 + 0], f[g * 8 + 1]);
            o.y = pack_bf16x2(f[g * 8 + 2], f[g * 8 + 3]);
            o.z = pack_bf16x2(f[g * 8 + 4], f[g * 8 + 5]);
            o.w = pack_bf16x2(f[g * 8 + 6], f[g * 8 + 7]);
          } else {
            o.x = pack_bf16x2_relu(f[g * 8 + 0], f[g * 8 + 1]);
            o.y = pack_bf16x2_relu(f[g * 8 + 2], f[g * 8 + 3]);
            o.z = pack_bf16x2_relu(f[g * 8 + 4], f[g * 8 + 5]);
            o.w = pack_bf16x2_relu(f[g * 8 + 6], f[g * 8 + 7]);
          }
          const int chunk = cc * 2 + g;
          *reinterpret_cast<uint4*>(so_row + ((chunk ^ (row & 7)) << 4)) = o;
          if (p.pool) {
            // fused nn.MaxPool2d(2): the 2x2 window of pixel (tx, ty) lives in lanes ^1 (x) and ^8 (y) of this warp
            uint4 m = o;
            m.x = bf16x2_max(m.x, __shfl_xor_sync(0xffffffffu, m.x, 1));
            m.y = bf16x2_max(m.y, __shfl_xor_sync(0xffffffffu, m.y, 1));
            m.z = bf16x2_max(m.z, __shfl_xor_sync(0xffffffffu, m.z, 1));
            m.w = bf16x2_max(m.w, __shfl_xor_sync(0xffffffffu, m.w, 1));
            m.x = bf16x2_max(m.x, __shfl_xor_sync(0xffffffffu, m.x, 8));
            m.y = bf16x2_max(m.y, __shfl_xor_sync(0xffffffffu, m.y, 8));
            m.z = bf16x2_max(m.z, __shfl_xor_sync(0xffffffffu, m.z, 8));
            m.w = bf16x2_max(m.w, __shfl_xor_sync(0xffffffffu, m.w, 8));
            if (((tx | ty) & 1) == 0) {
              const int pr = (ty >> 1) * 4 + (tx >> 1);
              *reinterpret_cast<uint4*>(sP + (i * p.obufs + obuf) * kPPoolBytes + pr * 128 + ((chunk ^ (pr & 7)) << 4)) = m;
            }
          }
        }
        }
      }
      // all TMEM reads of this accumulator are done: hand it back to the leader's issuers
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rank == 0) mbar_arrive(&acc_empty[i * kPAcc + acc]);
        else mbar_arrive_cluster(leader_addr(&acc_empty[i * kPAcc + acc]));
      }
      if constexpr (kMode == UG_EPI_OUTC) {
        if (valid) {
          const float logit = dot + p.outc_b;
          const long long o = ((long long)n * p.H + y) * p.W + x;
          p.logits[o] = logit;
          const float sg = 1.0f / (1.0f + expf(-logit));  // torch.sigmoid(seg_out) > 0.5 in fp32
          p.mask[o] = sg > 0.5f ? 1 : 0;
        }
      } else {
        fence_proxy_async_smem();
        named_bar_sync(1 + i, 128);
        if (etid == 0) {
          tma_store_4d(&tmO.out, sOi + obuf * obuf_bytes, 0, x0, y0, n);
          if (p.pool) tma_store_4d(&tmO.pool, sP + (i * p.obufs + obuf) * kPPoolBytes, 0, x0 >> 1, y0 >> 1, n);
          bulk_commit_group();
        }
        if (p.obufs == 2) obuf ^= 1;
      }
      if (++acc == kPAcc) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (p.tma_store && etid == 0) bulk_wait_group_all();
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync();  // the peer's accumulators are still written by MMAs issued from the leader until both are done
  if (warp == kPAllocWarp) tmem_dealloc_pair(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------ host side

// The instantiated (epilogue mode, TMA residual) forms (UG_PAIR_INSTANCES, engine.h).
struct PairInstance {
  int mode, rt;
  PairKernelFn fn;
};
#define UG_PAIR_CASE(M, RT) {M, RT, conv_pair_kernel<M, RT>},
static const PairInstance kPairInstances[] = {UG_PAIR_INSTANCES(UG_PAIR_CASE)};
#undef UG_PAIR_CASE

// Fills L for the CTA-pair kernel.  UG_EUNSUPPORTED when the layer is not one it takes (the caller falls back to
// conv_multi_prepare): 3x3 pad 1, ReLU, <= 64 output channels in one 64-column n-tile, STORE (optionally with the fused
// 2x2 pool), OUTC or GATE epilogue, weights resident at 36 KB per 64 input channels per CTA, an even number of SMs.
int conv_pair_prepare(ug_engine* h, const ug_conv_desc* d, ConvLaunch* L) {
  if (!get_encode_fn()) return set_error(h, UG_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
  if (!(d->R == 3 && d->S == 3 && d->pad == 1 && d->up != 2) || d->act != UG_ACT_RELU || d->N > 64 || d->N % 8 ||
      !(d->mode == UG_EPI_STORE || d->mode == UG_EPI_OUTC || d->mode == UG_EPI_GATE) || d->stats_sum || d->out2 ||
      d->in_rstride || d->in_bstride || (h->num_sms & 1))
    return set_error(h, UG_EUNSUPPORTED, "conv(pair): 3x3 ReLU layers with <= 64 output channels, STORE / OUTC / GATE epilogue");
  const int gate = d->mode == UG_EPI_GATE;
  if (gate && (!d->add || !d->gate || d->add_bstride <= 0 || d->add_cstride % 8 || (reinterpret_cast<uintptr_t>(d->add) & 15) ||
               d->pool_out))
    return set_error(h, UG_EUNSUPPORTED, "conv(pair): the GATE epilogue needs a per-image residual tensor (16-byte aligned rows)");
  const int cin_pad = ceil_div(d->Cin, 64) * 64;
  const int kchunks = cin_pad / 64;
  const long long ktot = 9LL * cin_pad;
  const int tma_store = d->mode != UG_EPI_OUTC;
  const int pool = d->pool_out != nullptr;
  const long long resB = 9LL * kchunks * 32 * 128;
  const int obuf_unit = tma_store ? kABytesPerStage + (pool ? kPPoolBytes : 0) : 0;
  const long long fixed = 1024 + 3 * 64 * sizeof(float) + 64 * sizeof(float) + 8 * (2 * kPI * 3 + 1 + 2 * kPI * kPAcc + 4 * kPI) + 16;
  // shared-memory plan, first fit: two tile streams with two activation stages each; else ONE stream with up to three
  // stages (resident weights of 192 / 256 input channels).  GATE needs both staging buffers (residual one tile ahead).
  const int TH = ceil_div(d->H, ceil_div(d->H, 16));
  const int a_stage = ((kPPitch * (TH + 2) * 128 + 1023) / 1024) * 1024;
  static const int cand[6][3] = {{2, 2, 2}, {2, 2, 1}, {1, 3, 2}, {1, 3, 1}, {1, 2, 2}, {1, 2, 1}};   // streams, stages, staging buffers
  int streams = 0, sa = 0, obufs = 0;
  long long smem = 0;
  for (int c = 0; c < 6; ++c) {
    const int ob = tma_store ? cand[c][2] : 0;
    if (gate && ob != 2) continue;
    if (!tma_store && cand[c][2] != 2) continue;   // (OUTC has no staging buffers: one candidate per shape)
    const long long need = fixed + cand[c][0] * cand[c][1] * (long long)a_stage + resB + cand[c][0] * ob * (long long)obuf_unit;
    if (need <= 227LL * 1024) {
      streams = cand[c][0]; sa = cand[c][1]; obufs = ob; smem = need;
      break;
    }
  }
  if (!streams) return set_error(h, UG_EUNSUPPORTED, "conv(pair): weights of %d input channels do not fit", d->Cin);
  if (pool && (!tma_store || (d->H & 1) || (d->W & 1) || (TH & 1) || d->pool_cstride % 8 || (reinterpret_cast<uintptr_t>(d->pool_out) & 15)))
    return set_error(h, UG_EUNSUPPORTED, "conv(pair): fused max-pool needs a STORE conv on an even map");

  ConvKParams& p = L->p;
  memset(&p, 0, sizeof(p));
  p.H = d->H; p.W = d->W; p.B = d->B;
  p.TW = 8; p.TH = TH; p.TN = 1;
  p.tiles_x = ceil_div(d->W, 8);
  p.tiles_y = ceil_div(d->H, TH);
  p.R = 3; p.S = 3; p.pad = 1;
  p.kchunks = kchunks; p.num_k = 9 * kchunks;
  p.N = d->N; p.BN = 64; p.stages = sa; p.tmem_cols = 512;
  p.scale = d->scale; p.bias = d->bias;
  p.act = d->act; p.mode = d->mode;
  p.out = d->out; p.out_cstride = d->out_cstride;
  p.up = 1; p.OH = d->H; p.OW = d->W;
  p.outc_w = d->outc_w; p.outc_b = d->outc_b; p.logits = d->logits; p.mask = d->mask;
  p.add = d->add; p.add_bstride = d->add_bstride; p.add_cstride = d->add_cstride; p.gate = d->gate;
  p.m_tiles = p.tiles_x * p.tiles_y * d->B; p.n_tiles = 1; p.acc_stages = kPAcc;
  p.tma_store = tma_store; p.obufs = obufs; p.npad = 64; p.pool = pool;
  PairParams& hp = L->pp;
  memset(&hp, 0, sizeof(hp));
  hp.TH = TH; hp.a_stage_bytes = a_stage; hp.sa = sa;
  hp.n_quads = ceil_div(p.m_tiles, 2 * streams);   // tile groups: streams x 2 CTAs
  hp.streams = streams;
  hp.d_tx = make_fastdiv(p.tiles_x);
  hp.d_ty = make_fastdiv(p.tiles_y);
  L->kernel = ConvKernel::Pair;
  L->pair_fn = nullptr;
  for (int i = 0; i < (int)(sizeof(kPairInstances) / sizeof(kPairInstances[0])); ++i)
    if (kPairInstances[i].mode == d->mode) {
      L->pair_fn = kPairInstances[i].fn;
      L->instance = i;
    }
  L->item_tiles = 2 * streams;
  L->block = kPThreads;

  {
    cuuint64_t dims[4] = {(cuuint64_t)d->Cin, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->in_cstride * 2, (cuuint64_t)d->W * d->in_cstride * 2,
                             (cuuint64_t)d->H * d->W * d->in_cstride * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)kPPitch, (cuuint32_t)(TH + 2), 1};
    const int r = encode_bf16_sw128(&L->tmA, d->in, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
    if (r) return set_error(h, UG_ECUDA, "conv(pair): activation tensor map encode failed (%d)", r);
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)d->N};   // rows beyond N are zero-filled
    cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
    cuuint32_t box[2] = {64, 32};
    const int r = encode_bf16_sw128(&L->tmB, d->w, 2, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
    if (r) return set_error(h, UG_ECUDA, "conv(pair): weight tensor map encode failed (%d)", r);
  }
  memset(&L->pmaps, 0, sizeof(L->pmaps));
  if (gate) {  // load map of the residual tensor, same box as the output store
    cuuint64_t dims[4] = {(cuuint64_t)d->N, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->add_cstride * 2, (cuuint64_t)d->W * d->add_cstride * 2, (cuuint64_t)d->add_bstride * 2};
    cuuint32_t box[4] = {64, 8, (cuuint32_t)TH, 1};
    const int r = encode_bf16_sw128(&L->pmaps.resid, d->add, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
    if (r) return set_error(h, UG_ECUDA, "conv(pair): residual tensor map encode failed (%d)", r);
  }
  if (tma_store) {
    cuuint32_t box[4] = {64, 8, (cuuint32_t)TH, 1};
    cuuint64_t dims[4] = {(cuuint64_t)d->N, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->out_cstride * 2, (cuuint64_t)d->W * d->out_cstride * 2,
                             (cuuint64_t)d->H * d->W * d->out_cstride * 2};
    const int r = encode_bf16_sw128(&L->pmaps.out, d->out, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_NONE);
    if (r) return set_error(h, UG_ECUDA, "conv(pair): output tensor map encode failed (%d)", r);
    if (pool) {
      const long long pcs = d->pool_cstride;
      cuuint64_t pdims[4] = {(cuuint64_t)d->N, (cuuint64_t)(d->W / 2), (cuuint64_t)(d->H / 2), (cuuint64_t)d->B};
      cuuint64_t pstrides[3] = {(cuuint64_t)(pcs * 2), (cuuint64_t)((d->W / 2) * pcs * 2),
                                (cuuint64_t)((long long)(d->H / 2) * (d->W / 2) * pcs * 2)};
      cuuint32_t pbox[4] = {64, 4, (cuuint32_t)(TH / 2), 1};
      const int rp = encode_bf16_sw128(&L->pmaps.pool, d->pool_out, 4, pdims, pstrides, pbox, CU_TENSOR_MAP_L2_PROMOTION_NONE);
      if (rp) return set_error(h, UG_ECUDA, "conv(pair): pooled output tensor map encode failed (%d)", rp);
    }
  }
  const int pairs = std::min(hp.n_quads, h->num_sms / 2);
  L->grid = dim3((unsigned)(2 * pairs), 1, 1);
  L->smem = (size_t)smem;
  return UG_OK;
}

int max_cluster_pairs(ug_engine* h) {
  if (h->max_pairs >= 0) return h->max_pairs;
  int pairs = h->num_sms / 2;
  cudaError_t e = cudaFuncSetAttribute((const void*)conv_pair_kernel<UG_EPI_STORE, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e == cudaSuccess) {
    cudaLaunchAttribute at[2];
    cudaLaunchConfig_t cfg = pair_config(at, 2 * (h->num_sms / 2), kPThreads, 200 * 1024, 0);
    cfg.numAttrs = 1;   // (the cluster shape only)
    int n = 0;
    e = cudaOccupancyMaxActiveClusters(&n, (const void*)conv_pair_kernel<UG_EPI_STORE, 0>, &cfg);
    if (e == cudaSuccess && n > 0) pairs = std::min(pairs, n);
  }
  if (e != cudaSuccess) cudaGetLastError();   // (the query is advisory: fall back to num_sms / 2)
  if (getenv("UG_VERBOSE")) fprintf(stderr, "ugnet: %d co-resident CTA pairs on %d SMs\n", pairs, h->num_sms);
  h->max_pairs = pairs;
  return pairs;
}

int conv_pair_launch(ug_engine* h, const ConvLaunch* L, cudaStream_t s) {
  if (!h->attr_pair) {
    for (const PairInstance& k : kPairInstances) {
      const cudaError_t e = cudaFuncSetAttribute((const void*)k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(conv_pair_kernel)");
    }
    h->attr_pair = true;
  }
  const cudaError_t e = launch_pairs(h, L->pair_fn, L->grid.x, L->block, L->smem, s, L->tmA, L->tmB, L->pmaps, L->p, L->pp);
  h->launches++;
  return check_cuda(h, e != cudaSuccess ? e : cudaGetLastError(), "conv_pair_kernel launch");
}

}  // namespace ug
