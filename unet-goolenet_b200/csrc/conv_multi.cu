// 3x3 convolution (stride 1, pad 1), one persistent CTA per SM with TWO MMA-issuing warps sharing the weights.
//
// Activation tiles: an 8 x TH block of output pixels (TH <= 16, 128 MMA rows) plus a one-pixel border is fetched
// ONCE per 64-channel chunk as a TMA box {64 ch, 10 px, TH+2 rows} (out-of-bounds coordinates are zero-filled =
// the conv padding); halo pixel (hy, hx) sits at smem row hy*10 + hx (128 B per row, SWIZZLE_128B).  For filter tap
// (r, s) the MMA row group g (= output row g of the tile) starts at ((g + r)*10 + s) * 128 B: stride-byte-offset
// 1280 and a start address that is only 128-byte aligned.  The 128B swizzle of tcgen05 operands is a function of
// the absolute shared-memory address (profiles/r01_halo_descriptor_probe.txt), so descriptors keep base_offset 0.
//
// Why two issuers: one thread's chain of M=128 tcgen05.mma instructions retires one MMA per ~110 cycles for any
// N <= 128; two issuing warps of ONE CTA interleave exactly like two co-resident CTAs (N=64: 63 cycles per MMA per
// SM, N=128: 72; profiles/r01_mma_multi_issuer.txt) but can share one copy of the weights:
//   * weights that fit (9*Cin_pad*BN*2 bytes, e.g. 72 KB for 64->64) stay RESIDENT in shared memory for the launch;
//   * otherwise every streamed weight tile is consumed by both issuers (each for its own pixel tile) before its
//     slot is released, which halves the weight traffic per FLOP (an effective 256 x BN CTA tile).
// Row-strip tiles (hp.strip, maps 28 pixels wide): 8-pixel-wide tiles cover a 28-wide row with 3.5 tile columns, so
// only 76.6 % of the MMA rows were output pixels.  In strip mode a tile is SR = 4 FULL image rows: the TMA box is
// {64 ch, W+2 px, SR+2 rows}, the MMA rows are the FLATTENED halo positions m = j*(W+2) + x (8-row groups contiguous:
// SBO 1024), tap (r, s) starts (r*(W+2) + s) pixels into the stage, and rows with x >= W (two per image row) plus the
// tail m >= SR*(W+2) are computed but never stored: 112 of 128 rows useful (87.5 %), 7 tiles per image instead of 8.
// The epilogue compacts its rows to the [SR][W] layout of the TMA store box; the fused 2x2 max-pool reads the staged
// tile instead of exchanging registers (row neighbours are W+2 lanes apart).
//
// TMA residual (kRT = 1, CoordAtt3 combine on 64-channel layers): the GATE epilogue adds the e1 tile.  Read by the
// epilogue threads themselves (16 bytes per lane at a 128-byte lane stride, eight times per tile) those loads were a
// fifth of the layer (0.348 -> 0.276 ms at 224x224 without them).  With kRT the otherwise idle weight-producer warp
// TMA-loads the residual tile of the NEXT sub-tile straight into the other output staging buffer (same box and swizzle
// as the store); the epilogue combines IN PLACE — every (row, 16-byte chunk) is read and rewritten by exactly one
// thread — and hands the buffer back (r_free) once the TMA store that followed has finished reading it.
//
// The issue loops are warp-uniform with the asynchronous instructions under elect_one_sync() (see common.cuh):
// with `if (lane == 0)` loops the issuing thread needed ~16 SASS instructions per MMA and bounded every N <= 128
// layer (224x224 64->64: 0.375 ms before, 0.236 ms after; profiles/r01_conv_sweep_multi_issuer.txt).
//
// Each issuer i owns a pixel-tile stream, a ring of activation stages, TMEM accumulators and a warpgroup of four
// epilogue warps (folded BN/bias + activation, residual / CoordAtt3 combine / outc epilogues, bf16 tile staged in
// swizzled smem and written with TMA stores).  Warp roles: warps 0-3 / 4-7 epilogue of tile stream 0 / 1,
// warp 8 TMEM allocator + weight producer, warp 9 activation producer, warps 10.. MMA issuers.
//
// K-split (kKS = 2, narrow tiles BN <= 64): the 36 (or 72) MMAs of a tile form ONE dependent chain on its accumulator
// and a chain retires an MMA only every ~110 cycles whatever N is (profiles/r01_mma_multi_issuer.txt), so two chains
// per SM left the N = 64 layers at 63 cycles per MMA against a shared-memory operand floor of 48.  With kKS = 2 every
// tile stream has TWO issuing warps that take alternate (chunk, tap) items of the same tile into their OWN TMEM
// accumulators (four independent chains per SM); the epilogue adds the two partial sums in fp32 while it reads them.
// The epilogue mode is a template parameter as well: its branches on ADD / GATE / OUTC were a third of the
// instructions of the chunk loop of a plain-store layer.
//
// CTA pairs (kPair = 1, 128-column n-tiles with streamed weights): the issuers of these layers waited for weight tiles
// 18 % of their time (profiles/r02_pair128.txt) — every CTA streams the whole weight matrix from L2 once per two pixel
// tiles, ~2 GB per layer and ~7.5 TB/s of L2 -> SM traffic at 128 images.  A cluster of two CTAs runs
// tcgen05.mma.cta_group::2 (M = 256 over both SMs): each CTA loads only HALF of the rows of every weight tile (the
// tensor cores exchange them), so the weight traffic per SM halves and the ring holds twice as many tiles.  Protocol as
// in conv_pair.cu: only the leader CTA issues; its a_full / b_full barriers collect the TMA bytes of both CTAs;
// tcgen05.commit multicasts to the a_empty / b_empty / acc_full barriers of both; the peer's epilogue warps return
// accumulators with remote arrives on the leader's acc_empty; pixel tiles past the end are zero-filled / clipped by TMA
// so that both CTAs run the same number of rounds.  With kRT the CoordAtt3 combine of a pair kernel gets its residual
// sub-tiles by TMA too: the weight warp is busy streaming, so ONE EXTRA WARP (warp 12, 416 threads) produces them.
#include <cfloat>
#include <cstring>
#include <algorithm>
#include "conv_common.cuh"

namespace ug {

static constexpr int kEpiUnroll = 1;   // unroll factor of the epilogue chunk loop (see there)
static constexpr int kMI = 2;           // tile streams per CTA (each with its own epilogue warpgroup)
// threads per CTA: 384 (kKS = 1) / 448 (kKS = 2); + one warp (residual producer) for the TMA-residual pair kernels, whose
// weight warp is busy streaming
__host__ __device__ constexpr int kMultiThreads(int ks, int extra = 0) { return 32 * (4 * kMI + 2 + kMI * ks + extra); }
static constexpr int kMPitch = 10;      // halo tile pitch of 8-pixel-wide tiles: 8 output pixels + one border pixel on each side
// Warp roles.  The warp scheduler prefers the highest warp id among eligible warps, and the MMA issuers are the
// latency-critical warps (every late tcgen05.mma is a tensor-pipe bubble), so they get the highest ids, then the
// TMA producer; the epilogue warps (which have plenty of slack but dense instruction streams) get the lowest.
// Measured on the 224x224 64->64 layer: issuers at warps 1-2 below a tightened epilogue: 0.29 ms, here: see
// profiles/r01_conv_sweep_multi_issuer.txt.
static constexpr int kMAllocWarp = 4 * kMI;          // 8: TMEM allocator + weight (B) producer
static constexpr int kMProducerWarp = 4 * kMI + 1;   // 9: activation (A) producer
static constexpr int kMIssuerWarp0 = 4 * kMI + 2;    // 10 ..: issuer of (stream i, K-half h) is warp 10 + i*kKS + h

static constexpr int kPoolBytes = 4096;

// tcgen05.mma / commit of one CTA or (kPair) of a CTA pair; pair commits arrive on the barrier at `bar`'s offset in
// BOTH CTAs
template <int kPair>
__device__ __forceinline__ void mp_umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (kPair) umma_bf16_pair(d_tmem, adesc, bdesc, idesc, accumulate);
  else umma_bf16(d_tmem, adesc, bdesc, idesc, accumulate);
}
template <int kPair>
__device__ __forceinline__ void mp_commit(uint64_t* bar) {
  if constexpr (kPair) umma_commit_pair(bar);
  else umma_commit(bar);
}

template <int kAct, int kTaps, int kMode, int kKS, int kRT, int kPair>
__global__ void __launch_bounds__(kMultiThreads(kKS, kRT && kPair), 1) conv_multi_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                           const __grid_constant__ CUtensorMap tmB,
                                                                           const __grid_constant__ StoreMaps tmO,
                                                                           const ConvKParams p, const MultiParams hp) {
  constexpr int kThreadsCta = kMultiThreads(kKS, kRT && kPair);
  constexpr int kResidWarp = kMIssuerWarp0 + kMI * kKS;   // extra warp of the TMA-residual pair kernels
  static_assert(!kPair || kTaps == 9, "CTA pairs: 3x3 halo tiles");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  const int b_tile_bytes = (kPair ? p.BN / 2 : p.BN) * 128;   // pairs: this CTA's half of the rows of a weight tile
  const int obuf_bytes = p.tma_store ? kABytesPerStage : 0;  // one 64-channel sub-tile per staging buffer
  const int nb_tiles = hp.b_resident ? kTaps * p.kchunks : hp.sb;
  uint8_t* sA = smem;                                        // [kMI][sa] activation stages
  uint8_t* sB = sA + kMI * hp.sa * hp.a_stage_bytes;
  uint8_t* sO = sB + nb_tiles * b_tile_bytes;                // [kMI][obufs] output staging
  uint8_t* sP = sO + kMI * p.obufs * obuf_bytes;              // [kMI][obufs] pooled staging (4 KB each) when p.pool
  float* sScale = reinterpret_cast<float*>(sP + (p.pool ? kMI * p.obufs * kPoolBytes : 0));  // 16-byte aligned
  float* sBias = sScale + p.npad;
  float* sGate = sBias + p.npad;                              // [kMI][128]: 1 + gate of the tile's image (GATE epilogue)
  float* sStat = sGate + kMI * 128;                           // [kMI][4 row quarters][64 ch][sum, max] (fused stats)
  uint64_t* a_full = reinterpret_cast<uint64_t*>(sStat + (p.stats_sum ? kMI * 512 : 0));   // [kMI][sa]
  uint64_t* a_empty = a_full + kMI * hp.sa;
  uint64_t* b_full = a_empty + kMI * hp.sa;                  // [sb] (entry 0 only when resident)
  uint64_t* b_empty = b_full + hp.sb;
  uint64_t* acc_full = b_empty + hp.sb;                      // [kMI][acc_stages]
  uint64_t* acc_empty = acc_full + kMI * p.acc_stages;
  uint64_t* r_full = acc_empty + kMI * p.acc_stages;          // [kMI][2] residual tile landed in staging buffer b (kRT)
  uint64_t* r_free = r_full + kMI * 2;                        // [kMI][2] staging buffer b may be overwritten (kRT)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(r_free + kMI * 2);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int total_super = hp.m_super * p.n_tiles;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;                        // CTA of the pair (0 = leader: issues every MMA)
  const int cta0 = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;     // first work item / stride of the persistent loops
  const int ncta = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  // pixel tile of (group ms, stream i): pairs interleave the two CTAs; tiles past the end stay in the loops of a pair
  // (zero-filled loads, clipped stores) so that both CTAs run the same rounds
  auto tile_of = [&](int ms, int i) { return kPair ? (ms * kMI + i) * 2 + (int)rank : ms * kMI + i; };
  auto tile_live = [&](int mt) { return kPair ? true : mt < p.m_tiles; };
  // work item -> (n-tile, pixel-tile group)
  auto decode = [&](int s, int& nt, int& ms) {
    if (hp.m_major) {
      ms = hp.d_nt.div(s);
      nt = s - ms * p.n_tiles;
    } else {
      nt = hp.d_msuper.div(s);
      ms = s - nt * hp.m_super;
    }
  };

  if (warp == kMProducerWarp && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (p.tma_store) {
      prefetch_tmap(&tmO.m[0]);
      if (p.pool) prefetch_tmap(&tmO.m[1]);
      if (p.up == 2) {
        prefetch_tmap(&tmO.m[1]);
        prefetch_tmap(&tmO.m[2]);
        prefetch_tmap(&tmO.m[3]);
      }
    }
    for (int i = 0; i < kMI * hp.sa; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], kKS);  // every issuer of the stream has finished reading the stage
    }
    for (int i = 0; i < hp.sb; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], kMI);  // released once every issuer has consumed (or skipped) the tile
    }
    for (int i = 0; i < kMI * p.acc_stages; ++i) {
      mbar_init(&acc_full[i], kKS);  // every K-half of the tile is complete
      mbar_init(&acc_empty[i], kPair ? 8 : 4);   // the epilogue warps of the stream (of both CTAs of a pair)
    }
    for (int i = 0; i < kMI * 2; ++i) {
      mbar_init(&r_full[i], 1);
      mbar_init(&r_free[i], 1);
    }
    if (kRT) prefetch_tmap(&tmO.m[4]);
    fence_mbar_init();
  }
  if (warp == kMAllocWarp) {
    if constexpr (kPair) {
      tmem_alloc_pair(tmem_ptr, p.tmem_cols);
    } else {
      tmem_alloc(tmem_ptr, p.tmem_cols);
      tmem_relinquish();
    }
  }
  for (int i = threadIdx.x; i < p.npad; i += kThreadsCta) {
    sScale[i] = (i < p.N) ? (p.scale ? p.scale[i] : 1.0f) : 0.0f;
    sBias[i] = (i < p.N && p.bias) ? p.bias[i] : 0.0f;
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) cluster_sync();   // the barriers of both CTAs exist before any remote arrive / TMA signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // Everything above touched only kernel parameters and constant weights; from here on the roles read activations /
  // write outputs, which must wait for the previous kernel of the stream.  The weight producer (kMAllocWarp) streams
  // constants only and starts right away.
  if (warp != kMAllocWarp) pdl_wait();
  pdl_launch_dependents();

  // Residual producer (kRT): the (tile, 64-column sub-tile) sequence of both streams, one sub-tile ahead of the epilogue,
  // TMA-loaded into the free staging buffer; the residual is an activation written by an earlier kernel of the stream.
  auto resid_loop = [&]() {
    const uint32_t r_tx = (uint32_t)(p.TW * p.TH * 128);
    const int obuf_b = kABytesPerStage;
    int rb[kMI] = {0, 0};
    uint32_t rph[kMI] = {0, 0};
    for (int s = cta0; s < total_super; s += ncta) {
      int nt, ms;
      decode(s, nt, ms);
      const int ncols = min(p.BN, p.N - nt * p.BN);
#pragma unroll
      for (int i = 0; i < kMI; ++i) {
        const int mt = tile_of(ms, i);
        if (!tile_live(mt)) continue;
        const int t1 = hp.d_tx.div(mt), t2 = hp.d_ty.div(t1);
        const int x0 = (mt - t1 * p.tiles_x) * p.TW, y0 = (t1 - t2 * p.tiles_y) * p.TH, n0 = t2 * p.TN;
        for (int sub = 0; sub * 64 < ncols; ++sub) {
          mbar_wait(&r_free[i * 2 + rb[i]], rph[i] ^ 1);
          if (elect_one_sync()) {
            mbar_arrive_expect_tx(&r_full[i * 2 + rb[i]], r_tx);
            tma_load_4d(sO + (i * p.obufs + rb[i]) * obuf_b, &tmO.m[4], &r_full[i * 2 + rb[i]], nt * p.BN + sub * 64, x0, y0, n0);
          }
          __syncwarp();
          if (++rb[i] == 2) {
            rb[i] = 0;
            rph[i] ^= 1;
          }
        }
      }
    }
  };

  if (warp == kMProducerWarp) {
    // ------------------------------------------------------------------ activation producer (whole warp, elected lane issues)
    int as[kMI] = {0, 0};
    uint32_t aph[kMI] = {0, 0};
    const uint32_t a_tx = kTaps == 9 ? (uint32_t)(hp.pitch * (hp.TH + 2) * 128) : p.a_bytes;
    for (int s = cta0; s < total_super; s += ncta) {
      int nt, ms;
      decode(s, nt, ms);
      int cx[kMI], cy[kMI], cn[kMI];
#pragma unroll
      for (int i = 0; i < kMI; ++i) {
        const int mt = tile_of(ms, i);
        const int t1 = hp.d_tx.div(mt), t2 = hp.d_ty.div(t1);
        cx[i] = (mt - t1 * p.tiles_x) * p.TW;
        cy[i] = (t1 - t2 * p.tiles_y) * p.TH;
        cn[i] = t2 * p.TN;
      }
      for (int kc = 0; kc < p.kchunks; ++kc) {
#pragma unroll
        for (int i = 0; i < kMI; ++i) {
          if (!tile_live(tile_of(ms, i))) continue;
          if (kTaps == 1 && hp.rowtaps == 2 && kc > 0) continue;   // row halo: the tile's single box was loaded at kc == 0
          const int x0 = cx[i], y0 = cy[i], n = cn[i];
          const int slot = i * hp.sa + as[i];
          mbar_wait(&a_empty[slot], aph[i] ^ 1);
          if (elect_one_sync()) {
            if constexpr (kPair) {   // the leader's barrier collects the bytes of both CTAs' loads
              if (rank == 0) mbar_arrive_expect_tx(&a_full[slot], 2 * a_tx);
              tma_load_4d_pair(sA + slot * hp.a_stage_bytes, &tmA, leader_addr(&a_full[slot]), kc * 64, x0 - 1, y0 - 1, n);
            } else {
              mbar_arrive_expect_tx(&a_full[slot], a_tx);
              if (kTaps == 9) tma_load_4d(sA + slot * hp.a_stage_bytes, &tmA, &a_full[slot], kc * 64, x0 - 1, y0 - 1, n);
              else if (hp.rowtaps) tma_load_4d(sA + slot * hp.a_stage_bytes, &tmA, &a_full[slot], 0, x0, y0 + kc, n);
              else tma_load_4d(sA + slot * hp.a_stage_bytes, &tmA, &a_full[slot], kc * 64, x0, y0, n);
            }
          }
          __syncwarp();
          if (++as[i] == hp.sa) {
            as[i] = 0;
            aph[i] ^= 1;
          }
        }
      }
    }
  } else if (warp == kMAllocWarp) {
    // ------------------------------------------------------------------ weight producer (its own warp: a full weight
    // ring must not delay the activation loads of the next chunk, and vice versa)
    if (hp.b_resident) {
      if (elect_one_sync()) {
        if constexpr (kPair) {
          if (rank == 0) mbar_arrive_expect_tx(&b_full[0], (uint32_t)(2 * kTaps * p.kchunks * b_tile_bytes));
          for (int kc = 0; kc < p.kchunks; ++kc)
            for (int tap = 0; tap < kTaps; ++tap)
              tma_load_2d_pair(sB + (kc * kTaps + tap) * b_tile_bytes, &tmB, &b_full[0],
                               (tap * p.kchunks + kc) * 64, (int)rank * (p.BN / 2));
        } else {
          mbar_arrive_expect_tx(&b_full[0], (uint32_t)(kTaps * p.kchunks * b_tile_bytes));
          for (int kc = 0; kc < p.kchunks; ++kc)
            for (int tap = 0; tap < kTaps; ++tap)
              tma_load_2d(sB + (kc * kTaps + tap) * b_tile_bytes, &tmB, &b_full[0], (tap * p.kchunks + kc) * 64, 0);
        }
      }
      __syncwarp();
      if constexpr (kRT && !kPair) {   // the weight warp is idle from here on: it produces the residual tiles
        pdl_wait();
        resid_loop();
      }
    } else {
      int bs = 0;
      uint32_t bph = 0;
      for (int s = cta0; s < total_super; s += ncta) {
        int nt, ms_unused;
        decode(s, nt, ms_unused);
        for (int kc = 0; kc < p.kchunks; ++kc) {
          // (CTA pairs: rolled.  Fully unrolled, the pair forms grow by ~430 SASS instructions, and this warp shares its
          // SMSP's 6 KB L0 instruction cache with two epilogue warps, DESIGN.md §3.1.  The single-CTA forms were
          // measured fully unrolled.)
#pragma unroll (kPair ? 1 : kTaps)
          for (int tap = 0; tap < kTaps; ++tap) {
            mbar_wait(&b_empty[bs], bph ^ 1);
            if (elect_one_sync()) {
              if constexpr (kPair) {
                if (rank == 0) mbar_arrive_expect_tx(&b_full[bs], (uint32_t)(2 * b_tile_bytes));
                tma_load_2d_pair(sB + bs * b_tile_bytes, &tmB, &b_full[bs], (tap * p.kchunks + kc) * 64,
                                 nt * p.BN + (int)rank * (p.BN / 2));
              } else {
                mbar_arrive_expect_tx(&b_full[bs], (uint32_t)b_tile_bytes);
                tma_load_2d(sB + bs * b_tile_bytes, &tmB, &b_full[bs], (tap * p.kchunks + kc) * 64, nt * p.BN);
              }
            }
            __syncwarp();
            if (++bs == hp.sb) {
              bs = 0;
              bph ^= 1;
            }
          }
        }
      }
    }
  } else if ((kRT && kPair) && warp == kResidWarp) {
    resid_loop();   // (this warp executed pdl_wait above)
  } else if (warp >= kMIssuerWarp0 && rank != 0) {
    // (the peer CTA of a pair issues nothing: the leader's MMAs read both CTAs' shared memory and write both TMEMs)
  } else if (warp >= kMIssuerWarp0) {
    // ------------------------------------------------------------------ MMA issuers (whole warp, one elected lane issues)
    const int iw = warp - kMIssuerWarp0;
    const int i = iw / kKS;       // tile stream
    const int h = iw - i * kKS;   // K-half: this warp issues the (chunk, tap) items whose index is h modulo kKS
    const uint32_t idesc = umma_idesc_bf16(kPair ? 256 : 128, p.BN);
    int as = 0, bs = 0, acc = 0;
    uint32_t aph = 0, bph = 0, acc_phase = 0;
    if (hp.b_resident) {
      mbar_wait(&b_full[0], 0);
      tc_fence_after();
    }
    const uint32_t sB_u32 = smem_u32(sB);
    for (int s = cta0; s < total_super; s += ncta) {
      int nt, ms;
      decode(s, nt, ms);
      const bool valid = tile_live(tile_of(ms, i));
      uint32_t d_tmem = 0;
      if (valid) {
        mbar_wait(&acc_empty[i * p.acc_stages + acc], acc_phase ^ 1);
        tc_fence_after();
        d_tmem = tmem_base + ((i * p.acc_stages + acc) * kKS + h) * p.BN;
      }
      for (int kc = 0; kc < p.kchunks; ++kc) {
        uint64_t ad0 = 0;
        const bool row_halo = kTaps == 1 && hp.rowtaps == 2;
        if (valid) {
          if (!(row_halo && kc > 0)) {
            mbar_wait(&a_full[i * hp.sa + as], aph);
            tc_fence_after();
          }
          ad0 = kTaps == 9 ? umma_desc_sw128_sbo(smem_u32(sA + (i * hp.sa + as) * hp.a_stage_bytes), hp.sbo)
                           : umma_desc_sw128(smem_u32(sA + (i * hp.sa + as) * hp.a_stage_bytes) + (row_halo ? kc * p.TW * 128 : 0));
        }
        // (tap loop unrolled by one filter row only: keeps the issue loop inside the L0 instruction cache)
#pragma unroll 3
        for (int tap = 0; tap < kTaps; ++tap) {
          const int r = tap / 3, sx = tap - r * 3;
          const int item = kc * kTaps + tap;
          const bool mine = kKS == 1 || (item % kKS) == h;
          uint32_t b_addr = 0;
          if (hp.b_resident) {
            b_addr = sB_u32 + (kc * kTaps + tap) * b_tile_bytes;
          } else if (mine) {
            mbar_wait(&b_full[bs], bph);
            tc_fence_after();
            b_addr = sB_u32 + bs * b_tile_bytes;
          }
          if (mine) {
            if (valid) {
              // tap (r, sx): the A rows start (r*pitch + sx) halo pixels (128 B each) into the stage
              const uint64_t ad = ad0 + (uint64_t)((r * hp.pitch + sx) * 8);
              const uint64_t bd = umma_desc_sw128(b_addr);
              const uint32_t first = item >= kKS ? 1u : 0u;   // this issuer's first item of the tile overwrites
              if (elect_one_sync()) {
                mp_umma<kPair>(d_tmem, ad, bd, idesc, first);
                mp_umma<kPair>(d_tmem, ad + 2, bd + 2, idesc, 1u);
                mp_umma<kPair>(d_tmem, ad + 4, bd + 4, idesc, 1u);
                mp_umma<kPair>(d_tmem, ad + 6, bd + 6, idesc, 1u);
                if (!hp.b_resident) mp_commit<kPair>(&b_empty[bs]);
              }
              __syncwarp();
            } else if (!hp.b_resident) {
              // a tile-less stream (odd tile count, last round) still has to hand the slot back
              if (elect_one_sync()) mbar_arrive(&b_empty[bs]);
              __syncwarp();
            }
          }
          if (!hp.b_resident) {
            if (++bs == hp.sb) {
              bs = 0;
              bph ^= 1;
            }
          }
        }
        if (valid && !(row_halo && kc + 1 < p.kchunks)) {   // (row halo: the stage is released after its last tap)
          if (elect_one_sync()) mp_commit<kPair>(&a_empty[i * hp.sa + as]);
          __syncwarp();
          if (++as == hp.sa) {
            as = 0;
            aph ^= 1;
          }
        }
      }
      if (valid) {
        if (elect_one_sync()) mp_commit<kPair>(&acc_full[i * p.acc_stages + acc]);
        __syncwarp();
        if (++acc == p.acc_stages) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp < 4 * kMI) {
    // ------------------------------------------------------------------ epilogue (4 warps per issuer)
    const int i = warp >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int etid = threadIdx.x - i * 128;
    // MMA row -> pixel of the tile.  8-pixel-wide 3x3 tiles: row = ty*8 + tx.  Row-strip 3x3 tiles: row = ty*pitch + tx
    // with tx >= W garbage.  1x1 tiles: row = (tn*TH + ty)*TW + tx.  `srow` is the row of the staged output tile.
    const bool strip = kTaps == 9 && hp.strip;
    const int sty = hp.d_pitch.div(row);
    const int tx = kTaps == 9 ? (strip ? row - sty * hp.pitch : (row & 7)) : row % p.TW;
    const int ty = kTaps == 9 ? (strip ? sty : (row >> 3)) : (row / p.TW) % p.TH;
    const int tn = kTaps == 9 ? 0 : row / (p.TW * p.TH);
    const bool row_in_tile = kTaps == 9 ? (ty < hp.TH && (!strip || tx < p.W)) : (row < p.TW * p.TH * p.TN);
    const int srow = strip ? ty * p.W + tx : row;
    uint8_t* sOi = sO + i * p.obufs * obuf_bytes;
    int acc = 0, obuf = 0;
    uint32_t acc_phase = 0;

    // Residual (ADD / GATE) rows: 16-byte pieces of this thread's own pixel row, prefetched into registers ONE
    // SUB-TILE AHEAD (right after the chunk loop of the previous sub-tile, whose residual registers are dead by
    // then): with the loads issued at the start of the same tile the HBM latency was exposed in the first chunk of
    // every tile of the epilogue-bound 64-channel layers (chunk loop 1000 cycles per chunk instead of 400).
    constexpr bool has_add = (kMode == UG_EPI_ADD || kMode == UG_EPI_GATE) && !kRT;   // register-prefetched residual
    constexpr bool smem_add = (kMode == UG_EPI_ADD || kMode == UG_EPI_GATE) && kRT;   // TMA-loaded residual, in place
    uint32_t r_uses = 0;   // kRT: sub-tiles processed so far by this group (buffer = r_uses & 1, phase = (r_uses >> 1) & 1)
    uint4 addv[8];
    auto prefetch_add = [&](int s2, int sub2) {
      int nt2, ms2;
      decode(s2, nt2, ms2);
      const int mt2 = tile_of(ms2, i);
      const int u1 = hp.d_tx.div(mt2), u2 = hp.d_ty.div(u1);
      const int x2 = (mt2 - u1 * p.tiles_x) * p.TW + tx, y2 = (u1 - u2 * p.tiles_y) * p.TH + ty, n2 = u2 * p.TN + tn;
      const bool v2 = row_in_tile && (x2 < p.W) && (y2 < p.H) && (n2 < p.B);
      const int col2 = nt2 * p.BN + sub2 * 64;
      const __nv_bfloat16* ar = reinterpret_cast<const __nv_bfloat16*>(p.add) + (long long)n2 * p.add_bstride +
                                ((long long)y2 * p.W + x2) * p.add_cstride + col2;
#pragma unroll
      for (int g = 0; g < 8; ++g)
        addv[g] = (v2 && col2 + g * 8 < p.N) ? __ldg(reinterpret_cast<const uint4*>(ar + g * 8)) : make_uint4(0, 0, 0, 0);
    };
    if (has_add) {
      int s0 = cta0;
      auto group_of = [&](int sx) { int a, b; decode(sx, a, b); return b; };
      while (s0 < total_super && !tile_live(tile_of(group_of(s0), i))) s0 += ncta;
      if (s0 < total_super) prefetch_add(s0, 0);
    }

    for (int s = cta0; s < total_super; s += ncta) {
      int nt, ms;
      decode(s, nt, ms);
      const int mt = tile_of(ms, i);
      if (!tile_live(mt)) continue;
      const int t1 = hp.d_tx.div(mt), t2 = hp.d_ty.div(t1);
      const int x0 = (mt - t1 * p.tiles_x) * p.TW;
      const int y0 = (t1 - t2 * p.tiles_y) * p.TH;
      const int n0 = t2 * p.TN;
      const int n = n0 + tn;
      const int ncol0 = nt * p.BN;
      const int x = x0 + tx, y = y0 + ty;
      const bool valid = row_in_tile && (x < p.W) && (y < p.H) && (n < p.B);
      const float* gate_row = p.gate + (long long)n * p.N + ncol0;
      const int ncols = min(p.BN, p.N - ncol0);
      if (kMode == UG_EPI_GATE && etid < ncols && n < p.B) sGate[i * 128 + etid] = 1.0f + __ldg(gate_row + etid);
      mbar_wait(&acc_full[i * p.acc_stages + acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (i * p.acc_stages + acc) * kKS * p.BN;
      float dot = 0.0f;

      uint32_t v[16];
      uint32_t v2[kKS == 2 ? 16 : 1];   // partial sums of the second K-half
      __syncwarp();
      tmem_ld16(taddr, v);
      if constexpr (kKS == 2) tmem_ld16(taddr + p.BN, reinterpret_cast<uint32_t(&)[16]>(v2));
      for (int sub = 0; sub * 64 < ncols; ++sub) {
        if (p.tma_store) {
          // staging buffer `obuf` must no longer be read by the TMA store issued obufs sub-tiles ago
          // (the barrier also publishes sGate of this tile)
          if constexpr (smem_add) {
            // the store of the previous sub-tile (other buffer) has finished reading: hand that buffer to the residual
            // producer for the NEXT sub-tile, then wait for this sub-tile's residual (loaded one sub-tile ago)
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
        uint8_t* so_row = sOi + obuf * obuf_bytes + srow * 128;
        // the chunk loop is not unrolled (kEpiUnroll): the epilogue warps of an SMSP share its 6 KB L0 instruction
        // cache with an MMA issuer / producer warp; with run-time epilogue modes a 4x larger loop body measurably slowed
        // the MMA issue (0.24 -> 0.29 ms), and x2 / x4 unrolling of this loop measured neutral / slower
        // (profiles/r02_epilogue_unroll.txt)
#pragma unroll kEpiUnroll
        for (int cc = 0; cc < 4; ++cc) {
          const int c0 = sub * 64 + cc * 16;
          if (c0 >= ncols) break;
          tmem_ld_wait();
          if constexpr (kKS == 2) {   // the two K-halves of the tile were accumulated separately: add them in fp32
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(v2[j < (kKS == 2 ? 16 : 1) ? j : 0]));
          }
          float f[16];
          epi_math16_linear<kAct>(v, f, sScale, sBias, ncol0 + c0);   // ReLU deferred (see conv_common.cuh)
          __syncwarp();
          if (c0 + 16 < ncols) {
            tmem_ld16(taddr + c0 + 16, v);
            if constexpr (kKS == 2) tmem_ld16(taddr + p.BN + c0 + 16, reinterpret_cast<uint32_t(&)[16]>(v2));
          }
          if (kMode != UG_EPI_STORE) epi_relu16<kAct>(f);  // stores fold the ReLU into the bf16 conversion below
          if (kMode == UG_EPI_OUTC) {
            const float4* ow = reinterpret_cast<const float4*>(p.outc_w + ncol0 + c0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 w4 = __ldg(ow + j);
              dot += f[4 * j] * w4.x + f[4 * j + 1] * w4.y + f[4 * j + 2] * w4.z + f[4 * j + 3] * w4.w;
            }
            continue;
          }
          const int groups = (c0 + 16 <= ncols) ? 2 : 1;
          if constexpr (smem_add) {   // residual pieces of this chunk sit where the result will be written
            const uint4 a0 = *reinterpret_cast<const uint4*>(so_row + (((cc * 2) ^ (srow & 7)) << 4));
            const uint4 a1 = *reinterpret_cast<const uint4*>(so_row + (((cc * 2 + 1) ^ (srow & 7)) << 4));
            if (kMode == UG_EPI_GATE) {
              const float4* gp = reinterpret_cast<const float4*>(sGate + i * 128 + c0);
              epi_gate8(f, a0, gp[0], gp[1]);
              if (groups == 2) epi_gate8(f + 8, a1, gp[2], gp[3]);
            } else {
              epi_add8(f, a0);
              if (groups == 2) epi_add8(f + 8, a1);
            }
          }
          if (has_add) {
            uint4 a0, a1;  // prefetched residual pieces of this chunk (register indices must be compile-time)
            switch (cc) {
              case 0: a0 = addv[0]; a1 = addv[1]; break;
              case 1: a0 = addv[2]; a1 = addv[3]; break;
              case 2: a0 = addv[4]; a1 = addv[5]; break;
              default: a0 = addv[6]; a1 = addv[7]; break;
            }
            if (kMode == UG_EPI_GATE) {
              const float4* gp = reinterpret_cast<const float4*>(sGate + i * 128 + c0);
              epi_gate8(f, a0, gp[0], gp[1]);
              if (groups == 2) epi_gate8(f + 8, a1, gp[2], gp[3]);
            } else {
              epi_add8(f, a0);
              if (groups == 2) epi_add8(f + 8, a1);
            }
          }
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            if (g < groups) {
              uint4 o;
              // (after a residual add / gate the values may be negative again: only the STORE epilogue's ReLU is
              // folded here; for the other modes f is already activated and the relu conversion is an identity on
              // the activation but NOT on the sum, so they use the plain conversion)
              if (kMode == UG_EPI_STORE) {
                o.x = epi_pack2<kAct>(f[g * 8 + 0], f[g * 8 + 1]);
                o.y = epi_pack2<kAct>(f[g * 8 + 2], f[g * 8 + 3]);
                o.z = epi_pack2<kAct>(f[g * 8 + 4], f[g * 8 + 5]);
                o.w = epi_pack2<kAct>(f[g * 8 + 6], f[g * 8 + 7]);
              } else {
                o.x = pack_bf16x2(f[g * 8 + 0], f[g * 8 + 1]);
                o.y = pack_bf16x2(f[g * 8 + 2], f[g * 8 + 3]);
                o.z = pack_bf16x2(f[g * 8 + 4], f[g * 8 + 5]);
                o.w = pack_bf16x2(f[g * 8 + 6], f[g * 8 + 7]);
              }
              const int chunk = cc * 2 + g;
              if (!strip || row_in_tile) *reinterpret_cast<uint4*>(so_row + ((chunk ^ (srow & 7)) << 4)) = o;
              if (p.pool && !strip) {
                // fused nn.MaxPool2d(2): the 2x2 window of pixel (tx, ty) lives in lanes ^1 (x) and ^8 (y) of this
                // warp (row = ty*8 + tx); max of the rounded bf16 values == rounded max (rounding is monotonic)
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
                  const int pr = (ty >> 1) * 4 + (tx >> 1);  // pooled pixel row of the 4 x TH/2 tile
                  *reinterpret_cast<uint4*>(sP + (i * p.obufs + obuf) * kPoolBytes + pr * 128 + ((chunk ^ (pr & 7)) << 4)) = m;
                }
              }
            }
          }
        }
        if (kMode == UG_EPI_OUTC) continue;
        if ((sub + 1) * 64 >= ncols) {  // all TMEM reads of this accumulator are done: hand it back to the MMA issuer
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (kPair && rank != 0) mbar_arrive_cluster(leader_addr(&acc_empty[i * p.acc_stages + acc]));
            else mbar_arrive(&acc_empty[i * p.acc_stages + acc]);
          }
        }
        if (p.pool && strip) {
          // fused nn.MaxPool2d(2) of a row-strip tile: row neighbours are not warp neighbours here, so the 2x2 windows
          // are read back from the staged tile ([TH][W] rows of 128 B) once every thread has written its row
          named_bar_sync(1 + i, 128);
          const uint8_t* sbuf = sOi + obuf * obuf_bytes;
          uint8_t* pbuf = sP + (i * p.obufs + obuf) * kPoolBytes;
          const int pw = p.W >> 1, items = (hp.TH >> 1) * pw * 8;
          for (int it = etid; it < items; it += 128) {
            const int ch = it & 7, pp = it >> 3;       // 16-byte channel chunk, pooled pixel of the tile
            const int py = pp / pw, px = pp - py * pw;
            uint4 m = make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              const int r = (2 * py + (w >> 1)) * p.W + 2 * px + (w & 1);
              const uint4 v4 = *reinterpret_cast<const uint4*>(sbuf + r * 128 + ((ch ^ (r & 7)) << 4));
              if (w == 0) m = v4;
              else {
                m.x = bf16x2_max(m.x, v4.x);
                m.y = bf16x2_max(m.y, v4.y);
                m.z = bf16x2_max(m.z, v4.z);
                m.w = bf16x2_max(m.w, v4.w);
              }
            }
            *reinterpret_cast<uint4*>(pbuf + pp * 128 + ((ch ^ (pp & 7)) << 4)) = m;
          }
        }
        fence_proxy_async_smem();
        // (issued after the proxy fence: the fence waits for outstanding loads, which would expose their latency here)
        if (has_add) {  // residual of the next sub-tile of this group (same tile, or the group's next tile)
          if ((sub + 1) * 64 < ncols) {
            prefetch_add(s, sub + 1);
          } else {
            const int s2 = s + ncta;
            int nt3, ms3;
            decode(s2 < total_super ? s2 : s, nt3, ms3);
            if (s2 < total_super && tile_live(tile_of(ms3, i))) prefetch_add(s2, 0);
          }
        }
        named_bar_sync(1 + i, 128);
        if (etid == 0) {
          const int col = ncol0 + sub * 64;
          if (p.up == 2) {  // ConvTranspose 2x2 s2: column block -> quadrant (dy,dx) map, channel inside the quadrant
            const int qd = col / p.convt_cout;
            tma_store_4d(&tmO.m[qd], sOi + obuf * obuf_bytes, col - qd * p.convt_cout, x0, y0, n0);
          } else {
            tma_store_4d(&tmO.m[0], sOi + obuf * obuf_bytes, col, x0, y0, n0);
            if (p.pool) tma_store_4d(&tmO.m[1], sP + (i * p.obufs + obuf) * kPoolBytes, col, x0 >> 1, y0 >> 1, n0);
          }
          bulk_commit_group();
        }
        if (p.stats_sum) {
          // CoordAtt3 statistics, stage 1: per-channel sum / max of this staged sub-tile (the bf16 values just stored).
          // Thread (channel pair cp, row quarter rq) folds 32 rows of two channels; the four quarters are combined in
          // a fixed order through smem and written as one partial per (image, tile, channel).
          const uint8_t* sbuf = sOi + obuf * obuf_bytes;
          const int cp = etid & 31, rq = etid >> 5;
          const int wvalid = min(8, p.W - x0);
          float s0 = 0.0f, s1 = 0.0f, m0 = -FLT_MAX, m1 = -FLT_MAX;
#pragma unroll 4
          for (int k = 0; k < 32; ++k) {
            const int r = rq * 32 + k;
            if ((r >> 3) >= hp.TH || (r & 7) >= wvalid) continue;
            const uint32_t wv = *reinterpret_cast<const uint32_t*>(sbuf + r * 128 + ((((cp >> 2) ^ (r & 7)) << 4) | ((cp & 3) << 2)));
            const float a = bf16_lo(wv), b = bf16_hi(wv);
            s0 += a;
            s1 += b;
            m0 = fmaxf(m0, a);
            m1 = fmaxf(m1, b);
          }
          *reinterpret_cast<float4*>(sStat + i * 512 + rq * 128 + cp * 4) = make_float4(s0, m0, s1, m1);
          named_bar_sync(1 + i, 128);
          const int nsub = min(64, ncols - sub * 64);
          if (etid < nsub) {
            const float* q0 = sStat + i * 512 + (etid >> 1) * 4 + (etid & 1) * 2;
            const float sum = ((q0[0] + q0[128]) + q0[256]) + q0[384];
            const float mx = fmaxf(fmaxf(q0[1], q0[129]), fmaxf(q0[257], q0[385]));
            const int tiles_pi = p.tiles_x * p.tiles_y;
            const long long o = ((long long)n0 * tiles_pi + (mt - n0 * tiles_pi)) * p.N + ncol0 + sub * 64 + etid;
            p.stats_sum[o] = sum;
            p.stats_max[o] = mx;
          }
        }
        if (p.obufs == 2) obuf ^= 1;
      }
      if (kMode == UG_EPI_OUTC) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kPair && rank != 0) mbar_arrive_cluster(leader_addr(&acc_empty[i * p.acc_stages + acc]));
          else mbar_arrive(&acc_empty[i * p.acc_stages + acc]);
        }
        if (valid) {
          const float logit = dot + p.outc_b;
          const long long o = ((long long)n * p.H + y) * p.W + x;
          p.logits[o] = logit;
          const float sg = 1.0f / (1.0f + expf(-logit));  // torch.sigmoid(seg_out) > 0.5 in fp32
          p.mask[o] = sg > 0.5f ? 1 : 0;
        }
      }
      if (++acc == p.acc_stages) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (p.tma_store && etid == 0) bulk_wait_group_all();
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (kPair) {
    cluster_sync();   // the leader's MMAs write the peer's tensor memory until both CTAs are done
    if (warp == kMAllocWarp) tmem_dealloc_pair(tmem_base, p.tmem_cols);
  } else {
    if (warp == kMAllocWarp) tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------ host side
void choose_tile(int B, int H, int W, int* TW, int* TH, int* TN);  // conv_gemm.cu

// The instantiated (activation, taps, epilogue mode, K-split, TMA residual, CTA pair) combinations (UG_MULTI_INSTANCES,
// engine.h); conv_multi_prepare admits exactly these.
struct MultiInstance {
  int act, taps, mode, ks, rt, pair;
  MultiKernelFn fn;
};
#define UG_MULTI_CASE(A, T, M, K, RT, P) {A, T, M, K, RT, P, conv_multi_kernel<A, T, M, K, RT, P>},
static const MultiInstance kMultiInstances[] = {UG_MULTI_INSTANCES(UG_MULTI_CASE)};
#undef UG_MULTI_CASE

// Fills L for the multi-issuer kernel: 3x3 pad-1 convolutions (halo tiles) and 1x1 convolutions / linear layers /
// ConvTranspose 2x2 s2 (plain pixel tiles).  Returns UG_EUNSUPPORTED when the shape does not fit it.
int conv_multi_prepare(ug_engine* h, const ug_conv_desc* d, int BN, ConvLaunch* L, int pair) {
  if (!get_encode_fn()) return set_error(h, UG_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
  const int up = d->up == 2 ? 2 : 1;
  // row taps (see ug_conv_desc.in_rstride): R x 1 "valid" convolution over an overlapping-window input, one 64-element
  // window per tap: runs as a 1x1 tile whose R k-chunks are the taps
  const int rowtaps = (d->R > 1 && d->S == 1 && d->pad == 0 && up == 1 && d->Cin <= 64) ? 1 : 0;
  const int taps = d->R == 3 && !rowtaps ? 9 : 1;
  if (!((d->R == 3 && d->S == 3 && d->pad == 1 && up == 1) || (d->R == 1 && d->S == 1 && d->pad == 0) || rowtaps))
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): 3x3 pad-1, 1x1, or R x 1 row-tap convolutions only");
  if ((d->in_rstride || d->in_bstride) && taps == 9)
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): explicit input strides are for 1x1 / row-tap layers");
  if (BN > 256) return set_error(h, UG_EUNSUPPORTED, "conv(multi): BN <= 256");
  // 3x3 with one n-tile wider than 128 columns (GoogLeNet N = 192 ... 224): plain stores only (the gate / statistics
  // staging is sized for 128 columns), one accumulator per issuer
  if (taps == 9 && BN > 128 && (d->N > BN || d->mode != UG_EPI_STORE || d->pool_out || d->stats_sum))
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): 3x3 n-tiles wider than 128 need a single-tile STORE layer");
  if (up == 2 && (d->convt_cout % 64 || BN % 64))  // every 64-column store block lies inside one quadrant
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): ConvTranspose needs cout %% 64 == 0 and BN %% 64 == 0");
  if (taps == 1 && d->mode == UG_EPI_OUTC) return set_error(h, UG_EUNSUPPORTED, "conv(multi): OUTC is a 3x3 epilogue");
  int TW, TH, TN;
  int strip = 0, pitch = kMPitch;
  if (taps == 9) {
    TW = 8;
    TH = ceil_div(d->H, ceil_div(d->H, 16));  // <= 16 rows per tile, no wasted tile rows
    TN = 1;
    // row-strip tiles (SR full image rows per tile) when they put more output pixels on the 128 MMA rows than the
    // 8-pixel-wide tiles do: 28-wide maps (87.5 % instead of 76.6 %)
    const int sr_max = 128 / (d->W + 2);
    if (sr_max >= 1 && !d->stats_sum) {
      int sr = std::min(sr_max, d->H);
      if (d->pool_out) sr &= ~1;                                   // pooled tiles need an even number of rows
      if (sr >= 1) {
        sr = ceil_div(d->H, ceil_div(d->H, sr));                   // no wasted tile rows
        if (d->pool_out && (sr & 1)) sr = 0;
      }
      if (sr >= 1) {
        const double fill_strip = (double)d->H * d->W / ((double)ceil_div(d->H, sr) * 128.0);
        const double fill_tile = (double)d->H * d->W / ((double)ceil_div(d->W, 8) * ceil_div(d->H, TH) * 128.0);
        if (fill_strip > fill_tile + 1e-6) {
          strip = 1;
          pitch = d->W + 2;
          TW = d->W;
          TH = sr;
        }
      }
    }
  } else {
    choose_tile(d->B, d->H, d->W, &TW, &TH, &TN);
    if (TW > 256 || TH > 256 || TN > 256) return set_error(h, UG_EUNSUPPORTED, "conv(multi): tile exceeds the TMA box limits");
  }
  const int cin_pad = ceil_div(d->Cin, 64) * 64;
  const int kchunks = rowtaps ? d->R : cin_pad / 64;
  const int n_tiles = ceil_div(d->N, BN);
  const int npad = n_tiles * BN;
  const long long ktot = rowtaps ? (long long)d->R * 64 : (long long)taps * cin_pad;
  const int tma_store = d->mode != UG_EPI_OUTC;
  const int pool = d->pool_out != nullptr;
  if (pool && (taps != 9 || d->mode != UG_EPI_STORE || (d->H & 1) || (d->W & 1) || (TH & 1) || d->pool_cstride % 8 ||
               (reinterpret_cast<uintptr_t>(d->pool_out) & 15) || (TW / 2) * (TH / 2) * 128 > kPoolBytes))
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): fused max-pool needs a 3x3 STORE conv on an even map");
  const int stats = d->stats_sum != nullptr;
  // CTA pairs (see the header comment): 3x3 ReLU layers with 128-column n-tiles, plain stores (optionally pooled) or the
  // CoordAtt3 combine; narrower layers have their own pair kernel (conv_pair.cu)
  if (pair && (taps != 9 || BN != 128 || d->N < 128 || stats || (h->num_sms & 1) ||
               !(d->mode == UG_EPI_STORE || d->mode == UG_EPI_GATE)))
    return set_error(h, UG_EUNSUPPORTED, "conv(multi, pairs): 3x3 layers with 128-column n-tiles, STORE / GATE epilogue");
  if (stats && (taps != 9 || d->mode != UG_EPI_STORE || !d->stats_max ||
                d->stats_tiles != ceil_div(d->W, 8) * ceil_div(d->H, TH)))
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): fused channel statistics need a 3x3 STORE conv and stats_tiles == %d",
                     ceil_div(d->W, 8) * ceil_div(d->H, TH));
  const int obuf_bytes = tma_store ? kABytesPerStage + (pool ? kPoolBytes : 0) : 0;  // per staging buffer, for sizing
  // K-split: two issuing warps per tile stream for narrow 3x3 tiles (see the header comment)
  const int ks = (taps == 9 && BN <= 64 && !pair && d->act == UG_ACT_RELU && d->mode != UG_EPI_ADD) ? 2 : 1;
  // instantiated (activation, taps, epilogue) combinations: 3x3 = ReLU with any epilogue; 1x1 = plain stores with any
  // activation, residual add without activation
  if (taps == 9 && d->act != UG_ACT_RELU)
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): 3x3 layers are instantiated for ReLU only");
  if (taps == 1 && !(d->mode == UG_EPI_STORE || (d->mode == UG_EPI_ADD && d->act == UG_ACT_NONE)))
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): 1x1 layers are instantiated for STORE (any activation) and ADD (no activation)");
  const int acc_stages = std::max(1, std::min(4, 512 / (kMI * ks * BN)));
  // TMA residual (see the header comment): CoordAtt3 combine layers with one 64-column n-tile and resident weights.
  // Needs two staging buffers per stream next to the weights: tiles of <= 14 rows make room (the layer is bound by its
  // epilogue, not by the 12.5 % of MMA rows this leaves empty).
  int rt = (!pair && taps == 9 && !strip && ks == 2 && d->mode == UG_EPI_GATE && d->N <= 64 && BN == 64 && d->add_bstride > 0 &&
            !pool && !stats) ? 1 : 0;
  // pair mode: the residual of every 64-column sub-tile by TMA (an extra warp produces them: the weight warp is streaming);
  // costs the second staging buffer per stream, i.e. four of the 8 KB weight-ring slots
  const int rt_pair = (pair && d->mode == UG_EPI_GATE && d->add_bstride > 0 && d->add_cstride % 8 == 0 &&
                       !(reinterpret_cast<uintptr_t>(d->add) & 15)) ? 1 : 0;
  if (rt_pair) rt = 1;
  if (rt && !pair) {
    const int th2 = ceil_div(d->H, ceil_div(d->H, 14));
    const long long need = (long long)taps * kchunks * BN * 128 + kMI * 2LL * (((kMPitch * (th2 + 2) * 128) + 1023) / 1024 * 1024) +
                           kMI * 2LL * kABytesPerStage + 4096;
    if (need <= 227LL * 1024) TH = th2;
    else rt = 0;
  }
  // row halo (rowtaps 2): one box of TH + R - 1 rows per tile instead of R boxes of TH rows; needs whole 1024-byte swizzle
  // atoms per tile row (TW % 8 == 0) and one image per tile; otherwise one box per tap
  const int row_halo = (rowtaps && TW % 8 == 0 && TN == 1) ? 1 : 0;
  const int a_bytes = taps == 9 ? pitch * (TH + 2) * 128 : TW * (TH + (row_halo ? d->R - 1 : 0)) * TN * 128;
  // strip mode: MMA row 127 of tap (2,2) reads halo position 127 + 2*pitch + 2, past the loaded box (garbage rows only)
  const int a_span = strip ? std::max(a_bytes, (128 + 2 * pitch + 2) * 128) : a_bytes;
  const int a_stage = ((a_span + 1023) / 1024) * 1024;
  const int b_tile = (pair ? BN / 2 : BN) * 128;   // pairs: each CTA holds half of the rows of a weight tile

  MultiParams& hp = L->mp;
  memset(&hp, 0, sizeof(hp));
  hp.TH = TH;
  hp.a_stage_bytes = a_stage;
  hp.strip = strip;
  hp.pitch = pitch;
  hp.sbo = strip ? 1024 : pitch * 128;
  const int fixed = 1024 + 8 * (2 * kMI * 4 + 2 * 16 + 2 * kMI * 4 + 4 * kMI) + 16 + 2 * npad * (int)sizeof(float) +
                    kMI * 128 * (int)sizeof(float) + (stats ? kMI * 512 * (int)sizeof(float) : 0);
  const long long budget = 227LL * 1024 - fixed;
  int obufs = tma_store ? 2 : 0;
  const long long resB = (long long)taps * kchunks * b_tile;
  if (n_tiles == 1 && resB + kMI * 2LL * a_stage + (tma_store ? kMI * obuf_bytes : 0) <= budget) {
    hp.b_resident = 1;
    hp.sb = 1;
    if (resB + kMI * 2LL * a_stage + kMI * obufs * obuf_bytes > budget) obufs = 1;
    hp.sa = (int)std::min<long long>(4, (budget - resB - kMI * obufs * obuf_bytes) / (kMI * a_stage));
  } else {
    // streamed weights: the MMA time per tile is long, so one staging buffer per epilogue group is enough and the
    // shared memory goes to a deep weight ring instead (a slot is only handed back when the MMAs that read it have
    // COMPLETED, so several slots are always "in flight"; with 8 slots the issuers waited on weights 18 % of the time)
    hp.b_resident = 0;
    hp.sa = 2;
    // (the TMA residual of pair mode keeps both staging buffers if that leaves at least six 8 KB ring slots)
    if (obufs == 2 && !(rt_pair && (budget - kMI * 2LL * a_stage - kMI * 2LL * obuf_bytes) / b_tile >= 6)) obufs = 1;
    long long rest = budget - kMI * 2LL * a_stage - kMI * obufs * obuf_bytes;
    hp.sb = (int)std::min<long long>(16, rest / b_tile);
    if (hp.sb < 3) return set_error(h, UG_EUNSUPPORTED, "conv(multi): tile does not fit in shared memory");
    if (hp.sb >= 12 && rest - 10LL * b_tile >= kMI * a_stage) {  // room for a third activation stage
      hp.sa = 3;
      hp.sb = (int)std::min<long long>(16, (rest - kMI * a_stage) / b_tile);
    }
  }

  if (rt && !(obufs == 2 && (hp.b_resident || pair))) rt = 0;   // (does not fit after all: register-prefetched residual)
  hp.resid_tma = rt;
  hp.rowtaps = rowtaps ? 1 + row_halo : 0;

  ConvKParams& p = L->p;
  memset(&p, 0, sizeof(p));
  p.H = d->H; p.W = d->W; p.B = d->B;
  p.TW = TW; p.TH = TH; p.TN = TN;
  p.tiles_x = ceil_div(d->W, TW);
  p.tiles_y = ceil_div(d->H, TH);
  p.R = d->R; p.S = d->S; p.pad = d->pad;
  p.kchunks = kchunks; p.num_k = taps * kchunks;
  p.N = d->N; p.BN = BN; p.stages = hp.sa;
  int tcols = 32;
  while (tcols < kMI * ks * acc_stages * BN) tcols <<= 1;
  p.tmem_cols = pair ? 512 : tcols;   // (pairs: whole tensor memory, so that the addresses coincide in both CTAs)
  p.a_bytes = (unsigned)a_bytes; p.b_bytes = (unsigned)b_tile;
  p.scale = d->scale; p.bias = d->bias;
  p.act = d->act; p.mode = d->mode;
  p.out = d->out; p.out_cstride = d->out_cstride;
  p.up = up; p.convt_cout = d->convt_cout;
  p.OH = d->H * up; p.OW = d->W * up;
  p.add = d->add; p.add_bstride = d->add_bstride; p.add_cstride = d->add_cstride;
  p.gate = d->gate; p.outc_w = d->outc_w; p.outc_b = d->outc_b;
  p.logits = d->logits; p.mask = d->mask;
  p.m_tiles = p.tiles_x * p.tiles_y * ceil_div(d->B, TN); p.n_tiles = n_tiles; p.acc_stages = acc_stages;
  p.tma_store = tma_store; p.obufs = obufs; p.npad = npad; p.pool = pool;
  p.stats_sum = d->stats_sum; p.stats_max = d->stats_max;
  hp.m_super = ceil_div(p.m_tiles, kMI * (pair ? 2 : 1));
  hp.d_msuper = make_fastdiv(hp.m_super);
  hp.d_tx = make_fastdiv(p.tiles_x);
  hp.d_ty = make_fastdiv(p.tiles_y);
  hp.m_major = n_tiles > 1 ? 1 : 0;
  hp.d_nt = make_fastdiv(n_tiles);
  hp.d_pitch = make_fastdiv(pitch);
  L->kernel = pair ? ConvKernel::MultiPair : ConvKernel::Multi;
  L->multi_fn = nullptr;
  for (int i = 0; i < (int)(sizeof(kMultiInstances) / sizeof(kMultiInstances[0])); ++i) {
    const MultiInstance& k = kMultiInstances[i];
    if (k.act == d->act && k.taps == taps && k.mode == d->mode && k.ks == ks && k.rt == rt && k.pair == pair) {
      L->multi_fn = k.fn;
      L->instance = i;
    }
  }
  L->item_tiles = kMI * (pair ? 2 : 1);
  if (!L->multi_fn) return set_error(h, UG_EUNSUPPORTED, "conv(multi): no kernel instantiated for this layer");
  L->block = kMultiThreads(ks, rt && pair);

  {
    const long long in_h = d->H + (rowtaps ? d->R - 1 : 0);
    const long long rs = d->in_rstride ? d->in_rstride : (long long)d->W * d->in_cstride;
    const long long bs = d->in_bstride ? d->in_bstride : in_h * rs;
    if (rs % 8 || bs % 8) return set_error(h, UG_EINVAL, "conv(multi): input strides must be multiples of 8 elements");
    cuuint64_t dims[4] = {(cuuint64_t)(rowtaps ? 64 : d->Cin), (cuuint64_t)d->W, (cuuint64_t)in_h, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->in_cstride * 2, (cuuint64_t)rs * 2, (cuuint64_t)bs * 2};
    cuuint32_t box9[4] = {64, (cuuint32_t)pitch, (cuuint32_t)(TH + 2), 1};
    cuuint32_t box1[4] = {64, (cuuint32_t)TW, (cuuint32_t)(TH + (row_halo ? d->R - 1 : 0)), (cuuint32_t)TN};
    const int r = encode_bf16_sw128(&L->tmA, d->in, 4, dims, strides, taps == 9 ? box9 : box1, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
    if (r) return set_error(h, UG_ECUDA, "conv(multi): activation tensor map encode failed (%d)", r);
  }
  {
    // rows beyond N are zero-filled by TMA (the packed matrix is only guaranteed to hold N rows rounded up to the
    // packer's own tile, which may differ from BN)
    cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)d->N};
    cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)(pair ? BN / 2 : BN)};
    const int r = encode_bf16_sw128(&L->tmB, d->w, 2, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
    if (r) return set_error(h, UG_ECUDA, "conv(multi): weight tensor map encode failed (%d)", r);
  }
  memset(&L->maps, 0, sizeof(L->maps));
  if (rt) {  // load map of the residual tensor, same box as the output store
    cuuint64_t dims[4] = {(cuuint64_t)d->N, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->add_cstride * 2, (cuuint64_t)d->W * d->add_cstride * 2, (cuuint64_t)d->add_bstride * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TN};
    const int r = encode_bf16_sw128(&L->maps.m[4], d->add, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
    if (r) return set_error(h, UG_ECUDA, "conv(multi): residual tensor map encode failed (%d)", r);
  }
  if (tma_store) {
    cuuint32_t box[4] = {64, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TN};
    if (up == 1) {
      cuuint64_t dims[4] = {(cuuint64_t)d->N, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
      cuuint64_t strides[3] = {(cuuint64_t)d->out_cstride * 2, (cuuint64_t)d->W * d->out_cstride * 2,
                               (cuuint64_t)d->H * d->W * d->out_cstride * 2};
      const int r = encode_bf16_sw128(&L->maps.m[0], d->out, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_NONE);
      if (r) return set_error(h, UG_ECUDA, "conv(multi): output tensor map encode failed (%d)", r);
      if (pool) {  // fused nn.MaxPool2d(2): pooled tile = 4 x TH/2 pixels of the half-resolution map
        const long long pcs = d->pool_cstride;
        cuuint64_t pdims[4] = {(cuuint64_t)d->N, (cuuint64_t)(d->W / 2), (cuuint64_t)(d->H / 2), (cuuint64_t)d->B};
        cuuint64_t pstrides[3] = {(cuuint64_t)(pcs * 2), (cuuint64_t)((d->W / 2) * pcs * 2),
                                  (cuuint64_t)((long long)(d->H / 2) * (d->W / 2) * pcs * 2)};
        cuuint32_t pbox[4] = {64, (cuuint32_t)(TW / 2), (cuuint32_t)(TH / 2), 1};
        const int rp = encode_bf16_sw128(&L->maps.m[1], d->pool_out, 4, pdims, pstrides, pbox, CU_TENSOR_MAP_L2_PROMOTION_NONE);
        if (rp) return set_error(h, UG_ECUDA, "conv(multi): pooled output tensor map encode failed (%d)", rp);
      }
    } else {
      // ConvTranspose 2x2 s2: quadrant (dy,dx) of input pixel (y,x) is output pixel (2y+dy, 2x+dx); one strided view
      // of the output per quadrant turns the pixel shuffle into plain TMA tile stores
      const long long cs = d->out_cstride, OW = 2LL * d->W, OH = 2LL * d->H;
      for (int q = 0; q < 4; ++q) {
        const int dy = q >> 1, dx = q & 1;
        void* base = static_cast<char*>(d->out) + ((long long)dy * OW + dx) * cs * 2;
        cuuint64_t dims[4] = {(cuuint64_t)d->convt_cout, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->B};
        cuuint64_t strides[3] = {(cuuint64_t)(2 * cs * 2), (cuuint64_t)(2 * OW * cs * 2), (cuuint64_t)(OH * OW * cs * 2)};
        const int r = encode_bf16_sw128(&L->maps.m[q], base, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_NONE);
        if (r) return set_error(h, UG_ECUDA, "conv(multi): ConvTranspose output tensor map encode failed (%d)", r);
      }
    }
  }
  const long long total_super = (long long)hp.m_super * n_tiles;
  if (pair) L->grid = dim3(2u * (unsigned)std::min<long long>(total_super, (long long)(h->num_sms / 2)), 1, 1);
  else L->grid = dim3((unsigned)std::min<long long>(total_super, (long long)h->num_sms), 1, 1);
  const int nb_tiles = hp.b_resident ? taps * kchunks : hp.sb;
  L->smem = 1024 + (size_t)kMI * hp.sa * a_stage + (size_t)nb_tiles * b_tile + (size_t)kMI * obufs * obuf_bytes +
            8 * (2 * kMI * hp.sa + 2 * hp.sb + 2 * kMI * acc_stages + 4 * kMI) + 16 + 2 * (size_t)npad * sizeof(float) +
            kMI * 128 * sizeof(float) + (stats ? kMI * 512 * sizeof(float) : 0);
  if (L->smem > (size_t)227 * 1024)
    return set_error(h, UG_EUNSUPPORTED, "conv(multi): shared memory request %zu too large", L->smem);
  return UG_OK;
}

int conv_multi_launch(ug_engine* h, const ConvLaunch* L, cudaStream_t s) {
  if (!h->attr_multi) {
    for (const MultiInstance& k : kMultiInstances) {
      const cudaError_t e = cudaFuncSetAttribute((const void*)k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e != cudaSuccess) return check_cuda(h, e, "cudaFuncSetAttribute(conv_multi_kernel)");
    }
    h->attr_multi = true;
  }
  const cudaError_t e =
      L->kernel == ConvKernel::MultiPair
          ? launch_pairs(h, L->multi_fn, L->grid.x, L->block, L->smem, s, L->tmA, L->tmB, L->maps, L->p, L->mp)
          : launch_pdl(L->multi_fn, L->grid, L->block, L->smem, s, L->tmA, L->tmB, L->maps, L->p, L->mp);
  h->launches++;
  return check_cuda(h, e != cudaSuccess ? e : cudaGetLastError(), "conv_multi_kernel launch");
}

}  // namespace ug
