// Internal engine declarations shared by the .cu translation units of libugnet.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <string>
#include <vector>
#include "../../include/ugnet.h"

struct ug_engine {
  int device = 0;
  int num_sms = 148;
  std::string last_error;
  long long launches = 0;
  // double-buffered host feeding (ug_program_run_host_pipelined): engine-owned copy stream and slot events
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr};   // staging slot filled (recorded on the copy stream)
  cudaEvent_t ev_free[2] = {nullptr, nullptr};  // staging slot consumed (recorded on the compute stream)
  long long pipelined_steps = 0;
  int pdl = 1;  // launch kernels with programmatic stream serialization (UG_PDL=0 turns it off)
  // cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the device that is current at the call, so the
  // "already raised" flags are per handle (= per device), not process-wide
  bool attr_gemm = false, attr_multi = false, attr_pair = false, attr_stem = false, attr_attn = false;
  int max_pairs = -1;  // co-resident clusters of two ~200 KB CTAs on this device (cudaOccupancyMaxActiveClusters), -1 = not queried
  size_t attr_resize = 0, attr_crop = 0, attr_ragged = 0;
};

namespace ug {
// Makes the handle's device current for the duration of an entry point and restores the caller's device afterwards
// (PyTorch and other libraries in the host process own the "current device" state).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(const ug_engine* h) {
    if (h && cudaGetDevice(&prev) == cudaSuccess && prev != h->device) switched = cudaSetDevice(h->device) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
}  // namespace ug

namespace ug {

// Kernel-side parameter block of the implicit-GEMM kernel (kept POD; passed by value).
struct ConvKParams {
  int H, W, B;
  int TW, TH, TN, tiles_x, tiles_y;
  int R, S, pad, kchunks, num_k;
  int N, BN, stages, tmem_cols;
  unsigned a_bytes, b_bytes;
  const float* scale;
  const float* bias;
  int act, mode;
  void* out;
  int out_cstride, OH, OW, up, convt_cout;
  const void* add;
  long long add_bstride;
  int add_cstride;
  const float* gate;
  const float* outc_w;
  float outc_b;
  float* logits;
  unsigned char* mask;
  // persistent variant
  int m_tiles, n_tiles, acc_stages, tma_store, obufs, npad;
  int pool;        // multi-issuer 3x3 kernel: fused 2x2 max-pool side output (second TMA store per sub-tile)
  int m_major;     // persistent GEMM kernel: tile order (pixel tile, n-tile) instead of (n-tile, pixel tile)
  float* stats_sum;  // multi-issuer 3x3 kernel: per-tile channel sums / maxima of the stored output
  float* stats_max;
  int stage_copy;  // ConvTranspose scatter: stage the tile in smem, then coalesced cooperative copy-out
  void* out2;      // second destination of a split 1x1 GEMM (see ug_conv_desc.out2): columns >= n_split
  int out2_cstride, n_split, n1;
  long long* prof;  // optional per-CTA cycle counters [grid][8] (debug / profiling builds of the plan)
};

// A fully prepared launch of the implicit-GEMM kernel.
struct ConvLaunch {
  alignas(64) CUtensorMap tmA;
  alignas(64) CUtensorMap tmB;
  alignas(64) CUtensorMap tmO;  // output map for the TMA-store epilogues
  alignas(64) CUtensorMap tmO2;    // persistent GEMM kernel: TMA-store map of the second destination (split 1x1 GEMM)
  alignas(64) CUtensorMap tmR;     // multi-issuer kernel: TMA load map of the residual tensor (kRT kernels)
  alignas(64) CUtensorMap tmQ[3];  // multi-issuer kernel, ConvTranspose: output views of quadrants 1..3 (tmO = quadrant 0)
  ConvKParams p;
  dim3 grid;
  size_t smem;
  int variant;  // 0 = persistent, 1 = one tile per CTA, 5 = multi-issuer kernel (halo_mode = taps: 9 or 1), 6 = CTA-pair kernel
  int halo_mode, halo_TH, halo_a_stage, halo_copy, halo_sa, halo_sb, halo_bres, halo_debug;
  int halo_strip, halo_pitch;  // multi-issuer kernel: row-strip tiles (full image rows per tile) and their halo pitch
  int halo_rt;  // multi-issuer kernel: residual tiles by TMA into the staging buffers (CoordAtt3 combine, 64 channels)
  int halo_rowtaps;  // multi-issuer kernel, 1x1 tiles: the k-chunks are R row taps of an overlapping-window input
  int halo_ks;  // multi-issuer kernel: issuing warps per tile stream (K-split), 1 or 2
  int halo_pair;  // multi-issuer kernel: clusters of two CTAs issuing tcgen05.mma.cta_group::2 (128-column n-tiles)
};

// Stem convolution (csrc/stem_conv.cu): kernel parameters and a prepared launch.
struct StemParams {
  const float* in_f32;
  const unsigned char* in_u8;
  const float* scale;
  const float* bias;
  int B, H, W;  // source image
  int OH, OW;   // output map
  int tiles_x, tiles_y, total_tiles;
  int pool;     // fused 2x2 max-pool side output
};
struct StemLaunch {
  alignas(64) CUtensorMap tmB;
  alignas(64) CUtensorMap tmO;
  alignas(64) CUtensorMap tmP;  // pooled output (kind 0 with pool_out)
  StemParams p;
  int kind;
  int groups;   // warpgroups (independent tile pipelines) per CTA
  unsigned grid;
  size_t smem;
};

int set_error(ug_engine* h, int code, const char* fmt, ...);
int check_cuda(ug_engine* h, cudaError_t e, const char* what);

// Launch `kernel` on `s`; with h->pdl the launch carries the programmatic-stream-serialization attribute, so the kernel
// may start its prologue while the previous kernel of the stream drains.  ONLY for kernels that execute pdl_wait()
// (common.cuh) before their first access to memory written by earlier kernels.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(const ug_engine* h, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = (h && h->pdl) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int conv_prepare(ug_engine* h, const ug_conv_desc* d, ConvLaunch* out);
int conv_launch(ug_engine* h, const ConvLaunch* l, cudaStream_t s);
int conv_multi_prepare(ug_engine* h, const ug_conv_desc* d, int BN, ConvLaunch* out, int pair = 0);
int conv_multi_launch(ug_engine* h, const ConvLaunch* l, cudaStream_t s);
// CTA-pair kernel (csrc/conv_pair.cu): 3x3 ReLU layers with <= 64 output channels, tcgen05.mma.cta_group::2
int conv_pair_prepare(ug_engine* h, const ug_conv_desc* d, ConvLaunch* out);
int conv_pair_launch(ug_engine* h, const ConvLaunch* l, cudaStream_t s);
// Number of CTA pairs (clusters of two CTAs with ~200 KB of shared memory each) the device can keep resident at once:
// the persistent pair kernels must not launch more, or the surplus clusters would run as a second wave.  Usually
// num_sms / 2; fewer when a GPC has an odd number of usable SMs.
int max_cluster_pairs(ug_engine* h);

int stem_prepare(ug_engine* h, const ug_stem_desc* d, StemLaunch* out);
int stem_launch(ug_engine* h, const StemLaunch* l, cudaStream_t s);

int launch_pool(ug_engine* h, const ug_pool_desc* d, cudaStream_t s);
int launch_layernorm(ug_engine* h, const ug_layernorm_desc* d, cudaStream_t s);
int launch_attention(ug_engine* h, const ug_attn_desc* d, cudaStream_t s);
int launch_chanstats(ug_engine* h, const ug_chanstats_desc* d, cudaStream_t s);
int launch_gate(ug_engine* h, const ug_gate_desc* d, cudaStream_t s);
int launch_bbox(ug_engine* h, const ug_bbox_desc* d, cudaStream_t s);
int launch_cropresize(ug_engine* h, const ug_cropresize_desc* d, cudaStream_t s);
int launch_head(ug_engine* h, const ug_head_desc* d, cudaStream_t s);
int launch_resize_u8(ug_engine* h, const ug_resize_desc* d, cudaStream_t s);
int launch_wavelet(ug_engine* h, const ug_wavelet_desc* d, cudaStream_t s);
int launch_s2d_pack(ug_engine* h, const ug_s2d_desc* d, cudaStream_t s);
int launch_resize_ragged(ug_engine* h, const ug_resize_ragged_desc* d, cudaStream_t s);
int launch_wavelet_ragged(ug_engine* h, const ug_wavelet_ragged_desc* d, cudaStream_t s);

}  // namespace ug
