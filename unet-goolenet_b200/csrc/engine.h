// Internal engine declarations shared by the .cu translation units of libugnet.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
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
};

// Division by a launch-time constant as multiply + shift (exact for n < 2^24): the role loops decode a tile index
// into (image, tile row, tile column) once per tile, and on the short K=64 / N=64 tiles that decode (four integer
// divisions, ~25 instructions each) was a third of the epilogue time.
struct FastDiv {
  unsigned mul, shift;
  __device__ __forceinline__ int div(int n) const {
    return (int)(((unsigned long long)(unsigned)n * mul) >> shift);
  }
};
inline FastDiv make_fastdiv(int d) {
  FastDiv f;
  int s = 0;
  while ((1 << s) < d) ++s;
  f.shift = 24 + s;
  f.mul = (unsigned)(((1ULL << f.shift) + d - 1) / d);
  return f;
}

// Parameter block of the multi-issuer kernel (csrc/conv_multi.cu).
struct MultiParams {
  int TH;             // output rows per tile (tile = 8 x TH pixels)
  int a_stage_bytes;  // bytes of one activation stage
  int sa, sb;         // activation stages per issuer / shared weight stages
  int b_resident;     // whole weight matrix kept in smem (requires n_tiles == 1)
  int m_super;        // ceil(m_tiles / kMI): pixel tiles are handed out in groups of kMI
  FastDiv d_msuper, d_tx, d_ty;   // dividers by m_super, tiles_x, tiles_y
  int m_major;        // work item s -> (pixel-tile group s / n_tiles, n-tile s % n_tiles): the n-tiles of one pixel-tile group
                      // run on neighbouring CTAs at the same time, so the activation tile comes from HBM once and from L2
                      // for the other n-tiles (n-major order re-read the whole input from HBM once per n-tile)
  FastDiv d_nt;       // divider by n_tiles
  int pitch;          // halo pixels per stage row: kMPitch (8-pixel-wide tiles) or W + 2 (row-strip tiles)
  int sbo;            // byte distance of consecutive 8-row groups of the A operand: pitch * 128 (tiles) or 1024 (strips)
  int strip;          // row-strip tiles (see the header comment); TH is then the number of image rows per tile
  FastDiv d_pitch;    // divider by pitch (strip mode: MMA row -> (image row, x))
  int rowtaps;        // 1x1 tiles: k-chunk kc is ROW TAP kc of an overlapping-window input.  1: one A box per tap (at row
                      // y0 + kc); 2: ONE box of TH + R - 1 rows per tile, tap kc reads it TW * 128 * kc bytes further in
                      // (a "row halo": the window rows of neighbouring taps are the same bytes)
  int resid_tma;      // kRT kernels: residual tiles arrive by TMA in the staging buffers (see the header comment)
};

struct StoreMaps {  // output maps: [0] for plain stores, [q] = quadrant (dy,dx) of a ConvTranspose 2x2 s2 scatter;
  CUtensorMap m[5];  // [1] = pooled output (fused max-pool); [4] = load map of the residual tensor (kRT)
};

// Parameter block of the CTA-pair kernel (csrc/conv_pair.cu).
struct PairParams {
  int TH, a_stage_bytes, sa, n_quads;   // rows per tile, bytes of one activation stage, stages per stream, tile groups
  int streams;                          // tile streams per CTA: 2, or 1 when the resident weights leave room for one
  FastDiv d_tx, d_ty;
};

struct PairMaps {
  CUtensorMap out, pool, resid;
};

// Which kernel a prepared conv launches.
enum class ConvKernel {
  OneTile,     // conv_gemm_kernel: one output tile per CTA
  Persistent,  // conv_gemm_persistent_kernel
  Multi,       // conv_multi_kernel: two MMA issuers per CTA
  MultiPair,   // conv_multi_kernel on clusters of two CTAs (128-column n-tiles)
  Pair,        // conv_pair_kernel: clusters of two CTAs, <= 64 output channels
};

typedef void (*MultiKernelFn)(CUtensorMap, CUtensorMap, StoreMaps, ConvKParams, MultiParams);
typedef void (*PairKernelFn)(CUtensorMap, CUtensorMap, PairMaps, ConvKParams, PairParams);

// The instantiated conv_multi_kernel<activation, taps, epilogue mode, K-split, TMA residual, CTA pair> combinations and
// conv_pair_kernel<epilogue mode, TMA residual> forms, in table order: conv_multi.cu / conv_pair.cu build their kernel
// tables from these lists (prepare admits exactly these), and the launch-plan query of libugnet_dev.so enumerates them.
#define UG_MULTI_INSTANCES(X)                   \
  X(UG_ACT_RELU, 9, UG_EPI_STORE, 1, 0, 0)      \
  X(UG_ACT_RELU, 9, UG_EPI_STORE, 2, 0, 0)      \
  X(UG_ACT_RELU, 9, UG_EPI_ADD, 1, 0, 0)        \
  X(UG_ACT_RELU, 9, UG_EPI_GATE, 1, 0, 0)       \
  X(UG_ACT_RELU, 9, UG_EPI_GATE, 2, 0, 0)       \
  X(UG_ACT_RELU, 9, UG_EPI_GATE, 2, 1, 0)       \
  X(UG_ACT_RELU, 9, UG_EPI_OUTC, 1, 0, 0)       \
  X(UG_ACT_RELU, 9, UG_EPI_OUTC, 2, 0, 0)       \
  X(UG_ACT_NONE, 1, UG_EPI_STORE, 1, 0, 0)      \
  X(UG_ACT_RELU, 1, UG_EPI_STORE, 1, 0, 0)      \
  X(UG_ACT_GELU, 1, UG_EPI_STORE, 1, 0, 0)      \
  X(UG_ACT_NONE, 1, UG_EPI_ADD, 1, 0, 0)        \
  X(UG_ACT_RELU, 9, UG_EPI_STORE, 1, 0, 1)      \
  X(UG_ACT_RELU, 9, UG_EPI_GATE, 1, 0, 1)       \
  X(UG_ACT_RELU, 9, UG_EPI_GATE, 1, 1, 1)
#define UG_PAIR_INSTANCES(X) X(UG_EPI_STORE, 0) X(UG_EPI_OUTC, 0) X(UG_EPI_GATE, 1)

// A fully prepared launch of one of the conv kernels: the prepare functions fill the kernel's parameter blocks and
// tensor maps, the launch functions only launch.
struct ConvLaunch {
  alignas(64) CUtensorMap tmA;
  alignas(64) CUtensorMap tmB;
  alignas(64) CUtensorMap tmO;   // persistent GEMM kernel: output map (TMA-store epilogue)
  alignas(64) CUtensorMap tmO2;  // persistent GEMM kernel: second destination of a split 1x1 GEMM
  StoreMaps maps;                // multi-issuer kernel
  PairMaps pmaps;                // CTA-pair kernel
  ConvKParams p;
  MultiParams mp;                // multi-issuer kernel
  PairParams pp;                 // CTA-pair kernel
  ConvKernel kernel;
  MultiKernelFn multi_fn;        // the conv_multi_kernel instantiation (activation, taps, epilogue, K-split, ...)
  PairKernelFn pair_fn;          // the conv_pair_kernel instantiation (epilogue)
  int instance;                  // row of UG_MULTI_INSTANCES (Multi, MultiPair) / UG_PAIR_INSTANCES (Pair); 0 otherwise
  int item_tiles;                // pixel tiles per work item: kMI (Multi), 2 kMI (MultiPair), 2 streams (Pair), 1 (GEMM)
  dim3 grid;
  unsigned block;
  size_t smem;
};

// Stem convolution (csrc/stem_conv.cu): kernel parameters and a prepared launch.
struct StemParams {
  const float* in_f32;
  const unsigned char* in_u8;   // (not read by the inc kernel)
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
  alignas(64) CUtensorMap tmP;  // pooled output (pool_out)
  StemParams p;
  unsigned grid, block;
  size_t smem;
};

int set_error(ug_engine* h, int code, const char* fmt, ...);
int check_cuda(ug_engine* h, cudaError_t e, const char* what);

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Driver entry point cuTensorMapEncodeTiled (nullptr when unavailable) and the one map format the kernels use: bf16
// elements, 128-byte swizzle (boxes with an inner extent of 64 elements), no interleave, zero fill.  Returns the CUresult.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn();
int encode_bf16_sw128(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                      const cuuint32_t* box, CUtensorMapL2promotion promo);

// Launch `kernel` on `s` with the programmatic-stream-serialization attribute, so the kernel may start its prologue
// while the previous kernel of the stream drains.  ONLY for kernels that execute pdl_wait() (common.cuh) before their
// first access to memory written by earlier kernels.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Launch configuration of a grid of CTA pairs (clusters of two CTAs along x), attribute 0 = the cluster shape,
// attribute 1 = programmatic stream serialization (as in launch_pdl); `at` holds the attributes.
inline cudaLaunchConfig_t pair_config(cudaLaunchAttribute (&at)[2], unsigned grid_x, unsigned block, size_t smem,
                                      cudaStream_t s) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid_x);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 2;
  return cfg;
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

// Launch a persistent CTA-pair kernel (pair_config) on at most max_cluster_pairs(h) pairs: its loops take any even grid.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pairs(ug_engine* h, void (*kernel)(KArgs...), unsigned grid_x, unsigned block, size_t smem,
                                cudaStream_t s, Args&&... args) {
  cudaLaunchAttribute at[2];
  const cudaLaunchConfig_t cfg = pair_config(at, std::min(grid_x, 2u * (unsigned)max_cluster_pairs(h)), block, smem, s);
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int stem_prepare(ug_engine* h, const ug_stem_desc* d, StemLaunch* out);
int stem_launch(ug_engine* h, const StemLaunch* l, cudaStream_t s);

// Which kernel a memory-bound op of csrc/mem_kernels.cu launches (same order as UG_MEMOP_KERNEL_* of ugnet_dev.h).
enum class MemKernel {
  Pool,            // pool_kernel: any window
  Pool3x3s1,       // pool3x3s1_kernel: sliding rows (maps under 196 pixels)
  Pool3x3s1Block,  // pool3x3s1_block_kernel: 2x2 output blocks
  Pool3x3s2,       // pool3x3s2_kernel: 2x2 output blocks, ceil mode
  LayerNorm,       // layernorm_kernel<C / 256>
  Attention,       // attention_mma_kernel
  ChanStats,       // chanstats_kernel
  Gate,            // gate_hidden_kernel + gate_out_kernel (two launches, same grid)
  BBox,            // bbox_kernel
  CropResize,      // resize_u8_kernel<kCrop>
  S2d,             // s2d_pack_kernel
  Head,            // head_kernel
};

// The launch of a memory-bound op: validation and every dispatch rule live in the op's plan_* function, which both the
// launcher and the launch-plan query of libugnet_dev.so (ug_memop_launch_info) call.
struct MemLaunch {
  MemKernel kernel;
  int variant;       // layernorm_kernel<kNV>: kNV; resize_u8_kernel<kMode>: kMode; -1 otherwise
  dim3 grid;
  unsigned block;
  size_t smem;       // dynamic shared memory
  int max_rows;      // resize_u8_kernel: source rows staged per block
};
int plan_pool(ug_engine* h, const ug_pool_desc* d, MemLaunch* L);
int plan_layernorm(ug_engine* h, const ug_layernorm_desc* d, MemLaunch* L);
int plan_attention(ug_engine* h, const ug_attn_desc* d, MemLaunch* L);
int plan_chanstats(ug_engine* h, const ug_chanstats_desc* d, MemLaunch* L);
int plan_gate(ug_engine* h, const ug_gate_desc* d, MemLaunch* L);
int plan_bbox(ug_engine* h, const ug_bbox_desc* d, MemLaunch* L);
int plan_cropresize(ug_engine* h, const ug_cropresize_desc* d, MemLaunch* L);
int plan_s2d_pack(ug_engine* h, const ug_s2d_desc* d, MemLaunch* L);
int plan_head(ug_engine* h, const ug_head_desc* d, MemLaunch* L);

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
int launch_cam(ug_engine* h, const ug_cam_desc* d, cudaStream_t s);
int launch_source_frame(ug_engine* h, const ug_source_frame_desc* d, cudaStream_t s);

}  // namespace ug
