/* ugnet_dev.h — development hooks of libugnet_dev.so (NOT part of the product ABI in ugnet.h).
 *
 * libugnet_dev.so links the same objects as libugnet.so plus csrc/dev_hooks.cu and csrc/microbench.cu; it exists so
 * that scripts/mma_bench*.py can run tcgen05 issue-rate micro-benchmarks, and tests/test_conv_coverage_gpu.py /
 * tests/test_memops_coverage_gpu.py can ask which kernel and configuration a conv, memory-bound or stem descriptor
 * selects, without those entry points shipping in the product library.  Load it with UG_DEV_LIB=1
 * (unet-goolenet_b200/engine.py); handles are not interchangeable between the two libraries. */
#ifndef UGNET_DEV_H_
#define UGNET_DEV_H_
#include "ugnet.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Average SM cycles per tcgen05.mma (M=128, N, K=16) with n_acc interleaved TMEM accumulators and ctas_per_sm
 * co-resident CTAs. */
int ug_mma_microbench(ug_handle h, int N, int n_acc, int iters, int ctas_per_sm, int distinct_ab,
                      double* cycles_per_mma);
/* Same with `issuers` (1..4) warps of one CTA each issuing their own chain(s): out2[0] = cycles per MMA of one issuer,
 * out2[1] = launch wall time in ms. */
int ug_mma_microbench2(ug_handle h, int N, int n_acc, int issuers, int iters, int ctas_per_sm, int a_off, int a_sbo,
                       int acc_stride, double* out2);

/* CTA pairs (cluster of 2) issuing tcgen05.mma.cta_group::2 (M = 256 over two SMs, N/2 of B per CTA) from `issuers`
 * (1..4) warps of the leader CTA: out2[0] = cycles per M=256 MMA of one issuer, out2[1] = launch wall time in ms. */
int ug_mma_microbench_pair(ug_handle h, int N, int issuers, int iters, double* out2);

/* Conv kernel kinds of a launch plan. */
enum {
  UG_CONV_KERNEL_ONETILE = 0,     /* conv_gemm_kernel: one output tile per CTA */
  UG_CONV_KERNEL_PERSISTENT = 1,  /* conv_gemm_persistent_kernel */
  UG_CONV_KERNEL_MULTI = 2,       /* conv_multi_kernel, one CTA per SM */
  UG_CONV_KERNEL_MULTI_PAIR = 3,  /* conv_multi_kernel on clusters of two CTAs */
  UG_CONV_KERNEL_PAIR = 4         /* conv_pair_kernel (clusters of two CTAs, <= 64 output channels) */
};

/* One compiled instantiation of a conv kernel: its template arguments; -1 where the kernel has no such argument (the
 * GEMM kernels are instantiated per activation only, the pair kernel per epilogue mode). */
typedef struct ug_conv_instance {
  int act, taps, mode, ks, rt, pair;
} ug_conv_instance_t;

/* Writes the instantiations of conv kernel `kernel` (UG_CONV_KERNEL_*) to out[0 .. min(n, cap)) and returns n, their
 * number (< 0 for an unknown kernel).  Row i is what ug_conv_launch_info reports as `instance` i. */
int ug_conv_instances(int kernel, ug_conv_instance_t* out, int cap);

/* The launch plan that ug_conv would run for a descriptor. */
typedef struct ug_conv_launch_info {
  int kernel;                  /* UG_CONV_KERNEL_* */
  int instance;                /* row of ug_conv_instances(kernel) */
  ug_conv_instance_t inst;     /* that row */
  int BN, n_tiles, TW, TH, TN; /* n-tile width and count; pixel tile (TN images per tile) */
  int strip;                   /* multi kernel: row-strip tiles (TH full image rows) */
  int rowtaps, row_halo;       /* multi kernel: R x 1 row-tap layer; one activation box of TH + R - 1 rows per tile */
  int kchunks;                 /* 64-channel k-chunks per tap (row taps: the taps) */
  int b_resident;              /* multi kernel: the whole weight matrix in shared memory */
  int sa, sb;                  /* activation stages (per tile stream); weight stages (multi kernel) */
  int obufs, acc_stages;       /* staging buffers per tile stream; accumulator stages */
  int pool, stats, split;      /* fused 2x2 max-pool; fused channel statistics; second destination (out2) */
  int up;                      /* 2: ConvTranspose 2x2 s2 */
  int streams, n_quads;        /* pair kernel: tile streams per CTA; tile groups */
  int block, grid;             /* threads per CTA; CTAs launched (pair kernels: after the co-residency clamp) */
  long long smem;              /* dynamic shared memory per CTA */
  long long m_tiles;           /* pixel tiles */
  long long items, units;      /* work items (item_tiles pixel tiles x one n-tile); CTAs or CTA pairs working at once */
  int item_tiles;              /* pixel tiles per work item */
  int rounds;                  /* ceil(items / units) */
  long long last_round_items;  /* work items of the last round */
  long long tiles_past_end;    /* tile slots of the last work item per n-tile that lie past the last pixel tile */
} ug_conv_launch_info_t;

/* Runs the conv's plan-time preparation (validation, kernel and configuration choice) and copies the plan out.  Launches
 * nothing and allocates no device memory.  Returns what ug_conv would return for a rejected descriptor. */
int ug_conv_launch_info(ug_handle h, const ug_conv_desc* d, ug_conv_launch_info_t* out);

/* Kernels of the memory-bound ops (csrc/mem_kernels.cu) and of the stem (csrc/stem_conv.cu). */
enum {
  UG_MEMOP_KERNEL_POOL = 0,              /* pool_kernel: any window */
  UG_MEMOP_KERNEL_POOL_3X3S1 = 1,        /* pool3x3s1_kernel: sliding rows */
  UG_MEMOP_KERNEL_POOL_3X3S1_BLOCK = 2,  /* pool3x3s1_block_kernel: 2x2 output blocks (H*W >= 196) */
  UG_MEMOP_KERNEL_POOL_3X3S2 = 3,        /* pool3x3s2_kernel: 2x2 output blocks */
  UG_MEMOP_KERNEL_LAYERNORM = 4,         /* layernorm_kernel<variant> */
  UG_MEMOP_KERNEL_ATTENTION = 5,         /* attention_mma_kernel */
  UG_MEMOP_KERNEL_CHANSTATS = 6,         /* chanstats_kernel */
  UG_MEMOP_KERNEL_GATE = 7,              /* gate_hidden_kernel + gate_out_kernel, same grid */
  UG_MEMOP_KERNEL_BBOX = 8,              /* bbox_kernel */
  UG_MEMOP_KERNEL_CROPRESIZE = 9,        /* resize_u8_kernel<variant> (1 = crop mode) */
  UG_MEMOP_KERNEL_S2D = 10,              /* s2d_pack_kernel */
  UG_MEMOP_KERNEL_HEAD = 11,             /* head_kernel */
  UG_MEMOP_KERNEL_STEM = 12              /* stem_conv_kernel (UNet inc) */
};

/* The launch that the single-op entry point would make for a memory-bound or stem op. */
typedef struct ug_memop_launch_info {
  int kernel;                  /* UG_MEMOP_KERNEL_* */
  int variant;                 /* layernorm: the template argument C / 256; cropresize: the resize mode; -1 otherwise */
  int grid_x, grid_y, block;   /* CTAs and threads per CTA */
  int launches;                /* kernels launched (gate: 2 with the same grid) */
  long long smem;              /* dynamic shared memory per CTA */
} ug_memop_launch_info_t;

/* Runs the op's validation and launch decision (the same host function its launcher calls) for op->kind in {POOL,
 * LAYERNORM, ATTN, CHANSTATS, GATE, BBOX, CROPRESIZE, HEAD, S2D, STEM} and copies the launch out.  Launches nothing.
 * Returns what the op's entry point would return for a rejected descriptor (UG_EINVAL for any other kind). */
int ug_memop_launch_info(ug_handle h, const ug_op* op, ug_memop_launch_info_t* out);

#ifdef __cplusplus
}
#endif
#endif /* UGNET_DEV_H_ */
