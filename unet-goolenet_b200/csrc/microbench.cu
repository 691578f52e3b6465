// Micro-benchmarks used to size the conv kernels (not on the product path):
//   ug_mma_microbench: cycles per tcgen05.mma (M=128, N, K=16, bf16, both operands in 128B-swizzled smem) when
//   `n_acc` independent TMEM accumulators are interleaved and `n_cta` CTAs share an SM.
#include <vector>
#include "conv_common.cuh"
#include "../../include/ugnet_dev.h"

namespace ug {

__global__ void __launch_bounds__(128) mma_bench_kernel(int N, int n_acc, int iters, int distinct_ab, long long* out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_ptr;
  // A: 4 tiles x 16 KB, B: 4 tiles x N*128 B (zero-filled: values are irrelevant for timing)
  for (int i = threadIdx.x; i < (4 * 16384 + 4 * N * 128) / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  int cols = 32;
  while (cols < n_acc * N) cols <<= 1;
  if (warp == 1) {
    tmem_alloc(&tmem_ptr, cols);
    tmem_relinquish();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_ptr;
  if (warp == 0 && lane == 0) {
    const uint32_t idesc = umma_idesc_bf16(128, N);
    const uint32_t a0 = smem_u32(smem), b0 = smem_u32(smem + 4 * 16384);
    const long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
      const int buf = distinct_ab ? (it & 3) : 0;
      const uint64_t ad = umma_desc_sw128(a0 + buf * 16384);
      const uint64_t bd = umma_desc_sw128(b0 + buf * N * 128);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        for (int g = 0; g < n_acc; ++g) umma_bf16(tmem_base + g * N, ad + 2 * k, bd + 2 * k, idesc, 1u);
    }
    umma_commit(&bar);
    mbar_wait(&bar, 0);
    const long long t1 = clock64();
    out[blockIdx.x] = t1 - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, cols);
}


// Second form: `issuers` warps of ONE CTA each issue their own dependent MMA chain(s) (n_acc accumulators per
// issuer, private A tile, shared B tile).  Answers whether several issuing threads of one CTA overlap the way
// co-resident CTAs do.  The smem footprint is small (issuers*16 KB + N*128 B) so up to 4 CTAs fit per SM.
__global__ void __launch_bounds__(128) mma_bench2_kernel(int N, int n_acc, int issuers, int iters, int a_off,
                                                         int a_sbo, int acc_stride, long long* out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  __shared__ uint64_t bar[4];
  __shared__ uint32_t tmem_ptr;
  for (int i = threadIdx.x; i < (issuers * 24576 + N * 128) / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(&bar[i], 1);
    fence_mbar_init();
  }
  int cols = 32;
  const int acc_step = acc_stride > 0 ? acc_stride : n_acc * N;  // TMEM columns between the issuers' accumulators
  while (cols < (issuers - 1) * acc_step + n_acc * N) cols <<= 1;
  if (warp == 0) {
    tmem_alloc(&tmem_ptr, cols);
    tmem_relinquish();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_ptr;
  if (warp < issuers && lane == 0) {
    const uint32_t idesc = umma_idesc_bf16(128, N);
    // A: start address shifted by a_off bytes (multiple of 128) and 8-row groups a_sbo bytes apart, as in the
    // halo layout of the 3x3 kernels (a_off = 0, a_sbo = 1024 is the plain tile)
    uint64_t ad = umma_desc_sw128(smem_u32(smem + warp * 24576 + a_off));
    ad = (ad & ~(0x3FFFULL << 32)) | (static_cast<uint64_t>(a_sbo >> 4) << 32);
    const uint64_t bd = umma_desc_sw128(smem_u32(smem + issuers * 24576));
    const uint32_t d0 = tmem_base + warp * acc_step;
    const long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        for (int g = 0; g < n_acc; ++g) umma_bf16(d0 + g * N, ad + 2 * k, bd + 2 * k, idesc, 1u);
    }
    umma_commit(&bar[warp]);
    mbar_wait(&bar[warp], 0);
    const long long t1 = clock64();
    if (warp == 0) out[blockIdx.x] = t1 - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, cols);
}


// Third form: a CTA PAIR (cluster of 2) issuing tcgen05.mma.cta_group::2 (M = 256 across the two SMs, each CTA supplies
// its own 128 A rows and N/2 of the B rows).  `issuers` warps of the LEADER CTA each run their own chain into their own
// accumulator.  Answers what MMA rate a 2-CTA conv kernel could reach for N = 64 / 128 tiles.
__global__ void __launch_bounds__(128) mma_bench_pair_kernel(int N, int issuers, int iters, long long* out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  __shared__ uint64_t bar[4];
  __shared__ uint32_t tmem_ptr;
  for (int i = threadIdx.x; i < (issuers * 16384 + (N / 2) * 128) / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(&bar[i], 1);
    fence_mbar_init();
  }
  int cols = 32;
  while (cols < issuers * N) cols <<= 1;
  if (warp == 0) {
    tmem_alloc_pair(&tmem_ptr, cols);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = tmem_ptr;
  if (rank == 0 && warp < issuers && lane == 0) {
    const uint32_t idesc = umma_idesc_bf16(256, N);
    const uint64_t ad = umma_desc_sw128(smem_u32(smem + warp * 16384));
    const uint64_t bd = umma_desc_sw128(smem_u32(smem + issuers * 16384));
    const uint32_t d0 = tmem_base + warp * N;
    const long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_bf16_pair(d0, ad + 2 * k, bd + 2 * k, idesc, 1u);
    }
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&bar[warp])) : "memory");
    mbar_wait(&bar[warp], 0);
    const long long t1 = clock64();
    if (warp == 0) out[blockIdx.x >> 1] = t1 - t0;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  if (warp == 0) tmem_dealloc_pair(tmem_base, cols);
}

}  // namespace ug

extern "C" int ug_mma_microbench(ug_handle h, int N, int n_acc, int iters, int ctas_per_sm, int distinct_ab,
                                 double* cycles_per_mma) {
  if (!h || !cycles_per_mma || N % 16 || N < 16 || N > 256 || n_acc < 1 || n_acc * N > 512) return UG_EINVAL;
  using namespace ug;
  const int ctas = h->num_sms * ctas_per_sm;
  long long* dev = nullptr;
  if (cudaMalloc(&dev, sizeof(long long) * ctas) != cudaSuccess) return UG_ENOMEM;
  const size_t smem = 1024 + 4 * 16384 + 4 * (size_t)N * 128;
  cudaFuncSetAttribute(mma_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaMemset(dev, 0, sizeof(long long) * ctas);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  mma_bench_kernel<<<ctas, 128, smem>>>(N, n_acc, 10, distinct_ab, dev);  // warm-up
  cudaEventRecord(e0);
  mma_bench_kernel<<<ctas, 128, smem>>>(N, n_acc, iters, distinct_ab, dev);
  cudaEventRecord(e1);
  int rc = check_cuda(h, cudaGetLastError(), "mma_bench launch");
  if (rc == UG_OK) rc = check_cuda(h, cudaDeviceSynchronize(), "mma_bench");
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cycles_per_mma[1] = ms;  // wall time of the launch: tells whether co-resident CTAs overlapped
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (rc == UG_OK) {
    std::vector<long long> host(ctas);
    cudaMemcpy(host.data(), dev, sizeof(long long) * ctas, cudaMemcpyDeviceToHost);
    double s = 0;
    for (long long v : host) s += (double)v;
    *cycles_per_mma = s / ctas / ((double)iters * 4 * n_acc);
  }
  cudaFree(dev);
  return rc;
}

extern "C" int ug_mma_microbench2(ug_handle h, int N, int n_acc, int issuers, int iters, int ctas_per_sm,
                                  int a_off, int a_sbo, int acc_stride, double* out2) {
  if (!h || !out2 || N % 16 || N < 16 || N > 256 || n_acc < 1 || issuers < 1 || issuers > 4 ||
      issuers * n_acc * N * ctas_per_sm > 512 || a_off % 128 || a_off < 0 || a_off > 3072 || a_sbo % 128 ||
      a_sbo < 1024 || a_sbo > 1280 || acc_stride < 0 || (acc_stride > 0 && acc_stride < n_acc * N) ||
      ((issuers - 1) * acc_stride + n_acc * N) * ctas_per_sm > 512)
    return UG_EINVAL;
  using namespace ug;
  const int ctas = h->num_sms * ctas_per_sm;
  long long* dev = nullptr;
  if (cudaMalloc(&dev, sizeof(long long) * ctas) != cudaSuccess) return UG_ENOMEM;
  const size_t smem = 1024 + (size_t)issuers * 24576 + (size_t)N * 128;
  cudaFuncSetAttribute(mma_bench2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaMemset(dev, 0, sizeof(long long) * ctas);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  mma_bench2_kernel<<<ctas, 128, smem>>>(N, n_acc, issuers, 10, a_off, a_sbo, acc_stride, dev);
  cudaEventRecord(e0);
  mma_bench2_kernel<<<ctas, 128, smem>>>(N, n_acc, issuers, iters, a_off, a_sbo, acc_stride, dev);
  cudaEventRecord(e1);
  int rc = check_cuda(h, cudaGetLastError(), "mma_bench2 launch");
  if (rc == UG_OK) rc = check_cuda(h, cudaDeviceSynchronize(), "mma_bench2");
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  out2[1] = ms;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (rc == UG_OK) {
    std::vector<long long> host(ctas);
    cudaMemcpy(host.data(), dev, sizeof(long long) * ctas, cudaMemcpyDeviceToHost);
    double s = 0;
    for (long long v : host) s += (double)v;
    out2[0] = s / ctas / ((double)iters * 4 * n_acc);  // cycles per MMA of one issuer chain set
  }
  cudaFree(dev);
  return rc;
}

extern "C" int ug_mma_microbench_pair(ug_handle h, int N, int issuers, int iters, double* out2) {
  if (!h || !out2 || N % 16 || N < 32 || N > 256 || issuers < 1 || issuers > 4 || issuers * N > 512) return UG_EINVAL;
  using namespace ug;
  const int ctas = h->num_sms & ~1;
  long long* dev = nullptr;
  if (cudaMalloc(&dev, sizeof(long long) * ctas) != cudaSuccess) return UG_ENOMEM;
  const size_t smem = 1024 + (size_t)issuers * 16384 + (size_t)(N / 2) * 128;
  cudaFuncSetAttribute(mma_bench_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaMemset(dev, 0, sizeof(long long) * ctas);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ctas);
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  cudaError_t le = cudaLaunchKernelEx(&cfg, mma_bench_pair_kernel, N, issuers, 10, dev);  // warm-up
  cudaEventRecord(e0);
  if (le == cudaSuccess) le = cudaLaunchKernelEx(&cfg, mma_bench_pair_kernel, N, issuers, iters, dev);
  cudaEventRecord(e1);
  int rc = check_cuda(h, le != cudaSuccess ? le : cudaGetLastError(), "mma_bench_pair launch");
  if (rc == UG_OK) rc = check_cuda(h, cudaDeviceSynchronize(), "mma_bench_pair");
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  out2[1] = ms;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (rc == UG_OK) {
    std::vector<long long> host(ctas / 2);
    cudaMemcpy(host.data(), dev, sizeof(long long) * (ctas / 2), cudaMemcpyDeviceToHost);
    double s = 0;
    for (long long v : host) s += (double)v;
    out2[0] = s / (ctas / 2) / ((double)iters * 4);  // cycles per M=256 MMA of one issuer
  }
  cudaFree(dev);
  return rc;
}
