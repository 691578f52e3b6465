// Development hooks (libugnet_dev.so only; declared in include/ugnet_dev.h): per-role cycle counters of the conv
// kernels.  Not part of the product library.
#include <vector>
#include "engine.h"
#include "../../include/ugnet_dev.h"

using namespace ug;

extern "C" {

int ug_conv_profile(ug_handle h, const ug_conv_desc* d, void* stream, double* out10) {
  if (!h || !d || !out10) return UG_EINVAL;
  DeviceGuard guard(h);
  ConvLaunch L;
  int rc = conv_prepare(h, d, &L);
  if (rc != UG_OK) return rc;
  if (L.kernel != ConvKernel::Persistent) return set_error(h, UG_EINVAL, "conv_profile: persistent variant only");
  const int ctas = (int)L.grid.x;
  long long* dev = nullptr;
  rc = check_cuda(h, cudaMalloc(&dev, sizeof(long long) * 8 * ctas), "cudaMalloc(prof)");
  if (rc != UG_OK) return rc;
  cudaMemset(dev, 0, sizeof(long long) * 8 * ctas);
  L.p.prof = dev;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  rc = conv_launch(h, &L, s);
  if (rc == UG_OK) rc = check_cuda(h, cudaStreamSynchronize(s), "conv_profile sync");
  std::vector<long long> host(8 * (size_t)ctas);
  if (rc == UG_OK) rc = check_cuda(h, cudaMemcpy(host.data(), dev, host.size() * sizeof(long long), cudaMemcpyDeviceToHost), "prof copy");
  cudaFree(dev);
  if (rc != UG_OK) return rc;
  for (int j = 0; j < 8; ++j) {
    double a = 0;
    for (int c = 0; c < ctas; ++c) a += (double)host[c * 8 + j];
    out10[j] = a / ctas;
  }
  out10[8] = ctas;
  out10[9] = (double)((L.p.m_tiles * (long long)L.p.n_tiles + ctas - 1) / ctas);
  return UG_OK;
}

int ug_conv_profile16(ug_handle h, const ug_conv_desc* d, void* stream, double* out16) {
  if (!h || !d || !out16) return UG_EINVAL;
  DeviceGuard guard(h);
  ConvLaunch L;
  int rc = conv_prepare(h, d, &L);
  if (rc != UG_OK) return rc;
  if (L.kernel != ConvKernel::Multi && L.kernel != ConvKernel::MultiPair)
    return set_error(h, UG_EINVAL, "conv_profile16: multi-issuer variant only");
  const int ctas = (int)L.grid.x;
  long long* dev = nullptr;
  rc = check_cuda(h, cudaMalloc(&dev, sizeof(long long) * 16 * ctas), "cudaMalloc(prof)");
  if (rc != UG_OK) return rc;
  cudaMemset(dev, 0, sizeof(long long) * 16 * ctas);
  L.p.prof = dev;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  rc = conv_launch(h, &L, s);
  if (rc == UG_OK) rc = check_cuda(h, cudaStreamSynchronize(s), "conv_profile16 sync");
  std::vector<long long> host(16 * (size_t)ctas);
  if (rc == UG_OK) rc = check_cuda(h, cudaMemcpy(host.data(), dev, host.size() * sizeof(long long), cudaMemcpyDeviceToHost), "prof copy");
  cudaFree(dev);
  if (rc != UG_OK) return rc;
  for (int j = 0; j < 16; ++j) {
    double a = 0;
    for (int c = 0; c < ctas; ++c) a += (double)host[c * 16 + j];
    // (CTA pairs: only the leader CTAs have issuers, slots 4-11)
    out16[j] = a / ((L.kernel == ConvKernel::MultiPair && j >= 4 && j < 12) ? ctas / 2 : ctas);
  }
  return UG_OK;
}

}  // extern "C"
