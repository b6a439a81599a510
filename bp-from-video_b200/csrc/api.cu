// libbpv: error plumbing + version.
#include <stdarg.h>
#include <map>
#include <mutex>
#include <utility>
#include "common.cuh"

namespace bpv {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a property of (kernel, device): remember what each pair was raised
// to, so that repeated launches skip the driver call and a host process that drives several GPUs (or several
// threads) still configures every one of them.
int ensure_dyn_smem(const void* kernel, size_t bytes, bool max_carveout) {
  if (bytes <= 48 * 1024 && !max_carveout) return 0;
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> raised;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { set_error("cudaGetDevice: %s", cudaGetErrorString(e)); return (int)e; }
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = raised[{kernel, dev}];
  if (bytes <= have) return 0;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && max_carveout) e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%zu B of dynamic shared memory): %s", bytes, cudaGetErrorString(e)); return (int)e; }
  have = bytes;
  return 0;
}
}  // namespace bpv

extern "C" int bpv_version(void) { return BPV_VERSION; }
extern "C" const char* bpv_last_error(void) { return bpv::g_err; }
extern "C" int bpv_sizeof_window_params(void) { return (int)sizeof(bpv_window_params); }

// L2 -> DRAM fetch granularity hint (32/64/128 B).  ROI rows are short, unaligned spans: a smaller
// granularity cuts the DRAM over-fetch around every row.  Device-wide limit of the primary context.
extern "C" int bpv_set_l2_fetch_granularity(int bytes) {
  cudaError_t e = cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)bytes);
  if (e != cudaSuccess) { bpv::set_error("cudaDeviceSetLimit(L2 fetch granularity): %s", cudaGetErrorString(e)); return (int)e; }
  return 0;
}
extern "C" int bpv_get_l2_fetch_granularity(void) {
  size_t v = 0;
  if (cudaDeviceGetLimit(&v, cudaLimitMaxL2FetchGranularity) != cudaSuccess) return -1;
  return (int)v;
}


// ---- FMA throughput probe (bench.py: measured FP64 / FP32 peaks for the roofline of the filter / spectrum families) ----
namespace bpv {
template <typename T>
__global__ void __launch_bounds__(256) probe_fma_kernel(long long iters, T* sink) {
  T a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = (T)(threadIdx.x + i) * (T)1e-3;
  const T m = (T)0.999999, c = (T)1e-7;
  for (long long it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = fma(a[i], m, c);
    }
  }
  T sres = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) sres += a[i];
  if (!(sres == sres)) *sink = sres;      // never true: keeps the chain alive
}
}  // namespace bpv

extern "C" int64_t bpv_probe_fma(int32_t dtype, int64_t iters, int32_t blocks, void* sink, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(sink && iters > 0 && blocks > 0 && (dtype == 0 || dtype == 1), BPV_E_INVALID, "bpv_probe_fma: bad arguments");
  if (dtype == 1) probe_fma_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>(iters, (double*)sink);
  else probe_fma_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>(iters, (float*)sink);
  if (int rc = check_launch("bpv_probe_fma")) return -(int64_t)rc;
  return (int64_t)blocks * 256 * iters * 32;
}
