// Shared helpers for libbpv (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/bpv.h"

namespace bpv {

void set_error(const char* fmt, ...);
// Opt `kernel` into `bytes` of dynamic shared memory on the current device (api.cu); 0 or a CUDA error code.
int ensure_dyn_smem(const void* kernel, size_t bytes, bool max_carveout = false);

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

#define BPV_REQUIRE(cond, code, ...)        \
  do {                                      \
    if (!(cond)) {                          \
      bpv::set_error(__VA_ARGS__);          \
      return (code);                        \
    }                                       \
  } while (0)

__device__ __forceinline__ double nan_f64() { return __longlong_as_double(0x7ff8000000000000LL); }

// Search range of a peak: Signal.get_peak(min_x, max_x) (signal_data.py:65-70) with explicit bounds.  A bin or lag is
// eligible iff lo <= x <= hi for the float64 x the kernel reports for it.  The peak kernels take it as a template switch
// BAND: the BAND = false instantiations are the unbanded search of process() and never read the bounds.
struct PeakBand {
  double lo, hi;
  __device__ __forceinline__ bool in(double x) const { return lo <= x && x <= hi; }
};
// (-inf, +inf) selects the unbanded kernels; the entry points reject NaN bounds before calling this
inline bool band_limits(double lo, double hi) { return !(lo == -INFINITY && hi == INFINITY); }

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of a double; every thread gets the result.  `red` = >= 33 doubles of smem.
__device__ __forceinline__ double block_sum(double v, double* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    double t = lane < nw ? red[lane] : 0.0;
    t = warp_sum(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

}  // namespace bpv
