// Tensor-core (tcgen05 + TMEM) 256-point DFT of many real segments — the dense contraction inside the Welch
// periodogram (scipy.signal.welch defaults: nperseg = 256; signal_processor.py:260) and the "batched DFT against a
// twiddle matrix" the north_star assigns to the 5th-generation tensor cores:
//
//     D[m, c] = sum_j Z[m, j] * T[j, c],    m = segment (M = 128 per CTA),  j = sample 0..255 (K),  c = 0..255 (N)
//     T[j, c] = cos(2 pi j c / 256)          for c = 0..128      (real parts of bins 0..128)
//             = sin(2 pi j (c-128) / 256)    for c = 129..255    (imaginary parts of bins 1..127, sign dropped)
//
// so one M=128, N=256 accumulator tile (256 TMEM columns of fp32) holds the whole one-sided spectrum of 128 segments.
// Precision: kind::tf32 keeps 11 mantissa bits.  Two uses, two recipes:
//   tc_dft256<NT, true>   both operands split hi + lo (hi = fp32 with the low 13 mantissa bits cleared, lo = the residual),
//                         three MMAs per k-step: Zhi*Thi + Zlo*Thi + Zhi*Tlo -> 3.6e-6 of the row maximum (bpv_dft256_tc)
//   tc_dft256<NT, false>  one MMA per k-step straight from the fp32 segment tile (the tensor core truncates to tf32) against
//                         the tf32-rounded twiddles: |dX| <= 1.5e-3 * sum|z|, i.e. <= 3.4 % of the power of any bin that
//                         competes for the maximum (|X| >= rms X = 22.6 rms z).  Enough to SELECT the candidate bins; the
//                         Welch kernel below then decides among them in float64.
// Operand layout (no TMA, no swizzle): K-major "interleaved" canonical layout — 16-byte chunks of 4 consecutive k for
// one row; the 8 rows of a core matrix contiguous (128 B), 8-row groups SBO = 128 B apart, k-chunks LBO apart
// (LBO = rows * 16 B).  I.e. operand[chunk][row][4].  Tiles are written by ordinary threads (generic proxy) and made
// visible to the tensor core with fence.proxy.async; one thread issues the MMAs; tcgen05.commit -> mbarrier tells the
// CTA when the chunk buffers may be overwritten and when the accumulator is complete; tcgen05.ld (32 lanes x 32 columns
// per warp) brings each row's spectrum back to the thread that owns that segment.
#include <stdlib.h>
#include "common.cuh"

namespace bpv {

constexpr int TC_M = 128, TC_N = 256, TC_K = 256;
constexpr uint32_t TC_A_LBO = TC_M * 16, TC_B_LBO = TC_N * 16, TC_SBO = 128;
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) @4, a/b_format TF32 (2) @7/@10, K-major A and B,
// n_dim = N >> 3 @17, m_dim = M >> 4 @24
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TC_N >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);

// shared-memory plan (bytes).  The chunk area holds, per pipeline stage (2 stages): A hi | A lo | B hi | B lo of one
// 16-sample k block (split mode) or B of one 32-sample k block (single mode) — 24 KB / 32 KB per stage.
constexpr int TC_OFF_Z = 0;                                    // float [64 chunks][128 rows][4]   all of K, full fp32
constexpr int TC_OFF_CHUNK = TC_OFF_Z + TC_M * TC_K * 4;
constexpr int TC_STAGE = 32 * 1024;
constexpr int TC_OFF_TW = TC_OFF_CHUNK + 2 * TC_STAGE;         // double2 [256] exp(+2 pi i k / 256)
constexpr int TC_OFF_BAR = TC_OFF_TW + 256 * 16;               // 2 x uint64 mbarrier, uint32 tmem slot
constexpr int TC_SMEM = TC_OFF_BAR + 32;

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// cute::UMMA::SmemDescriptor, version 1, SWIZZLE_NONE: start >> 4 @0, LBO >> 4 @16, SBO >> 4 @32
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) |
         (1ull << 46);
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
               :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(TC_IDESC), "r"(accumulate) : "memory");
}
// same, with the N of the instruction chosen at run time (bin chunks narrower than 128 bins): n_dim = N >> 3 @17
__device__ __forceinline__ void tc_mma_tf32_n(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
               :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done)
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ float tc_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

// TMEM allocation (warp 0) + mbarrier init; every thread returns the TMEM base address.  Ends with a CTA barrier.
__device__ __forceinline__ uint32_t tc_setup(uint8_t* smem) {
  const uint32_t bar = tc_smem_u32(smem + TC_OFF_BAR), slot = bar + 16;
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(slot), "n"(TC_N) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar + 8) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  return *reinterpret_cast<volatile uint32_t*>(smem + TC_OFF_BAR + 16);
}
__device__ __forceinline__ void tc_teardown(uint32_t tmem) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "n"(TC_N) : "memory");
}

// The contraction: Z (full fp32, [64][128][4] in shared memory) x twiddles -> the CTA's TMEM accumulator.
// Called by all NT threads of the CTA; on return the accumulator is complete and visible (after_thread_sync done).
// Two-stage pipeline over k blocks: while the tensor core consumes stage s, the threads build stage s^1 (operand
// chunks from the float64 twiddle table); an mbarrier per stage (tcgen05.commit) says when a stage may be rebuilt.
template <int NT, bool SPLIT>
__device__ __forceinline__ void tc_dft256(uint8_t* smem, uint32_t tmem) {
  constexpr int KB = SPLIT ? 8 : 32;                   // samples per k block
  constexpr int CH = KB / 4;                           // 16-byte chunks per block
  constexpr int NB = TC_K / KB;
  constexpr int OFF_ALO = CH * TC_M * 16, OFF_BHI = 2 * CH * TC_M * 16, OFF_BLO = OFF_BHI + CH * TC_N * 16;
  static_assert((SPLIT ? OFF_BLO + CH * TC_N * 16 : CH * TC_N * 16) <= TC_STAGE, "stage too small");
  const int tid = threadIdx.x;
  const float4* Z = reinterpret_cast<const float4*>(smem + TC_OFF_Z);
  const double2* tw = reinterpret_cast<const double2*>(smem + TC_OFF_TW);
  const uint32_t bar = tc_smem_u32(smem + TC_OFF_BAR);
  const uint32_t z_addr = tc_smem_u32(smem + TC_OFF_Z);
  for (int kb = 0; kb < NB; ++kb) {
    const int st = kb & 1;
    uint8_t* stage = smem + TC_OFF_CHUNK + st * TC_STAGE;
    if (kb >= 2) tc_wait(bar + 8 * st, (uint32_t)(((kb - 2) >> 1) & 1));   // the MMAs of block kb-2 have consumed this stage
    if (SPLIT) {
      float4* Ahi = reinterpret_cast<float4*>(stage);
      float4* Alo = reinterpret_cast<float4*>(stage + OFF_ALO);
      for (int it = tid; it < CH * TC_M; it += NT) {
        const float4 z = Z[kb * CH * TC_M + it];
        const float4 h = make_float4(tc_hi(z.x), tc_hi(z.y), tc_hi(z.z), tc_hi(z.w));
        Ahi[it] = h;
        Alo[it] = make_float4(z.x - h.x, z.y - h.y, z.z - h.z, z.w - h.w);
      }
    }
    // B: the twiddle matrix rows j0 .. j0+3 of chunk c, column n, from the float64 table
    float4* Bhi = reinterpret_cast<float4*>(stage + (SPLIT ? OFF_BHI : 0));
    float4* Blo = reinterpret_cast<float4*>(stage + OFF_BLO);
    for (int it = tid; it < CH * TC_N; it += NT) {
      const int c = it / TC_N, n = it % TC_N;
      const int j0 = kb * KB + c * 4;
      const int kbin = n <= 128 ? n : n - 128;
      float hv[4], lv[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const double2 t = tw[((j0 + e) * kbin) & 255];
        const double v = n <= 128 ? t.x : t.y;
        if (SPLIT) { hv[e] = tc_hi((float)v); lv[e] = (float)(v - (double)hv[e]); }
        else {                                          // round to nearest tf32 (half an ulp of the 10-bit mantissa)
          hv[e] = __uint_as_float((__float_as_uint((float)v) + 0x1000u) & 0xFFFFE000u);
        }
      }
      Bhi[it] = make_float4(hv[0], hv[1], hv[2], hv[3]);
      if (SPLIT) Blo[it] = make_float4(lv[0], lv[1], lv[2], lv[3]);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
    __syncthreads();
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t sa = tc_smem_u32(stage);
#pragma unroll
      for (int ks = 0; ks < KB / 8; ++ks) {                         // UMMA K = 8 for tf32 = 2 chunks
        if (SPLIT) {
          const uint64_t dah = tc_desc(sa + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO), dal = tc_desc(sa + OFF_ALO + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO);
          const uint64_t dbh = tc_desc(sa + OFF_BHI + ks * 2 * TC_B_LBO, TC_B_LBO, TC_SBO), dbl = tc_desc(sa + OFF_BLO + ks * 2 * TC_B_LBO, TC_B_LBO, TC_SBO);
          tc_mma_tf32(tmem, dah, dbh, (kb | ks) != 0);
          tc_mma_tf32(tmem, dal, dbh, 1);
          tc_mma_tf32(tmem, dah, dbl, 1);
        } else {                                                    // A straight from the fp32 segment tile
          const uint64_t da = tc_desc(z_addr + (kb * CH + ks * 2) * TC_A_LBO, TC_A_LBO, TC_SBO);
          const uint64_t db = tc_desc(sa + ks * 2 * TC_B_LBO, TC_B_LBO, TC_SBO);
          tc_mma_tf32(tmem, da, db, (kb | ks) != 0);
        }
      }
      tc_commit(bar + 8 * st);
    }
  }
  // the last commit (stage (NB-1)&1) completes after every earlier MMA: accumulator done
  tc_wait(bar + 8 * ((NB - 1) & 1), (uint32_t)(((NB - 1) >> 1) & 1));
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// 32 consecutive accumulator columns of this thread's row (lane = 32 * warp + lane id)
__device__ __forceinline__ void tc_load32(uint32_t tmem, int col, float (&v)[32]) {
  const uint32_t addr = tmem + ((uint32_t)((threadIdx.x >> 5) * 32) << 16) + (uint32_t)col;
  uint32_t r[32];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
               "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                 "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                 "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(addr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Development / test entry: D[rows, 256] = Z[rows, 256] x T (see the header comment), one CTA per 128 rows.
__global__ void __launch_bounds__(TC_M, 1) dft256_tc_kernel(const float* __restrict__ z, int rows, float* __restrict__ d) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x;
  double2* tw = reinterpret_cast<double2*>(smem + TC_OFF_TW);
  for (int i = tid; i < 256; i += TC_M) { double s_, c_; sincospi((double)i / 128.0, &s_, &c_); tw[i] = make_double2(c_, s_); }
  float* Z = reinterpret_cast<float*>(smem + TC_OFF_Z);
  const long long row0 = (long long)blockIdx.x * TC_M;
  for (int m = 0; m < TC_M; ++m) {                       // coalesced: thread = sample pair
    const long long row = row0 + m;
    for (int j = tid; j < TC_K; j += TC_M) Z[(j >> 2) * (TC_M * 4) + m * 4 + (j & 3)] = row < rows ? z[row * TC_K + j] : 0.f;
  }
  const uint32_t tmem = tc_setup(smem);
  tc_dft256<TC_M, true>(smem, tmem);
  const long long row = row0 + tid;
  for (int c0 = 0; c0 < TC_N; c0 += 32) {
    float v[32];
    tc_load32(tmem, c0, v);
    if (row < rows)
      for (int i = 0; i < 32; ++i) d[row * TC_N + c0 + i] = v[i];
  }
  tc_teardown(tmem);
}


// (A Welch periodogram on this block — single-pass tf32 candidates + float64 decision, `welch_tc_kernel` — was built in
// round 1 and measured at 82 + 8 us against 76 us for the float64 shared-memory FFT kernel per 16 384 windows: the
// contraction is 23 % of it, the per-window front end and the float64 decision are the same scalar work the FFT kernel
// does.  It did not win and was removed in round 2; profiles/r1i_welch_tc_summary.md keeps the measurement.)

// ---------------------------------------------------------------------------------------------
// DFT_RFFT on the tensor cores (signal_processor.py:254-258: mags = 2 |rfft(y)| / n) for windows whose n valid samples
// fill the whole window (n == W: every steady-state window of a pipeline that resamples with INTERP_*, and every clean
// window otherwise), so that all signals of a launch share ONE twiddle matrix exp(-2 pi i j k / W) — the dense
// contraction [signals x W] . [W x 2F] the north_star assigns to tcgen05.
//   dft_tc_kernel   grid (signal tiles of 128, bin chunks of 128): K loop over 16-sample blocks, two-stage pipeline;
//                   A block = the float64 samples split hi/lo on the fly, B block = cos / sin columns from a float64
//                   table (running index j*k mod n per column), 6 tcgen05.mma (3xTF32) per block into 256 TMEM columns
//                   (re columns 0..127, im columns 128..255); epilogue: fp32 magnitudes 2 |X| / n straight into the spectrum rows.
//                   Rows with a non-finite sample are flagged num_bins = -2 for the float64 kernel.
//   dft_peak_kernel warp per signal: fs and the frequency axis, fp32 maximum, float64 re-evaluation of every bin within
//                   DFT_TC_BAND of it (the peak bin and value are float64 decisions, first-max rule).
// ---------------------------------------------------------------------------------------------
constexpr int DTC_THREADS = 512;
constexpr int DTC_KB = 16;                               // samples per k block
constexpr float DFT_TC_BAND = 1.0e-4f;                   // relative band below the fp32 maximum (3xTF32: 4e-6 of the maximum)
constexpr int DTC_STAGE = 48 * 1024;                     // A hi | A lo [4][128][4] + B hi | B lo [4][256][4]
constexpr int DTC_OFF_TW = 2 * DTC_STAGE;                // double2 [W]
__host__ __device__ inline int dtc_smem(int W) { return DTC_OFF_TW + W * 16 + 128 * 4 + 32; }

__global__ void __launch_bounds__(DTC_THREADS, 1) dft_tc_kernel(const double* __restrict__ proc_y, int W, long long nsig, int max_bins,
                                                                float* __restrict__ mags, int32_t* __restrict__ num_bins) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x;
  const int n = W, F = n / 2 + 1;
  float4* tw = reinterpret_cast<float4*>(smem + DTC_OFF_TW);   // exp(2 pi i j / n) pre-split: (cos_hi, sin_hi, cos_lo, sin_lo)
  int* bad = reinterpret_cast<int*>(smem + DTC_OFF_TW + W * 16);
  uint8_t* barp = smem + DTC_OFF_TW + W * 16 + 128 * 4;
  const uint32_t bar = tc_smem_u32(barp), slot = bar + 16;
  for (int i = tid; i < n; i += DTC_THREADS) {
    double s_, c_;
    sincospi(2.0 * (double)i / (double)n, &s_, &c_);
    const float ch_ = tc_hi((float)c_), sh_ = tc_hi((float)s_);
    tw[i] = make_float4(ch_, sh_, (float)(c_ - (double)ch_), (float)(s_ - (double)sh_));
  }
  if (tid < 128) bad[tid] = 0;
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(slot), "n"(TC_N) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar + 8) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(barp + 16);

  const long long sig0 = (long long)blockIdx.x * TC_M;
  const int k0 = blockIdx.y * 128;                        // first bin of this chunk
  // this thread's B item: bin kcol = k0 + bbin (column bbin = cos, column 128 + bbin = sin: consecutive lanes write
  // consecutive 16-byte slots), chunk bch of every k block (4 consecutive samples); running table index (j * kcol) mod n,
  // advanced past the other chunks' 12 samples per block
  const int bbin = tid & 127, bch = tid >> 7;
  const int kcol = k0 + bbin;
  const bool col_live = kcol < F;
  const int kstep = col_live ? kcol : 0;             // kcol <= n/2 for live columns: one conditional subtraction keeps idx < n
  const int kskip = (int)((12LL * kstep) % n);
  int idx = (int)((4LL * bch * kstep) % n);
  // this thread's A items: row arow, samples {2q, 2q+1} and {8+2q, 8+2q+1} of every 16-sample k block (q = tid & 3):
  // the four lanes of a row read 64 contiguous bytes per 16-byte vector load, so a warp-level load touches 8 rows x 2
  // full sectors instead of 32 scattered sectors (the per-row loads were the bottleneck: rows are 8 W bytes apart)
  const int arow = tid >> 2, aq = tid & 3;
  const long long asig = sig0 + arow;
  const double* ay = proc_y + (asig < nsig ? asig : 0) * W;
  const bool vec_ok = (W & 1) == 0 && (reinterpret_cast<uintptr_t>(proc_y) & 15) == 0;   // 16-byte aligned rows
  int mybad = 0;
  const int NB = (n + DTC_KB - 1) / DTC_KB;
  // software prefetch: the samples of the NEXT k block are requested before this block is converted and issued
  double cur[4], nxt[4];
  auto fetch = [&](int kb, double (&dst)[4]) {
#pragma unroll
    for (int hlf = 0; hlf < 2; ++hlf) {
      const int j = kb * DTC_KB + 8 * hlf + 2 * aq;
      if (asig < nsig && j + 1 < n && vec_ok) {
        const double2 v = *reinterpret_cast<const double2*>(ay + j);
        dst[2 * hlf] = v.x; dst[2 * hlf + 1] = v.y;
      } else {
        dst[2 * hlf] = (asig < nsig && j < n) ? ay[j] : 0.0;
        dst[2 * hlf + 1] = (asig < nsig && j + 1 < n) ? ay[j + 1] : 0.0;
      }
    }
  };
  fetch(0, cur);
  for (int kb = 0; kb < NB; ++kb) {
    const int st = kb & 1;
    uint8_t* stage = smem + st * DTC_STAGE;
    if (kb + 1 < NB) fetch(kb + 1, nxt);
    if (kb >= 2) tc_wait(bar + 8 * st, (uint32_t)(((kb - 2) >> 1) & 1));
    float4* Ahi = reinterpret_cast<float4*>(stage);
    float4* Alo = reinterpret_cast<float4*>(stage + 8192);
    float4* Bhi = reinterpret_cast<float4*>(stage + 16384);
    float4* Blo = reinterpret_cast<float4*>(stage + 32768);
    {
      float hv[4], lv[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const double v = cur[e];
        if (!isfinite(v)) mybad = 1;
        hv[e] = tc_hi((float)v);
        lv[e] = (float)(v - (double)hv[e]);
      }
      // samples 2q, 2q+1 -> chunk q >> 1, slots 2 (q & 1) ..; samples 8 + 2q .. -> chunk 2 + (q >> 1)
      float2* Ah2 = reinterpret_cast<float2*>(Ahi);
      float2* Al2 = reinterpret_cast<float2*>(Alo);
      const int o0 = (((aq >> 1) * TC_M + arow) << 1) + (aq & 1), o1 = (((2 + (aq >> 1)) * TC_M + arow) << 1) + (aq & 1);
      Ah2[o0] = make_float2(hv[0], hv[1]); Al2[o0] = make_float2(lv[0], lv[1]);
      Ah2[o1] = make_float2(hv[2], hv[3]); Al2[o1] = make_float2(lv[2], lv[3]);
    }
    {
      float4 t4[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        t4[e] = col_live ? tw[idx] : make_float4(0.f, 0.f, 0.f, 0.f);
        idx += kstep; if (idx >= n) idx -= n;
      }
      idx += kskip; if (idx >= n) idx -= n;            // the 12 samples of this block that the other chunks generate
      const int o = bch * TC_N + bbin;
      Bhi[o] = make_float4(t4[0].x, t4[1].x, t4[2].x, t4[3].x);
      Bhi[o + 128] = make_float4(t4[0].y, t4[1].y, t4[2].y, t4[3].y);
      Blo[o] = make_float4(t4[0].z, t4[1].z, t4[2].z, t4[3].z);
      Blo[o + 128] = make_float4(t4[0].w, t4[1].w, t4[2].w, t4[3].w);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t sa = tc_smem_u32(stage);
#pragma unroll
      for (int ks = 0; ks < DTC_KB / 8; ++ks) {
        const uint64_t dah = tc_desc(sa + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO), dal = tc_desc(sa + 8192 + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO);
        const uint64_t dbh = tc_desc(sa + 16384 + ks * 2 * TC_B_LBO, TC_B_LBO, TC_SBO), dbl = tc_desc(sa + 32768 + ks * 2 * TC_B_LBO, TC_B_LBO, TC_SBO);
        tc_mma_tf32(tmem, dah, dbh, (kb | ks) != 0);
        tc_mma_tf32(tmem, dal, dbh, 1);
        tc_mma_tf32(tmem, dah, dbl, 1);
      }
      tc_commit(bar + 8 * st);
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) cur[e] = nxt[e];
  }
  if (mybad) bad[arow] = 1;
  tc_wait(bar + 8 * ((NB - 1) & 1), (uint32_t)(((NB - 1) >> 1) & 1));
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  __syncthreads();                                         // bad[] complete
  if (tid < TC_M) {
    const long long sig = sig0 + tid;
    const bool rowbad = bad[tid] != 0;
    const float sc = 2.f / (float)n;
    for (int c32 = 0; c32 < 4; ++c32) {
      float re[32], im[32];
      __syncwarp();
      tc_load32(tmem, 32 * c32, re);
      tc_load32(tmem, 128 + 32 * c32, im);
      if (sig < nsig && !rowbad) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int k = k0 + 32 * c32 + i;
          if (k < F && k < max_bins) mags[sig * max_bins + k] = sc * sqrtf(re[i] * re[i] + im[i] * im[i]);
        }
      }
    }
    if (sig < nsig && rowbad && blockIdx.y == 0) num_bins[sig] = -2;     // the float64 kernel takes this window
    if (sig < nsig && !rowbad && blockIdx.y == 0) num_bins[sig] = -1;    // marker: coarse spectrum ready for dft_peak_kernel
  }
  tc_teardown(tmem);
}

// warp per signal; smem: double2 tw[W] shared by the CTA's warps.
// BAND: the peak is searched over the bins with band.lo <= k * fval <= band.hi; their fp32 maximum and count are taken over those
// bins alone.  The float64 values written back into the spectrum are those of the unbanded candidates, whatever the band.
template <bool BAND>
__global__ void __launch_bounds__(128) dft_peak_kernel(const double* __restrict__ proc_x, const double* __restrict__ proc_y, int W,
                                                       long long nsig, int max_bins, float* __restrict__ spec_f,
                                                       float* __restrict__ mags, int32_t* __restrict__ num_bins,
                                                       int32_t* __restrict__ peak_idx, double* __restrict__ peak_freq,
                                                       double* __restrict__ peak_mag, const PeakBand band) {
  extern __shared__ __align__(16) uint8_t psm[];
  double2* tw = reinterpret_cast<double2*>(psm);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n = W, F = n / 2 + 1;
  for (int i = tid; i < n; i += blockDim.x) { double s_, c_; sincospi(2.0 * (double)i / (double)n, &s_, &c_); tw[i] = make_double2(c_, s_); }
  __syncthreads();
  const long long sig = (long long)blockIdx.x * (blockDim.x >> 5) + wid;
  if (sig >= nsig || num_bins[sig] != -1) return;          // -2: float64 kernel; anything else: not ours
  const double* px = proc_x + sig * W;
  const double* py = proc_y + sig * W;
  // fs over the finite-x mask (Signal.get_fs); y is finite everywhere here
  int m = 0; double xfirst = 0.0, xlast = 0.0;
  for (int k0 = 0; k0 < W; k0 += 32) {
    const int k = k0 + lane;
    const double x = k < W ? px[k] : nan_f64();
    const unsigned bx = __ballot_sync(0xffffffffu, isfinite(x));
    if (bx) {
      const double xf = __shfl_sync(0xffffffffu, x, __ffs(bx) - 1), xl = __shfl_sync(0xffffffffu, x, 31 - __clz(bx));
      if (m == 0) xfirst = xf;
      xlast = xl;
    }
    m += __popc(bx);
  }
  const double fs = m >= 2 ? 1.0 / ((xlast - xfirst) / (double)(m - 1)) : nan_f64();
  if (!(n >= 2 && isfinite(fs))) {                         // guard signal_processor.py:252 -> empty spectrum
    if (lane == 0) { num_bins[sig] = 0; peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
    return;
  }
  const double fval = 1.0 / ((double)n * (1.0 / fs));      // rfftfreq(n, d=1/fs)[k] = k * (1/(n*d))
  float* row = mags + sig * max_bins;
  float cmax = -INFINITY; int cnt = 0;
  float bmax = -INFINITY; int cb = 0;                      // BAND: over the finite in-band bins
  for (int k = lane; k < F; k += 32) {
    const float v = row[k];
    if (isfinite(v)) { ++cnt; cmax = fmaxf(cmax, v); if (BAND && band.in((double)k * fval)) { ++cb; bmax = fmaxf(bmax, v); } }
    if (spec_f) spec_f[sig * max_bins + k] = (float)((double)k * fval);
  }
  for (int o = 16; o > 0; o >>= 1) { cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o)); cnt += __shfl_xor_sync(0xffffffffu, cnt, o); }
  if (BAND)
    for (int o = 16; o > 0; o >>= 1) { bmax = fmaxf(bmax, __shfl_xor_sync(0xffffffffu, bmax, o)); cb += __shfl_xor_sync(0xffffffffu, cb, o); }
  const float thr = cmax - DFT_TC_BAND * fabsf(cmax);
  const float thr_b = bmax - DFT_TC_BAND * fabsf(bmax);
  double best = -INFINITY; int bi = 0x7fffffff;
  for (int kk0 = 0; kk0 < F; kk0 += 32) {
    const int k = kk0 + lane;
    bool cand = false, cand_b = false;
    if (k < F) {
      const float v = row[k];
      cand = cnt >= 2 ? (isfinite(v) && v >= thr) : true;
      if (BAND) cand_b = band.in((double)k * fval) && (cb >= 2 ? (isfinite(v) && v >= thr_b) : true);
    }
    // BAND: mw = bins whose float64 value is written back (the unbanded candidates), mb = in-band candidates
    unsigned mk = __ballot_sync(0xffffffffu, cand || cand_b);
    const unsigned mw = BAND ? __ballot_sync(0xffffffffu, cand) : 0u, mb = BAND ? __ballot_sync(0xffffffffu, cand_b) : 0u;
    while (mk) {
      const int b = __ffs(mk) - 1, kc = kk0 + b;
      mk &= mk - 1;
      double re = 0.0, im = 0.0;
      int idx = (int)(((long long)lane * kc) % n);
      const int step = (int)((32LL * kc) % n);
      for (int j = lane; j < n; j += 32) {
        const double2 t = tw[idx];
        const double v = py[j];
        re = fma(v, t.x, re); im = fma(-v, t.y, im);
        idx += step; if (idx >= n) idx -= n;
      }
      re = warp_sum(re); im = warp_sum(im);
      const double mg = 2.0 * hypot(re, im) / (double)n;
      if (lane == 0 && (!BAND || ((mw >> b) & 1u))) row[kc] = (float)mg;
      if ((!BAND || ((mb >> b) & 1u)) && isfinite(mg) && (mg > best || (mg == best && kc < bi))) { best = mg; bi = kc; }
    }
  }
  if (lane == 0) {
    num_bins[sig] = F;
    if ((BAND ? cb : cnt) >= 2 && bi != 0x7fffffff) { peak_idx[sig] = bi; peak_freq[sig] = (double)bi * fval; peak_mag[sig] = best; }
    else { peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
  }
}

// ---------------------------------------------------------------------------------------------
// TMA-fed, warp-specialised variant of dft_tc_kernel (round 2).  The kernel above spends ~4x longer generating its B
// operand (table look-ups, hi / lo splits, 4 shared-memory stores per thread and k block) than the tensor core spends
// consuming it, and paces every k block with a CTA barrier.  The twiddle matrix depends only on n = W, so it is computed
// ONCE (dft_image_kernel, into the caller's workspace, kept across launches: a header remembers the n it was built for)
// as ready-made operand images — for every (bin chunk, k block) the 32 KB [B hi | B lo] block in exactly the K-major
// canonical shared-memory layout the UMMA descriptors expect.  Roles in the CTA (17 warps, no CTA barrier in the loop):
//   warps 0-15    A producers: float64 samples of k block kb -> hi / lo tf32 operand in A stage kb % 3, then
//                 fence.proxy.async + one mbarrier arrive per warp on fullA
//   warp 16       lane 0 is the TMA producer AND the MMA issuer: keeps the B images of the next 3 k blocks in flight
//                 (one cp.async.bulk = UBLKCP of 32 KB each, completing on fullB with expect_tx; 5-stage ring), waits
//                 fullA / fullB, issues the 6 tcgen05.mma of the block and commits them to emptyA / emptyB
// Waits are bounded: a barrier that never completes traps instead of hanging the GPU.
// ---------------------------------------------------------------------------------------------
// Ring stages of the A / B operands inside one 208 KB ring area: the B ring takes DTM_NSB images of this launch's size (32 KB at
// 128 bins per CTA, 18 KB at 72), the A ring (16 KB per k block) everything that is left — 3 stages at 128 bins, 7 at 72.
// The A stages are what hides the producer <-> tensor-core round trip (commit -> producers wake -> convert -> proxy fence ->
// arrive -> issue): with 3 stages a k block costs ~1 us however narrow the MMA is.
constexpr int DTM_NSB = 5, DTM_NSA_MIN = 3, DTM_NSA_MAX = 8;
constexpr int DTM_A_BYTES = 16 * 1024, DTM_B_BYTES = 32 * 1024;
constexpr int DTM_RING = DTM_NSA_MIN * DTM_A_BYTES + DTM_NSB * DTM_B_BYTES;
constexpr int DTM_OFF_BAD = DTM_RING;                       // int [128]
constexpr int DTM_OFF_BAR = DTM_OFF_BAD + 512;              // fullA[8] emptyA[8] fullB[5] emptyB[5] (u64 each) | tmem slot (u32)
constexpr int DTM_NBAR = 2 * DTM_NSA_MAX + 2 * DTM_NSB;
constexpr int DTM_SMEM = DTM_OFF_BAR + 8 * DTM_NBAR + 16;
constexpr int DTM_THREADS = DTC_THREADS + 32;               // 16 producer warps + the control warp
constexpr int DTM_PF = 4;                                   // A operand: k blocks of float64 samples held in registers
constexpr unsigned long long DTM_MAGIC = 0x62707644465431ULL;   // "bpvDFT1"

// Bin chunk width BC (bins per CTA, multiple of 8, <= 128): the MMA is M 128 x N 2*BC, the image of one (bin chunk, k block)
// is [B hi | B lo] = 2 x (4 k-chunks x 2*BC columns x 16 B) = 256 * BC bytes.  Whatever BC a launch picks, the chunks cover
// fewer than F + 128 bins.
__host__ __device__ inline long long dtc_image_bytes(int W) {
  const long long NB = (W + DTC_KB - 1) / DTC_KB, F = W / 2 + 1;
  return 256 + NB * 256 * (F + 128);                        // header (magic, n, BC) + images
}

// One CTA per (k block, bin chunk): 1024 operand items (chunk c, column col) of 4 consecutive samples each.
__global__ void __launch_bounds__(256) dft_image_kernel(int n, int BC, unsigned char* __restrict__ ws) {
  const unsigned long long* hdr = reinterpret_cast<const unsigned long long*>(ws);
  if (hdr[0] == DTM_MAGIC && hdr[1] == (unsigned long long)n && hdr[2] == (unsigned long long)BC) return;   // built by an earlier launch
  const int F = n / 2 + 1, NB = (n + DTC_KB - 1) / DTC_KB, N = 2 * BC;
  const int kb = blockIdx.x, bc = blockIdx.y;
  float4* Bhi = reinterpret_cast<float4*>(ws + 256 + ((long long)bc * NB + kb) * (256LL * BC));
  float4* Blo = Bhi + 4 * N;
  for (int it = threadIdx.x; it < 4 * N; it += blockDim.x) {
    const int c = it / N, col = it % N;
    const int kcol = bc * BC + (col < BC ? col : col - BC);
    float hv[4], lv[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = kb * DTC_KB + 4 * c + e;
      double v = 0.0;
      if (kcol < F && j < n) {
        const long long idx = ((long long)j * kcol) % n;
        double s_, c_;
        sincospi(2.0 * (double)idx / (double)n, &s_, &c_);
        v = col < BC ? c_ : s_;
      }
      hv[e] = tc_hi((float)v);
      lv[e] = (float)(v - (double)hv[e]);
    }
    Bhi[it] = make_float4(hv[0], hv[1], hv[2], hv[3]);
    Blo[it] = make_float4(lv[0], lv[1], lv[2], lv[3]);
  }
}
__global__ void dft_image_seal_kernel(int n, int BC, unsigned char* __restrict__ ws) {
  unsigned long long* hdr = reinterpret_cast<unsigned long long*>(ws);
  hdr[0] = DTM_MAGIC; hdr[1] = (unsigned long long)n; hdr[2] = (unsigned long long)BC;
}

__device__ __forceinline__ void tc_wait_bounded(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  const long long t0 = clock64();
  while (!done) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (!done && clock64() - t0 > 2000000000LL) __trap();   // ~1 s: a protocol error must not hang the device
  }
}
__device__ __forceinline__ void tc_bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}

__global__ void __launch_bounds__(DTM_THREADS, 1) dft_tc_tma_kernel(const double* __restrict__ proc_y, int W, long long nsig, int max_bins,
                                                                    int BC, const unsigned char* __restrict__ img,
                                                                    float* __restrict__ mags, int32_t* __restrict__ num_bins) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const int n = W, F = n / 2 + 1;
  int* bad = reinterpret_cast<int*>(smem + DTM_OFF_BAD);
  uint8_t* barp = smem + DTM_OFF_BAR;
  const uint32_t bar = tc_smem_u32(barp), slot = bar + 8 * DTM_NBAR;
  const uint32_t fullA = bar, emptyA = bar + 8 * DTM_NSA_MAX, fullB = bar + 16 * DTM_NSA_MAX, emptyB = fullB + 8 * DTM_NSB;
  const uint32_t b_stride = (256u * (uint32_t)BC + 1023u) & ~1023u;        // one B image (256 BC bytes), 1 KB aligned
  constexpr int NSB = DTM_NSB;
  int NSA = (DTM_RING - NSB * (int)b_stride) / DTM_A_BYTES;
  if (NSA > DTM_NSA_MAX) NSA = DTM_NSA_MAX;
  const int PREF = NSB - 2;
  const uint32_t off_b = (uint32_t)NSA * DTM_A_BYTES;                       // B ring behind the A ring
  if (tid < 128) bad[tid] = 0;
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(slot), "n"(TC_N) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    if (tid == 0) {
      for (int s_ = 0; s_ < DTM_NSA_MAX; ++s_) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(fullA + 8u * s_), "r"(DTC_THREADS / 32) : "memory");   // one arrive per producer warp
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(emptyA + 8u * s_) : "memory");
      }
      for (int s_ = 0; s_ < DTM_NSB; ++s_) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(fullB + 8u * s_) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(emptyB + 8u * s_) : "memory");
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(barp + 8 * DTM_NBAR);

  const long long sig0 = (long long)blockIdx.x * TC_M;
  const int k0 = blockIdx.y * BC;
  const int NB = (n + DTC_KB - 1) / DTC_KB;
  const uint32_t smem0 = tc_smem_u32(smem);
  if (wid == DTC_THREADS / 32) {
    // ---- control warp: TMA producer + MMA issuer (one thread)
    if (lane == 0) {
      const uint32_t img_bytes = 256u * (uint32_t)BC, b_lbo = 32u * (uint32_t)BC, b_lo_off = 128u * (uint32_t)BC;   // N = 2 BC columns
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)((2 * BC) >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
      const unsigned char* my_img = img + 256 + (long long)blockIdx.y * NB * img_bytes;
      for (int kb = 0; kb < PREF && kb < NB; ++kb)
        tc_bulk_load(smem0 + off_b + (uint32_t)(kb % NSB) * b_stride, my_img + (long long)kb * img_bytes, img_bytes,
                     fullB + 8u * (kb % NSB));
      for (int kb = 0; kb < NB; ++kb) {
        const int k2 = kb + PREF;
        if (k2 < NB) {
          const int s2 = k2 % NSB;
          if (k2 >= NSB) tc_wait_bounded(emptyB + 8u * s2, (uint32_t)((k2 / NSB - 1) & 1));    // its previous image has been consumed
          tc_bulk_load(smem0 + off_b + (uint32_t)s2 * b_stride, my_img + (long long)k2 * img_bytes, img_bytes, fullB + 8u * s2);
        }
        const int sa_ = kb % NSA, sb_ = kb % NSB;
        tc_wait_bounded(fullA + 8u * sa_, (uint32_t)((kb / NSA) & 1));
        tc_wait_bounded(fullB + 8u * sb_, (uint32_t)((kb / NSB) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sa = smem0 + (uint32_t)sa_ * DTM_A_BYTES, sb = smem0 + off_b + (uint32_t)sb_ * b_stride;
#pragma unroll
        for (int ks = 0; ks < DTC_KB / 8; ++ks) {
          const uint64_t dah = tc_desc(sa + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO), dal = tc_desc(sa + 8192 + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO);
          const uint64_t dbh = tc_desc(sb + ks * 2 * b_lbo, b_lbo, TC_SBO), dbl = tc_desc(sb + b_lo_off + ks * 2 * b_lbo, b_lbo, TC_SBO);
          tc_mma_tf32_n(tmem, dah, dbh, idesc, (kb | ks) != 0);
          tc_mma_tf32_n(tmem, dal, dbh, idesc, 1);
          tc_mma_tf32_n(tmem, dah, dbl, idesc, 1);
        }
        tc_commit(emptyA + 8u * sa_);
        tc_commit(emptyB + 8u * sb_);
      }
    }
  } else {
    // ---- producer warps: the A operand.  The float64 samples of the next DTM_PF - 1 k blocks are in flight in registers
    // while a block is converted.  (Measured alternatives, profiles/r2w_dft_tc.txt: one block ahead 78 us, four ahead 72 us;
    // deeper A or B rings change nothing; one signal row per thread with the warps taking k blocks in turn — fewer proxy
    // fences per warp, but one 128-byte line per thread instead of 64 bytes per 4 lanes — 93 us.)
    const int arow = tid >> 2, aq = tid & 3;
    const long long asig = sig0 + arow;
    const double* ay = proc_y + (asig < nsig ? asig : 0) * W;
    const bool vec_ok = (W & 1) == 0 && (reinterpret_cast<uintptr_t>(proc_y) & 15) == 0;
    int mybad = 0;
    double buf[DTM_PF][4];
    auto fetch = [&](int kb, double (&dst)[4]) {
#pragma unroll
      for (int hlf = 0; hlf < 2; ++hlf) {
        const int j = kb * DTC_KB + 8 * hlf + 2 * aq;
        if (asig < nsig && j + 1 < n && vec_ok) {
          const double2 v = *reinterpret_cast<const double2*>(ay + j);
          dst[2 * hlf] = v.x; dst[2 * hlf + 1] = v.y;
        } else {
          dst[2 * hlf] = (asig < nsig && j < n) ? ay[j] : 0.0;
          dst[2 * hlf + 1] = (asig < nsig && j + 1 < n) ? ay[j + 1] : 0.0;
        }
      }
    };
#pragma unroll
    for (int u = 0; u < DTM_PF - 1; ++u)
      if (u < NB) fetch(u, buf[u]);
    for (int kb0 = 0; kb0 < NB; kb0 += DTM_PF) {
#pragma unroll
      for (int u = 0; u < DTM_PF; ++u) {
        const int kb = kb0 + u;
        if (kb < NB) {
          if (kb + DTM_PF - 1 < NB) fetch(kb + DTM_PF - 1, buf[(u + DTM_PF - 1) % DTM_PF]);
          const int st = kb % NSA;
          uint8_t* stage = smem + st * DTM_A_BYTES;
          if (kb >= NSA) tc_wait_bounded(emptyA + 8u * st, (uint32_t)((kb / NSA - 1) & 1));      // block kb - NSA has been consumed
          float hv[4], lv[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const double v = buf[u][e];
            if (!isfinite(v)) mybad = 1;
            hv[e] = tc_hi((float)v);
            lv[e] = (float)(v - (double)hv[e]);
          }
          float2* Ah2 = reinterpret_cast<float2*>(stage);
          float2* Al2 = reinterpret_cast<float2*>(stage + 8192);
          const int o0 = (((aq >> 1) * TC_M + arow) << 1) + (aq & 1), o1 = (((2 + (aq >> 1)) * TC_M + arow) << 1) + (aq & 1);
          Ah2[o0] = make_float2(hv[0], hv[1]); Al2[o0] = make_float2(lv[0], lv[1]);
          Ah2[o1] = make_float2(hv[2], hv[3]); Al2[o1] = make_float2(lv[2], lv[3]);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
          __syncwarp();
          if (lane == 0) tc_arrive(fullA + 8u * st);
        }
      }
    }
    if (mybad) bad[arow] = 1;
  }
  // the commit of the last block completes when every MMA has: the accumulator is final
  tc_wait_bounded(emptyA + 8u * ((NB - 1) % NSA), (uint32_t)(((NB - 1) / NSA) & 1));
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  __syncthreads();                                         // bad[] complete
  if (tid < TC_M) {
    const long long sig = sig0 + tid;
    const bool rowbad = bad[tid] != 0;
    const float sc = 2.f / (float)n;
    for (int c32 = 0; 32 * c32 < BC; ++c32) {              // re columns [0, BC), im columns [BC, 2 BC); 256 columns are allocated
      float re[32], im[32];
      __syncwarp();
      tc_load32(tmem, 32 * c32, re);
      tc_load32(tmem, BC + 32 * c32, im);
      if (sig < nsig && !rowbad) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int k = k0 + 32 * c32 + i;
          if (32 * c32 + i < BC && k < F && k < max_bins) mags[sig * max_bins + k] = sc * sqrtf(re[i] * re[i] + im[i] * im[i]);
        }
      }
    }
    if (sig < nsig && rowbad && blockIdx.y == 0) num_bins[sig] = -2;     // the float64 kernel takes this window
    if (sig < nsig && !rowbad && blockIdx.y == 0) num_bins[sig] = -1;    // marker: coarse spectrum ready for dft_peak_kernel
  }
  tc_teardown(tmem);
}

// ---------------------------------------------------------------------------------------------
// Both operands by TMA (round 2, last step).  In dft_tc_tma_kernel the 16 producer warps convert the float64 samples of every
// k block into the hi / lo tf32 A operand while the tensor core waits: wait for the stage, convert, store, proxy fence, arrive
// — ~0.95 us per 16-sample block whatever the ring depths are (profiles/README.md), against 0.23 us of MMAs.  The split does
// not depend on the bin chunk, so it is done ONCE per launch by dft_split_kernel into ready-made A images (one 16 KB image
// per (128-signal tile, k block), the same canonical layout) in the caller's workspace; every CTA of a signal tile then
// fetches them with cp.async.bulk exactly like the twiddle images.  The CTA is three roles and no conversion:
//   warp 4, lane 0   TMA producer: A image + B image of k block kb into stage kb % NST (one mbarrier, expect_tx of both)
//   warp 5, lane 0   MMA issuer: waits the stage, 6 tcgen05.mma (3xTF32), tcgen05.commit releases the stage
//   warps 0-3        epilogue: tcgen05.ld of the 128 accumulator rows once the last commit has landed
// ---------------------------------------------------------------------------------------------
constexpr int DT2_THREADS = 192;
constexpr int DT2_NST_MAX = 8;
constexpr int DT2_RING = 208 * 1024;
constexpr int DT2_OFF_BAR = DT2_RING;                        // full[8] empty[8] done (u64 each) | tmem slot (u32)
constexpr int DT2_NBAR = 2 * DT2_NST_MAX + 1;
constexpr int DT2_SMEM = DT2_OFF_BAR + 8 * DT2_NBAR + 16;

__host__ __device__ inline long long dtc_split_bytes(int W, long long nsig) {
  const long long NB = (W + DTC_KB - 1) / DTC_KB, mt = (nsig + TC_M - 1) / TC_M;
  return mt * NB * DTM_A_BYTES + ((mt * TC_M * 4 + 255) / 256) * 256;      // A images | int bad[rows]
}

// thread = (signal row, chunk of 4 consecutive samples): the lanes of a warp take 32 consecutive rows of one chunk, so the
// image stores are coalesced (512 contiguous bytes per warp) and every lane reads exactly one 32-byte sector of its row
__global__ void __launch_bounds__(256) dft_split_kernel(const double* __restrict__ proc_y, int W, long long nsig,
                                                        unsigned char* __restrict__ a_img, int* __restrict__ bad) {
  const int NB = (W + DTC_KB - 1) / DTC_KB, NC = NB * 4;
  const long long rows = ((nsig + TC_M - 1) / TC_M) * TC_M;
  const long long item = (long long)blockIdx.x * 256 + threadIdx.x;
  const long long rblk = item / (32LL * NC);
  const int within = (int)(item - rblk * (32LL * NC));
  const int g = within >> 5, lr = within & 31;
  const long long row = rblk * 32 + lr;
  if (row >= rows) return;
  double v[4] = {0.0, 0.0, 0.0, 0.0};
  if (row < nsig) {
    const double* y = proc_y + row * W;
    const int j = 4 * g;
    if (j + 3 < W && (W & 1) == 0 && (reinterpret_cast<uintptr_t>(proc_y) & 15) == 0) {
      const double2 p0 = *reinterpret_cast<const double2*>(y + j), p1 = *reinterpret_cast<const double2*>(y + j + 2);
      v[0] = p0.x; v[1] = p0.y; v[2] = p1.x; v[3] = p1.y;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) if (j + e < W) v[e] = y[j + e];
    }
  }
  float hv[4], lv[4];
  bool isbad = false;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    isbad |= !isfinite(v[e]);
    hv[e] = tc_hi((float)v[e]);
    lv[e] = (float)(v[e] - (double)hv[e]);
  }
  const long long mt = row / TC_M;
  const int r = (int)(row % TC_M), kb = g >> 2, c = g & 3;
  float4* img = reinterpret_cast<float4*>(a_img + (mt * NB + kb) * DTM_A_BYTES);
  img[c * TC_M + r] = make_float4(hv[0], hv[1], hv[2], hv[3]);
  img[4 * TC_M + c * TC_M + r] = make_float4(lv[0], lv[1], lv[2], lv[3]);
  if (isbad) bad[row] = 1;                                   // zeroed by the launcher (cudaMemsetAsync) before this kernel
}

__global__ void __launch_bounds__(DT2_THREADS, 1) dft_tc_tma2_kernel(int W, long long nsig, int max_bins, int BC,
                                                                     const unsigned char* __restrict__ a_img, const int* __restrict__ bad,
                                                                     const unsigned char* __restrict__ img,
                                                                     float* __restrict__ mags, int32_t* __restrict__ num_bins) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const int n = W, F = n / 2 + 1;
  uint8_t* barp = smem + DT2_OFF_BAR;
  const uint32_t bar = tc_smem_u32(barp), slot = bar + 8 * DT2_NBAR;
  const uint32_t full = bar, empty = bar + 8 * DT2_NST_MAX, done = bar + 16 * DT2_NST_MAX;
  const uint32_t img_bytes = 256u * (uint32_t)BC;
  const uint32_t stage_bytes = DTM_A_BYTES + ((img_bytes + 1023u) & ~1023u);
  int NST = DT2_RING / (int)stage_bytes;
  if (NST > DT2_NST_MAX) NST = DT2_NST_MAX;
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(slot), "n"(TC_N) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    if (tid == 0) {
      for (int s_ = 0; s_ < 2 * DT2_NST_MAX + 1; ++s_)
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar + 8u * s_) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(barp + 8 * DT2_NBAR);

  const long long sig0 = (long long)blockIdx.x * TC_M;
  const int k0 = blockIdx.y * BC;
  const int NB = (n + DTC_KB - 1) / DTC_KB;
  const uint32_t smem0 = tc_smem_u32(smem);
  if (wid == 4) {
    if (lane == 0) {                                         // ---- TMA producer
      const unsigned char* my_a = a_img + (long long)blockIdx.x * NB * DTM_A_BYTES;
      const unsigned char* my_b = img + 256 + (long long)blockIdx.y * NB * img_bytes;
      for (int kb = 0; kb < NB; ++kb) {
        const int s_ = kb % NST;
        if (kb >= NST) tc_wait_bounded(empty + 8u * s_, (uint32_t)((kb / NST - 1) & 1));       // the MMAs of block kb - NST have read the stage
        const uint32_t dst = smem0 + (uint32_t)s_ * stage_bytes, fb = full + 8u * s_;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(fb), "r"((uint32_t)DTM_A_BYTES + img_bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(dst), "l"(my_a + (long long)kb * DTM_A_BYTES), "r"((uint32_t)DTM_A_BYTES), "r"(fb) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(dst + (uint32_t)DTM_A_BYTES), "l"(my_b + (long long)kb * img_bytes), "r"(img_bytes), "r"(fb) : "memory");
      }
    }
  } else if (wid == 5) {
    if (lane == 0) {                                         // ---- MMA issuer
      const uint32_t b_lbo = 32u * (uint32_t)BC, b_lo_off = 128u * (uint32_t)BC;   // N = 2 BC columns
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)((2 * BC) >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
      for (int kb = 0; kb < NB; ++kb) {
        const int s_ = kb % NST;
        tc_wait_bounded(full + 8u * s_, (uint32_t)((kb / NST) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sa = smem0 + (uint32_t)s_ * stage_bytes, sb = sa + (uint32_t)DTM_A_BYTES;
#pragma unroll
        for (int ks = 0; ks < DTC_KB / 8; ++ks) {
          const uint64_t dah = tc_desc(sa + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO), dal = tc_desc(sa + 8192 + ks * 2 * TC_A_LBO, TC_A_LBO, TC_SBO);
          const uint64_t dbh = tc_desc(sb + ks * 2 * b_lbo, b_lbo, TC_SBO), dbl = tc_desc(sb + b_lo_off + ks * 2 * b_lbo, b_lbo, TC_SBO);
          tc_mma_tf32_n(tmem, dah, dbh, idesc, (kb | ks) != 0);
          tc_mma_tf32_n(tmem, dal, dbh, idesc, 1);
          tc_mma_tf32_n(tmem, dah, dbl, idesc, 1);
        }
        tc_commit(empty + 8u * s_);
      }
      tc_commit(done);                                       // arrives when every MMA issued so far has completed
    }
  }
  tc_wait_bounded(done, 0u);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (tid < TC_M) {
    const long long sig = sig0 + tid;
    const bool rowbad = bad[sig] != 0;                       // bad[] covers the padded rows of the last tile
    const float sc = 2.f / (float)n;
    for (int c32 = 0; 32 * c32 < BC; ++c32) {
      float re[32], im[32];
      __syncwarp();
      tc_load32(tmem, 32 * c32, re);
      tc_load32(tmem, BC + 32 * c32, im);
      if (sig < nsig && !rowbad) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int k = k0 + 32 * c32 + i;
          if (32 * c32 + i < BC && k < F && k < max_bins) mags[sig * max_bins + k] = sc * sqrtf(re[i] * re[i] + im[i] * im[i]);
        }
      }
    }
    if (sig < nsig && rowbad && blockIdx.y == 0) num_bins[sig] = -2;     // the float64 kernel takes this window
    if (sig < nsig && !rowbad && blockIdx.y == 0) num_bins[sig] = -1;    // marker: coarse spectrum ready for dft_peak_kernel
  }
  tc_teardown(tmem);
}

long long dft_tc_split_bytes(int W, long long nsig) { return dtc_split_bytes(W, nsig); }
long long dft_tc_image_bytes(int W) { return dtc_image_bytes(W); }

// image_ws: caller-owned, persistent device memory of dft_tc_image_bytes(W) bytes (zero-initialised once) for the TMA-fed
// kernel, or NULL for the kernel that generates its operands itself.  BPV_DFT_TMA=0 forces the latter (measurement switch).
int launch_dft_tc(const double* proc_x, const double* proc_y, int W, long long nsig, int max_bins, float* spec_f, float* mags,
                  int32_t* num_bins, int32_t* peak_idx, double* peak_freq, double* peak_mag, void* image_ws, void* split_ws,
                  bool banded, PeakBand band, cudaStream_t st) {
  const int smem = dtc_smem(W), smem_p = W * 16;
  if (int rc = ensure_dyn_smem(banded ? (const void*)dft_peak_kernel<true> : (const void*)dft_peak_kernel<false>, smem_p)) return rc;
  const int F = W / 2 + 1;
  dim3 grid((unsigned)((nsig + TC_M - 1) / TC_M), (unsigned)((F + 127) / 128));
  const char* env = getenv("BPV_DFT_TMA");
  if (image_ws && !(env && env[0] == '0')) {
    if (int rc = ensure_dyn_smem((const void*)dft_tc_tma_kernel, DTM_SMEM)) return rc;
    const int NB = (W + DTC_KB - 1) / DTC_KB;
    // bins per CTA: one CTA per SM (209 KB of shared memory), so the launch costs waves x (MMA time ~ 2 BC columns + the
    // per-block operand conversion, ~64 columns' worth).  2048 signals x 601 bins: 16 x 5 CTAs of 128 bins leave 68 SMs idle,
    // 16 x 9 CTAs of 72 bins fill 144 of the 148 (BPV_DFT_BC overrides: measurement switch).
    static int sms = 0;
    if (sms == 0) {
      int dev = 0;
      cudaGetDevice(&dev);
      if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    int BC = 128;
    {
      long long best = -1;
      for (int bc = 16; bc <= 128; bc += 8) {
        const long long ctas = (long long)grid.x * ((F + bc - 1) / bc);
        const long long cost = ((ctas + sms - 1) / sms) * (2 * bc + 64);
        if (best < 0 || cost < best || (cost == best && bc > BC)) { best = cost; BC = bc; }
      }
      const char* ebc = getenv("BPV_DFT_BC");
      if (ebc && atoi(ebc) >= 16 && atoi(ebc) <= 128 && atoi(ebc) % 8 == 0) BC = atoi(ebc);
    }
    grid.y = (unsigned)((F + BC - 1) / BC);
    dft_image_kernel<<<dim3((unsigned)NB, grid.y), 256, 0, st>>>(W, BC, (unsigned char*)image_ws);
    if (int rc = check_launch("dft_image_kernel")) return rc;
    dft_image_seal_kernel<<<1, 1, 0, st>>>(W, BC, (unsigned char*)image_ws);
    if (int rc = check_launch("dft_image_seal_kernel")) return rc;
    const char* esp = getenv("BPV_DFT_SPLIT");               // BPV_DFT_SPLIT=0: convert the samples inside the kernel (measurement switch)
    if (split_ws && !(esp && esp[0] == '0')) {
      if (int rc = ensure_dyn_smem((const void*)dft_tc_tma2_kernel, DT2_SMEM)) return rc;
      const long long mt = (nsig + TC_M - 1) / TC_M, rows = mt * TC_M;
      unsigned char* a_img = (unsigned char*)split_ws;
      int* bad = (int*)(a_img + mt * NB * DTM_A_BYTES);
      cudaError_t e = cudaMemsetAsync(bad, 0, (size_t)rows * sizeof(int), st);
      if (e != cudaSuccess) { set_error("dft split: cudaMemsetAsync: %s", cudaGetErrorString(e)); return (int)e; }
      const long long items = rows * NB * 4;
      dft_split_kernel<<<(unsigned)((items + 255) / 256), 256, 0, st>>>(proc_y, W, nsig, a_img, bad);
      if (int rc = check_launch("dft_split_kernel")) return rc;
      dft_tc_tma2_kernel<<<grid, DT2_THREADS, DT2_SMEM, st>>>(W, nsig, max_bins, BC, a_img, bad, (const unsigned char*)image_ws, mags, num_bins);
      if (int rc = check_launch("dft_tc_tma2_kernel")) return rc;
    } else {
      dft_tc_tma_kernel<<<grid, DTM_THREADS, DTM_SMEM, st>>>(proc_y, W, nsig, max_bins, BC, (const unsigned char*)image_ws, mags, num_bins);
      if (int rc = check_launch("dft_tc_tma_kernel")) return rc;
    }
  } else {
    if (int rc = ensure_dyn_smem((const void*)dft_tc_kernel, smem)) return rc;
    dft_tc_kernel<<<grid, DTC_THREADS, smem, st>>>(proc_y, W, nsig, max_bins, mags, num_bins);
    if (int rc = check_launch("dft_tc_kernel")) return rc;
  }
  if (banded)
    dft_peak_kernel<true><<<(unsigned)((nsig + 3) / 4), 128, smem_p, st>>>(proc_x, proc_y, W, nsig, max_bins, spec_f, mags, num_bins,
                                                                           peak_idx, peak_freq, peak_mag, band);
  else
    dft_peak_kernel<false><<<(unsigned)((nsig + 3) / 4), 128, smem_p, st>>>(proc_x, proc_y, W, nsig, max_bins, spec_f, mags, num_bins,
                                                                            peak_idx, peak_freq, peak_mag, band);
  return check_launch("dft_peak_kernel");
}

}  // namespace bpv

extern "C" int bpv_dft256_tc(const float* z, int32_t rows, float* d, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(z && d && rows >= 0, BPV_E_INVALID, "bpv_dft256_tc: bad arguments");
  if (rows == 0) return 0;
  if (int rc = ensure_dyn_smem((const void*)dft256_tc_kernel, TC_SMEM)) return rc;
  dft256_tc_kernel<<<(rows + TC_M - 1) / TC_M, TC_M, TC_SMEM, (cudaStream_t)stream>>>(z, rows, d);
  return check_launch("bpv_dft256_tc");
}
