// PGRAM_WELCH warp-per-signal kernel body (moved out of spectrum.cu so that a second translation unit can instantiate it).
#pragma once
#include "filters.cuh"

namespace bpv {

__device__ __forceinline__ double shfl_dd(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// ---------------------------------------------------------------------------------------------
// PGRAM_WELCH fast kernel: one WARP per signal, no CTA barrier after the shared twiddle table is built.
// scipy.signal.welch(y, fs) with every default (signal_processor.py:260): periodic Hann, nperseg = min(256, n),
// 50 % overlap, per-segment mean removal, one-sided density, mean over segments.  In steady state (n >= 256) a
// segment is a 256-point radix-2 FFT held in the warp's shared-memory slice (4 butterflies per lane per stage,
// __syncwarp between stages); shorter windows (warm-up) use a warp-level direct DFT with their own twiddles.
// The CTA-per-signal version spent its time in ~25 __syncthreads with little work between them (197 us per
// 16 384 signals); this one is ~1 k warp instructions per signal.
// smem: CTA table tw[256] (cos, sin) | per warp: ys[W] | buf[576]   (windows shorter than 256 samples are ONE segment of
// nperseg = n: their windowed segment overwrites ys in place and their <= 128 bins stay in registers)
// ---------------------------------------------------------------------------------------------
constexpr int WELCH_WPB = 4;
constexpr int WELCH_MINB = 5;          // 96 registers; 6 CTAs per SM (80 registers, small spills) measured no faster: the kernel
                                       // is bound by shared-memory wavefronts (64 % of peak), not by occupancy
__host__ __device__ inline int welch_warp_doubles(int W) { return W + 576; }
// FFT buffer index padding: one spare complex slot per 8 keeps the strided accesses of the late passes and the
// 4-element groups of the last pass on distinct banks
__device__ __forceinline__ int wpad(int e) { return e + (e >> 3); }
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
// d * conj(t) for a unit twiddle t = (cos, sin): multiplication by exp(-i * angle)
__device__ __forceinline__ double2 cmulc(double2 d, double2 t) {
  return make_double2(fma(d.x, t.x, d.y * t.y), fma(d.y, t.x, -(d.x * t.y)));
}
// Two fused radix-2 decimation-in-frequency stages (spans 2Q and Q) of a 256-point FFT held in shared memory:
// each lane owns two groups of four elements i, i+Q, i+2Q, i+3Q (i mod 4Q < Q).  Natural-order input, after the four
// passes Q = 64, 16, 4, 1 the output is in bit-reversed order.  Twiddles: A = W_4Q^p, -iA = W_4Q^(p+Q), C = W_2Q^p with
// p = i mod Q, read from the CTA's table tw[k] = exp(+2 pi i k / 256).
template <int Q, int GROUPS = 2>      // GROUPS x 32 groups of four elements: 2 for 256 points, 1 for 128
__device__ __forceinline__ void welch_fft_pass(double2* __restrict__ fz, const double2* __restrict__ tw, int lane) {
#pragma unroll
  for (int j = 0; j < GROUPS; ++j) {
    const int g = lane + 32 * j;
    const int pq = g & (Q - 1);
    const int i = (g / Q) * (4 * Q) + pq;
    const int a0 = wpad(i), a1 = wpad(i + Q), a2 = wpad(i + 2 * Q), a3 = wpad(i + 3 * Q);
    const double2 e0 = fz[a0], e1 = fz[a1], e2 = fz[a2], e3 = fz[a3];
    const double2 t0 = cadd(e0, e2), t1 = cadd(e1, e3);
    double2 t2 = csub(e0, e2), t3 = csub(e1, e3);
    if (Q > 1) {
      const double2 A = tw[pq * (64 / Q)];
      t2 = cmulc(t2, A);
      t3 = cmulc(t3, A);
    }
    t3 = make_double2(t3.y, -t3.x);                 // * (-i)
    const double2 o0 = cadd(t0, t1), o2 = cadd(t2, t3);
    double2 o1 = csub(t0, t1), o3 = csub(t2, t3);
    if (Q > 1) {
      const double2 C2 = tw[pq * (128 / Q)];
      o1 = cmulc(o1, C2);
      o3 = cmulc(o3, C2);
    }
    fz[a0] = o0; fz[a1] = o1; fz[a2] = o2; fz[a3] = o3;
  }
  __syncwarp();
}

// The kernel's body as a device function of (CTA index, shared memory): welch_warp_kernel (spectrum.cu) is a CTA of four such
// warps; welch_xcorr_kernel (welch_xcorr.cu) interleaves CTAs of this role with cross-correlation CTAs in one grid.
// BAND: the peak is searched over the bins with band.lo <= k * fval <= band.hi only (common.cuh PeakBand).
template <bool BAND = false>
__device__ __forceinline__ void welch_warp_body(unsigned blk, double* __restrict__ sm, const double* __restrict__ proc_x,
                                                const double* __restrict__ proc_y, const bpv_window_params& p, int max_bins,
                                                long long nsig, int only_flagged, float* __restrict__ spec_f,
                                                float* __restrict__ spec_mag, int32_t* __restrict__ num_bins,
                                                int32_t* __restrict__ peak_idx, double* __restrict__ peak_freq,
                                                double* __restrict__ peak_mag, const PeakBand band = PeakBand{}) {
  const int W = p.window, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  double2* tw = reinterpret_cast<double2*>(sm);                 // [256] exp(+2*pi*i*k/256) as (cos, sin)
  const long long sig = (long long)blk * WELCH_WPB + wid;
  // only_flagged: second pass behind a kernel that marks the windows it does not take with num_bins = -2 (unused since the
  // Welch tensor-core path was removed; kept for the DFT path's twin in spectrum_dense_kernel)
  const bool mine = sig < nsig && (!only_flagged || num_bins[sig] == -2);
  if (!__syncthreads_or(mine)) return;
  for (int i = tid; i < 256; i += blockDim.x) { double s_, c_; sincospi((double)i / 128.0, &s_, &c_); tw[i] = make_double2(c_, s_); }
  __syncthreads();
  if (!mine) return;
  double* ys = sm + 512 + (size_t)wid * welch_warp_doubles(W);
  double* buf = ys + W;            // FFT: 256 complex (re, im interleaved); direct DFT: cos[256] | sin[256]
  const double* px = proc_x + sig * W;
  const double* py = proc_y + sig * W;

  // ---- gather: stage (independent loads), then ballot-compact finite y in place; fs from the finite-x mask
  double* xst = buf;               // x staging (W <= 512 checked by the host)
  bool allf = true;
  for (int k = lane; k < W; k += 32) {
    const double x = px[k], y = py[k];
    xst[k] = x; ys[k] = y;
    allf &= isfinite(x) && isfinite(y);
  }
  __syncwarp();
  int n = 0, m = 0;
  double xfirst = 0.0, xlast = 0.0;
  if (__all_sync(0xffffffffu, allf)) {     // a window without holes is its own compaction (one vote instead of W / 32 ballot rounds)
    n = m = W;
    xfirst = xst[0]; xlast = xst[W - 1];
  } else {
    const unsigned lt = (1u << lane) - 1u;
    for (int k0 = 0; k0 < W; k0 += 32) {
      const int k = k0 + lane;
      double x = nan_f64(), y = nan_f64();
      if (k < W) { x = xst[k]; y = ys[k]; }
      const bool fx = isfinite(x), fy = isfinite(y);
      const unsigned bx = __ballot_sync(0xffffffffu, fx), by = __ballot_sync(0xffffffffu, fy);
      if (bx) {
        if (m == 0) xfirst = shfl_dd(x, __ffs(bx) - 1);
        xlast = shfl_dd(x, 31 - __clz(bx));
      }
      __syncwarp();
      if (fy) ys[n + __popc(by & lt)] = y;
      __syncwarp();
      n += __popc(by); m += __popc(bx);
    }
  }
  const double fs = m >= 2 ? 1.0 / ((xlast - xfirst) / (double)(m - 1)) : nan_f64();
  if (!(n >= 2 && isfinite(fs))) {        // guard signal_processor.py:252 -> empty spectrum
    if (lane == 0) { num_bins[sig] = 0; peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
    return;
  }
  const int N = n < 256 ? n : 256, F = N / 2 + 1;
  const int nov = N / 2, hop = N - nov, nseg = (n - nov) / hop;
  const bool fft = N == 256;
  double* dc = buf;                // direct path: cos table
  double* ds = buf + 256;          // direct path: sin table
  if (!fft) {
    for (int i = lane; i < N; i += 32) sincospi(2.0 * (double)i / (double)N, &ds[i], &dc[i]);
  }
  // density scaling 1 / (fs * sum(win^2)) (scipy.signal._spectral_helper).  For the periodic 256-point Hann window the sum is
  // 256 * 3 / 8 = 96, and (win * win).sum() evaluates to exactly 96.0 in float64 (checked against scipy 1.18.1)
  double swsum = 96.0;
  if (!fft) {
    double sw = 0.0;
    for (int i = lane; i < N; i += 32) { const double wj = 0.5 - 0.5 * dc[i]; sw = fma(wj, wj, sw); }
    swsum = warp_sum(sw);
  }
  const double scale = 1.0 / (fs * swsum);
  double facc[5] = {0, 0, 0, 0, 0};               // FFT path: power sums of the bins this lane owns (lane + 32 j; lane 0: bin 128)
  double dm[4] = {0, 0, 0, 0};                    // direct path: bins lane + 32 j (F <= 128)
  for (int sg = 0; sg < nseg; ++sg) {
    const double* seg = ys + sg * hop;
    double a = 0.0;
    for (int i = lane; i < N; i += 32) a += seg[i];
    const double mean = warp_sum(a) / (double)N;
    if (fft) {
      // The segment is real: its 256-point transform comes from ONE 128-point complex FFT of z[m] = x[2m] + i x[2m+1]
      // (half the butterflies and — what bounds this kernel — half the shared-memory wavefronts of the complex 256-point FFT):
      //   E[k] = (Z[k] + conj Z[128-k]) / 2,  O[k] = (Z[k] - conj Z[128-k]) / 2i,  X[k] = E[k] + exp(-2 pi i k / 256) O[k],  k = 0..128
      double2* fz = reinterpret_cast<double2*>(buf);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int m = lane + 32 * j;
        const double2 sv = *reinterpret_cast<const double2*>(seg + 2 * m);
        fz[wpad(m)] = make_double2((sv.x - mean) * (0.5 - 0.5 * tw[2 * m].x), (sv.y - mean) * (0.5 - 0.5 * tw[2 * m + 1].x));
      }
      __syncwarp();
      welch_fft_pass<32, 1>(fz, tw, lane);         // 128-point radix-2 DIF: spans 64 + 32, 16 + 8, 4 + 2, then the last stage
      welch_fft_pass<8, 1>(fz, tw, lane);
      welch_fft_pass<2, 1>(fz, tw, lane);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int i = 2 * (lane + 32 * j);
        const double2 e0 = fz[wpad(i)], e1 = fz[wpad(i + 1)];
        fz[wpad(i)] = cadd(e0, e1);
        fz[wpad(i + 1)] = csub(e0, e1);
      }
      __syncwarp();
      // Z[k] sits at position brev7(k); lane owns the bins k = lane + 32 j (j < 4), lane 0 also bin 128
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const int k = j < 4 ? lane + 32 * j : 128;
        if (j < 4 || lane == 0) {
          const double2 A = fz[wpad((int)(__brev((unsigned)(k & 127)) >> 25))];
          const double2 B = fz[wpad((int)(__brev((unsigned)((128 - k) & 127)) >> 25))];
          const double er = 0.5 * (A.x + B.x), ei = 0.5 * (A.y - B.y);
          const double orr = 0.5 * (A.y + B.y), oi = -0.5 * (A.x - B.x);
          const double2 t = tw[k];                                  // exp(+2 pi i k / 256): X = E + conj(t) O
          const double xr = er + (t.x * orr + t.y * oi), xi = ei + (t.x * oi - t.y * orr);
          double pw = (xr * xr + xi * xi) * scale;
          if (k >= 1 && k < F - 1) pw *= 2.0;
          facc[j] += pw;
        }
      }
      __syncwarp();
    } else {
      // n < 256: nperseg = n, exactly one segment (sg == 0, seg == ys): windowed in place
      for (int i = lane; i < N; i += 32) ys[i] = (seg[i] - mean) * (0.5 - 0.5 * dc[i]);
      __syncwarp();
#pragma unroll
      for (int jb = 0; jb < 4; ++jb) {
        const int k = lane + 32 * jb;
        if (k < F) {
          double re = 0.0, im = 0.0;
          int idx = 0;
          for (int j = 0; j < N; ++j) {
            const double v = ys[j];
            re = fma(v, dc[idx], re);
            im = fma(-v, ds[idx], im);
            idx += k; if (idx >= N) idx -= N;
          }
          double pw = (re * re + im * im) * scale;
          const bool dbl = (N % 2 == 0) ? (k >= 1 && k < F - 1) : (k >= 1);
          if (dbl) pw *= 2.0;
          dm[jb] += pw;
        }
      }
      __syncwarp();
    }
  }
  // rfftfreq(N, d=1/fs)[k] = k * (1/(N*d)); mean over segments; argmax with numpy's first-max rule over finite (BAND: and
  // in-band) bins
  const double fval = 1.0 / ((double)N * (1.0 / fs));
  double bv = -INFINITY; int bi = 0x7fffffff, cnt = 0;
  if (fft) {
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      const int k = j < 4 ? lane + 32 * j : 128;
      if (j < 4 || lane == 0) {
        const double v = nseg == 1 ? facc[j] : facc[j] / (double)nseg;     // mean over ONE segment (n < 384): x / 1 == x
        if (spec_mag && k < max_bins) {
          spec_f[sig * max_bins + k] = (float)((double)k * fval);
          spec_mag[sig * max_bins + k] = (float)v;
        }
        if (isfinite(v) && (!BAND || band.in((double)k * fval))) { ++cnt; if (v > bv || (v == bv && k < bi)) { bv = v; bi = k; } }
      }
    }
  } else {
#pragma unroll
    for (int jb = 0; jb < 4; ++jb) {
      const int k = lane + 32 * jb;
      if (k < F) {
        const double v = nseg == 1 ? dm[jb] : dm[jb] / (double)nseg;
        if (spec_mag && k < max_bins) {
          spec_f[sig * max_bins + k] = (float)((double)k * fval);
          spec_mag[sig * max_bins + k] = (float)v;
        }
        if (isfinite(v) && (!BAND || band.in((double)k * fval))) { ++cnt; if (v > bv) { bv = v; bi = k; } }
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (lane == 0) {
    num_bins[sig] = F;
    if (cnt >= 2) { peak_idx[sig] = bi; peak_freq[sig] = (double)bi * fval; peak_mag[sig] = bv; }
    else { peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
  }
}

}  // namespace bpv
