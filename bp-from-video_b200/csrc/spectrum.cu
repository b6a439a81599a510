// F3 spectra + F4(a) heart-rate peak (SignalProcessor.transform_signal(s) and the get_peaks() that
// follows it: signal_processor.py:248-277, 310; signal_data.py:65-70).
//
//   DFT_RFFT / PGRAM_WELCH  one CTA per signal, float64 direct DFT against a shared-memory twiddle
//                           table (n <= window, so the whole problem is shared-memory resident);
//                           argmax fused into the same kernel.
//   PGRAM_LS                signal x frequency-tile grid.  Coarse pass in fp32: each thread owns one
//                           frequency, loops over the shared-memory time tile, phase reduced to
//                           [-0.5, 0.5) turns with an exact two-float product, MUFU sin/cos, six
//                           running sums (C, S, CC, CS, YC, YS); the tau rotation and the
//                           floating-mean corrections are applied once per frequency in closed form
//                           (scipy/signal/_spectral_py.py:284-349).  Peak pass: candidates within
//                           LS_DELTA of the fp32 maximum are re-evaluated in float64 with scipy's own
//                           two-pass formulation so that the winning bin is decided in float64.
#include <stdlib.h>
#include "filters.cuh"
#include "welch.cuh"

namespace bpv {

long long dft_tc_image_bytes(int W);
long long dft_tc_split_bytes(int W, long long nsig);
int launch_dft_tc(const double* proc_x, const double* proc_y, int W, long long nsig, int max_bins, float* spec_f, float* mags,
                  int32_t* num_bins, int32_t* peak_idx, double* peak_freq, double* peak_mag, void* image_ws, void* split_ws,
                  bool banded, PeakBand band, cudaStream_t st);

constexpr float LS_DELTA = 1.0e-4f;     // candidate band below the fp32 maximum (PSD is in [0, 1])
constexpr int LS_SMALL_N = 24;          // below this every bin is evaluated in float64
constexpr double EPSNEG = 1.1102230246251565e-16;  // np.finfo(float64).epsneg

struct SigInfo { int n, m; double fs, xfirst; };

// Block-cooperative gather of one processed signal.  All threads first stage the window into shared memory
// (coalesced, one round trip to global memory); warp 0 then compacts the samples with finite y IN PLACE (a
// compacted index never exceeds the position it came from) into ys[] and their x into xs[].
// Returns n (finite y), m (finite x), fs = (m-1)/(x_last - x_first).  Signal.get_fs (signal_data.py:55-58) uses
// the finite-x mask v.  xs and ys are shared-memory arrays of W doubles.
__device__ SigInfo gather_signal(const double* __restrict__ px, const double* __restrict__ py, int W,
                                 double* xs, double* ys, int* s_cnt /* >= 4 ints smem */, double* s_d /* >= 2 doubles */) {
  const int tid = threadIdx.x, lane = tid & 31;
  for (int k = tid; k < W; k += blockDim.x) { xs[k] = px[k]; ys[k] = py[k]; }
  __syncthreads();
  if (tid < 32) {
    int n = 0, m = 0, kfirst = 0x7fffffff;
    double xfirst = nan_f64(), xlast = nan_f64();
    const unsigned lt = (1u << lane) - 1u;
    for (int k0 = 0; k0 < W; k0 += 32) {
      const int k = k0 + lane;
      double x = nan_f64(), y = nan_f64();
      if (k < W) { x = xs[k]; y = ys[k]; }
      const bool fx = isfinite(x), fy = isfinite(y);
      const unsigned bx = __ballot_sync(0xffffffffu, fx), by = __ballot_sync(0xffffffffu, fy);
      if (bx) {
        if (kfirst == 0x7fffffff) { kfirst = k0 + __ffs(bx) - 1; xfirst = __shfl_sync(0xffffffffu, x, __ffs(bx) - 1); }
        xlast = __shfl_sync(0xffffffffu, x, 31 - __clz(bx));
      }
      __syncwarp();
      if (fy) { const int idx = n + __popc(by & lt); ys[idx] = y; xs[idx] = x; }
      __syncwarp();
      n += __popc(by); m += __popc(bx);
    }
    if (lane == 0) { s_cnt[0] = n; s_cnt[1] = m; s_d[0] = xfirst; s_d[1] = xlast; }
  }
  __syncthreads();
  SigInfo si;
  si.n = s_cnt[0]; si.m = s_cnt[1];
  si.xfirst = s_d[0];
  si.fs = si.m >= 2 ? 1.0 / ((s_d[1] - s_d[0]) / (double)(si.m - 1)) : nan_f64();
  return si;
}

// Block argmax with numpy's first-max rule over finite values; also counts finite entries.
// vals in shared/global memory (double).  Result broadcast through smem.  BAND: only bins with band.lo <= k * fval <= band.hi.
struct Peak { int idx; double val; int nfinite; };
template <bool BAND>
__device__ Peak block_argmax(const double* vals, int F, double* s_val, int* s_idx, double fval, const PeakBand band) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = (blockDim.x + 31) >> 5;
  double bv = -INFINITY; int bi = 0x7fffffff, cnt = 0;
  for (int k = tid; k < F; k += blockDim.x) {
    const double v = vals[k];
    if (isfinite(v) && (!BAND || band.in((double)k * fval))) { ++cnt; if (v > bv || (v == bv && k < bi)) { bv = v; bi = k; } }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  __syncthreads();
  if (lane == 0) { s_val[wid] = bv; s_idx[wid] = bi; s_idx[32 + wid] = cnt; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < nw; ++w) {
      if (s_val[w] > bv || (s_val[w] == bv && s_idx[w] < bi)) { bv = s_val[w]; bi = s_idx[w]; }
      cnt += s_idx[32 + w];
    }
    s_val[0] = bv; s_idx[0] = bi; s_idx[32] = cnt;
  }
  __syncthreads();
  Peak p; p.val = s_val[0]; p.idx = s_idx[0]; p.nfinite = s_idx[32];
  __syncthreads();
  return p;
}

// ---------------------------------------------------------------------------------------------
// DFT_RFFT and PGRAM_WELCH: one CTA per signal.
// smem doubles: ys[W] | tw_c[N] | tw_s[N] | z[N] | mags[F]   (N = n or nperseg <= W, F <= W/2+1)
// ---------------------------------------------------------------------------------------------
template <bool BAND>
__global__ void __launch_bounds__(128) spectrum_dense_kernel(const double* __restrict__ proc_x,
                                                             const double* __restrict__ proc_y,
                                                             const bpv_window_params p, int max_bins, int only_flagged,
                                                             float* __restrict__ spec_f, float* __restrict__ spec_mag,
                                                             int32_t* __restrict__ num_bins, int32_t* __restrict__ peak_idx,
                                                             double* __restrict__ peak_freq, double* __restrict__ peak_mag,
                                                             const PeakBand band) {
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_cnt[4];
  if (only_flagged && num_bins[blockIdx.x] != -2) return;   // second pass behind dft_tc_kernel (CTA uniform)
  __shared__ double s_d[2];
  __shared__ double s_val[33];
  __shared__ int s_idx[64];
  const int W = p.window, tid = threadIdx.x;
  const long long sig = blockIdx.x;
  double* ys = sm;
  double* twc = ys + W;
  double* tws = twc + W;
  double* z = tws + W;
  double* mags = z + W;
  double* fim = mags + (W / 2 + 2);   // [256] FFT imaginary parts (Welch fast path)
  const SigInfo si = gather_signal(proc_x + sig * W, proc_y + sig * W, W, twc /* x staging, overwritten below */, ys, s_cnt, s_d);
  const int n = si.n;
  if (!(n >= 2 && isfinite(si.fs))) {        // guard signal_processor.py:252 -> empty spectrum
    if (tid == 0) { num_bins[sig] = 0; peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
    return;
  }
  const double fs = si.fs;
  int N, F;
  if (p.transform == BPV_DFT_RFFT) {
    // mags = 2*|rfft(y)|/n, freqs = rfftfreq(n, 1/fs)   (signal_processor.py:254-258)
    N = n; F = n / 2 + 1;
    for (int i = tid; i < N; i += blockDim.x) sincospi(2.0 * (double)i / (double)N, &tws[i], &twc[i]);
    __syncthreads();
    for (int k = tid; k < F; k += blockDim.x) {
      double re = 0.0, im = 0.0;
      int idx = 0;
      for (int j = 0; j < N; ++j) {
        const double v = ys[j];
        re = fma(v, twc[idx], re);
        im = fma(-v, tws[idx], im);
        idx += k; if (idx >= N) idx -= N;
      }
      mags[k] = 2.0 * hypot(re, im) / (double)N;
    }
  } else {
    // scipy.signal.welch(y, fs) defaults (signal_processor.py:260): periodic Hann, nperseg=min(256,n),
    // 50 % overlap, per-segment mean removal, one-sided density, mean over segments.
    N = n < 256 ? n : 256; F = N / 2 + 1;
    const int nov = N / 2, hop = N - nov, nseg = (n - nov) / hop;
    for (int i = tid; i < N; i += blockDim.x) sincospi(2.0 * (double)i / (double)N, &tws[i], &twc[i]);
    for (int k = tid; k < F; k += blockDim.x) mags[k] = 0.0;
    __syncthreads();
    // sum of squared window: w_j = 0.5 - 0.5*cos(2*pi*j/N) = 0.5 - 0.5*twc[j]
    double sw = 0.0;
    for (int i = tid; i < N; i += blockDim.x) { const double wj = 0.5 - 0.5 * twc[i]; sw += wj * wj; }
    const double sumw2 = block_sum(sw, s_val);
    const double scale = 1.0 / (fs * sumw2);
    for (int s = 0; s < nseg; ++s) {
      const double* seg = ys + s * hop;
      double a = 0.0;
      for (int i = tid; i < N; i += blockDim.x) a += seg[i];
      const double mean = block_sum(a, s_val) / (double)N;
      for (int i = tid; i < N; i += blockDim.x) z[i] = (seg[i] - mean) * (0.5 - 0.5 * twc[i]);
      __syncthreads();
      if (N == 256) {
        // steady state (n >= 256): radix-2 FFT of the 256 real samples in shared memory — 8 stages of 128
        // butterflies, one per thread — instead of a 129 x 256 direct DFT.  fr/fi reuse z[] and ys-free space.
        double* fr = z;            // [256] real parts (bit-reversed load done below)
        double* fi = fim;          // [256] imaginary parts
        const double v0 = z[tid], v1 = z[tid + 128];
        __syncthreads();
        fr[__brev((unsigned)tid) >> 24] = v0;
        fr[__brev((unsigned)(tid + 128)) >> 24] = v1;
        fi[tid] = 0.0; fi[tid + 128] = 0.0;
        __syncthreads();
#pragma unroll
        for (int st = 0; st < 8; ++st) {
          const int half = 1 << st;
          const int pos = tid & (half - 1);
          const int i0 = ((tid >> st) << (st + 1)) + pos, i1 = i0 + half;
          const int tw = pos << (7 - st);                       // twiddle exp(-2*pi*i*tw/256)
          const double wr = twc[tw], wi = -tws[tw];
          const double xr = fr[i1], xi = fi[i1];
          const double tr = wr * xr - wi * xi, ti = wr * xi + wi * xr;
          const double ur = fr[i0], ui = fi[i0];
          fr[i0] = ur + tr; fi[i0] = ui + ti;
          fr[i1] = ur - tr; fi[i1] = ui - ti;
          __syncthreads();
        }
        for (int k = tid; k < F; k += blockDim.x) {
          double pw = (fr[k] * fr[k] + fi[k] * fi[k]) * scale;
          if (k >= 1 && k < F - 1) pw *= 2.0;
          mags[k] += pw;
        }
        __syncthreads();
        continue;
      }
      for (int k = tid; k < F; k += blockDim.x) {
        double re = 0.0, im = 0.0;
        int idx = 0;
        for (int j = 0; j < N; ++j) {
          const double v = z[j];
          re = fma(v, twc[idx], re);
          im = fma(-v, tws[idx], im);
          idx += k; if (idx >= N) idx -= N;
        }
        double pw = (re * re + im * im) * scale;
        const bool dbl = (N % 2 == 0) ? (k >= 1 && k < F - 1) : (k >= 1);
        if (dbl) pw *= 2.0;
        mags[k] += pw;
      }
      __syncthreads();
    }
    for (int k = tid; k < F; k += blockDim.x) mags[k] /= (double)nseg;
  }
  __syncthreads();
  // rfftfreq(N, d=1/fs)[k] = k * (1/(N*d))
  const double fval = 1.0 / ((double)N * (1.0 / fs));
  if (spec_mag) {
    for (int k = tid; k < F && k < max_bins; k += blockDim.x) {
      spec_f[sig * max_bins + k] = (float)((double)k * fval);
      spec_mag[sig * max_bins + k] = (float)mags[k];
    }
  }
  const Peak pk = block_argmax<BAND>(mags, F, s_val, s_idx, fval, band);
  if (tid == 0) {
    num_bins[sig] = F;
    if (pk.nfinite >= 2) { peak_idx[sig] = pk.idx; peak_freq[sig] = (double)pk.idx * fval; peak_mag[sig] = pk.val; }
    else { peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
  }
}

// PGRAM_WELCH: the warp-per-signal kernel lives in welch.cuh (welch_warp_body)
template <bool BAND>
__global__ void __launch_bounds__(32 * WELCH_WPB, WELCH_MINB) welch_warp_kernel(const double* __restrict__ proc_x,
                                                                    const double* __restrict__ proc_y,
                                                                    const bpv_window_params p, int max_bins, long long nsig,
                                                                    int only_flagged, float* __restrict__ spec_f, float* __restrict__ spec_mag,
                                                                    int32_t* __restrict__ num_bins, int32_t* __restrict__ peak_idx,
                                                                    double* __restrict__ peak_freq, double* __restrict__ peak_mag,
                                                                    const PeakBand band) {
  extern __shared__ __align__(16) double sm[];
  welch_warp_body<BAND>(blockIdx.x, sm, proc_x, proc_y, p, max_bins, nsig, only_flagged, spec_f, spec_mag, num_bins, peak_idx, peak_freq,
                        peak_mag, band);
}

// ---------------------------------------------------------------------------------------------
// Lomb-Scargle
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double ls_freq(int k, int F, double fmin, double fmax) {  // np.linspace(fmin, fmax, F)[k]
  if (F == 1) return fmin;
  if (k == F - 1) return fmax;
  const double step = (fmax - fmin) / (double)(F - 1);
  return __dadd_rn(__dmul_rn((double)k, step), fmin);
}

// Generalised LS (floating mean, normalised) at one frequency, float64, scipy's two passes.
// t: times relative to the first sample (the estimator is shift invariant), y: samples, n of them.
// Executed by one warp; returns the value on every lane.
__device__ double ls_eval_f64(const double* __restrict__ t, const double* __restrict__ y, int n, double f,
                              double Y, double YY /* already minus Y*Y */) {
  const int lane = threadIdx.x & 31;
  const double w = 1.0 / (double)n;
  double C = 0, S = 0, CC = 0, CS = 0;
  for (int j = lane; j < n; j += 32) {
    double ph = f * t[j];
    ph -= rint(ph);
    double s, c;
    sincospi(2.0 * ph, &s, &c);
    C += c; S += s; CC = fma(c, c, CC); CS = fma(c, s, CS);
  }
  C = warp_sum(C) * w; S = warp_sum(S) * w; CC = warp_sum(CC) * w; CS = warp_sum(CS) * w;
  double SS = 1.0 - CC;
  CC -= C * C; SS -= S * S; CS -= C * S;
  const double tau = 0.5 * atan2(2.0 * CS, CC - SS);
  const double tau_turns = tau / (2.0 * 3.141592653589793);
  double YC = 0, YS = 0, C2 = 0, S2 = 0, CC2 = 0;
  for (int j = lane; j < n; j += 32) {
    double ph = f * t[j];
    ph -= rint(ph);
    ph -= tau_turns;
    double s, c;
    sincospi(2.0 * ph, &s, &c);
    YC = fma(y[j], c, YC); YS = fma(y[j], s, YS);
    C2 += c; S2 += s; CC2 = fma(c, c, CC2);
  }
  YC = warp_sum(YC) * w; YS = warp_sum(YS) * w; C2 = warp_sum(C2) * w; S2 = warp_sum(S2) * w; CC2 = warp_sum(CC2) * w;
  double SS2 = 1.0 - CC2;
  YC -= Y * C2; YS -= Y * S2; CC2 -= C2 * C2; SS2 -= S2 * S2;
  if (CC2 < EPSNEG) CC2 = EPSNEG;
  if (SS2 < EPSNEG) SS2 = EPSNEG;
  const double a = YC / CC2, b = YS / SS2;
  return 2.0 * (a * YC + b * YS) * (0.5 / YY);
}

// Coarse fp32 pass (LS_NF = 4..8, chosen per launch).  grid = (nsig, ceil(Fmax / (LS_NF * blockDim))), thread t of tile T owns the LS_NF
// frequencies k = T*LS_NF*blockDim + t + m*blockDim, m = 0..LS_NF-1.  The grid is uniform, so consecutive
// frequencies of a thread differ by D = blockDim*df and exp(i*2pi*(f+D)*t_j) = exp(i*2pi*f*t_j) * rot_j with
// rot_j = exp(i*2pi*D*t_j) shared by the whole CTA: one sincos (2 MUFU + exact phase reduction) per sample
// per thread, then LS_NF-1 complex rotations (4 FP32 ops each) — the kernel is issue-bound, and this cuts
// the instructions per (sample, frequency) pair from ~26 to ~13.
// smem: doubles xs[W] | ys[W] (gather scratch), then float4 {t_hi, t_lo, y - mean, 0}[W], float2 rot[W].
template <int LS_NF>
__global__ void __launch_bounds__(128) ls_coarse_kernel(const double* __restrict__ proc_x, const double* __restrict__ proc_y,
                                                        const bpv_window_params p, int max_bins,
                                                        float* __restrict__ spec_f, float* __restrict__ psd) {
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_cnt[4];
  __shared__ double s_d[2];
  __shared__ double s_red[33];
  const int W = p.window, tid = threadIdx.x, BD = blockDim.x;
  const long long sig = blockIdx.x;
  double* xs = sm;            // [W]
  double* ys = xs + W;        // [W]
  float4* smp = reinterpret_cast<float4*>(ys + W);    // [W]
  float2* rot = reinterpret_cast<float2*>(smp + W);   // [W]
  const SigInfo si = gather_signal(proc_x + sig * W, proc_y + sig * W, W, xs, ys, s_cnt, s_d);
  const int n = si.n;
  if (!(n >= 2 && isfinite(si.fs))) return;              // peak kernel reports the empty spectrum
  const int F = p.ls_num_freqs > 0 ? p.ls_num_freqs : n;
  const int kbase = blockIdx.y * LS_NF * BD;
  if (kbase >= F) return;
  // centre y (floating mean makes this a no-op mathematically; it is what keeps fp32 usable)
  double a = 0.0;
  for (int j = tid; j < n; j += BD) a += ys[j];
  const double mean = block_sum(a, s_red) / (double)n;
  double q = 0.0;
  const double t0 = xs[0];
  const double dstep = F > 1 ? (p.max_freq - p.min_freq) / (double)(F - 1) : 0.0;
  const double D = dstep * (double)BD;                    // frequency distance between a thread's bins
  for (int j = tid; j < n; j += BD) {
    const double d = ys[j] - mean, t = xs[j] - t0;
    q = fma(d, d, q);
    const float hi = (float)t;
    smp[j] = make_float4(hi, (float)(t - (double)hi), (float)d, 0.f);
    double ph = D * t;
    ph -= rint(ph);
    double sr, cr;
    sincospi(2.0 * ph, &sr, &cr);
    rot[j] = make_float2((float)cr, (float)sr);
  }
  const double YY = block_sum(q, s_red) / (double)n;     // variance (Y = 0 after centring); barrier inside
  const int k0 = kbase + tid;
  const double f = ls_freq(k0 < F ? k0 : F - 1, F, p.min_freq, p.max_freq);
  const float fh = (float)f, fl = (float)(f - (double)fh);
  // (Packed float instructions — FADD2 / FMUL2 / FFMA2 on (c, s) pairs, 5 instead of 10 instructions per (sample, frequency)
  // slot, bit-identical results — were measured on B200 and are slower here: config 3 2.24 -> 2.28 ms, config 5 8.94 -> 9.10 ms
  // per step (profiles/r4a): a packed instruction holds the FP32 pipe for two issue slots, and the pairs cost registers.)
  float C[LS_NF], S[LS_NF], CC[LS_NF], CS[LS_NF], YC[LS_NF], YS[LS_NF];
#pragma unroll
  for (int m = 0; m < LS_NF; ++m) { C[m] = S[m] = CC[m] = CS[m] = YC[m] = YS[m] = 0.f; }
#pragma unroll 2
  for (int j = 0; j < n; ++j) {
    const float4 sv = smp[j];
    const float2 rv = rot[j];
    const float ph = fh * sv.x;
    const float e1 = fmaf(fh, sv.x, -ph);                 // exact low part of the product
    const float e2 = fmaf(fh, sv.y, fl * sv.x);
    const float r = (ph - rintf(ph)) + (e1 + e2);          // phase in turns, [-0.5, 0.5]
    float s, c;
    __sincosf(6.283185307179586f * r, &s, &c);
#pragma unroll
    for (int m = 0; m < LS_NF; ++m) {
      C[m] += c; S[m] += s;
      CC[m] = fmaf(c, c, CC[m]); CS[m] = fmaf(c, s, CS[m]);
      YC[m] = fmaf(sv.z, c, YC[m]); YS[m] = fmaf(sv.z, s, YS[m]);
      if (m + 1 < LS_NF) {                                 // advance to the next bin: (c, s) *= rot_j
        const float c2 = fmaf(c, rv.x, -s * rv.y), s2 = fmaf(s, rv.x, c * rv.y);
        c = c2; s = s2;
      }
    }
  }
  // closed-form tau rotation + floating-mean corrections, once per frequency, in float64
  const double w = 1.0 / (double)n;
#pragma unroll
  for (int m = 0; m < LS_NF; ++m) {
    const int k = k0 + m * BD;
    if (k >= F) break;
    const double dC = C[m] * w, dS = S[m] * w, dCC = CC[m] * w, dCS = CS[m] * w, dYC = YC[m] * w, dYS = YS[m] * w;
    const double cc0 = dCC - dC * dC, ss0 = (1.0 - dCC) - dS * dS, cs0 = dCS - dC * dS;
    // cos / sin of tau = 0.5 * atan2(2 cs0, cc0 - ss0) by the half-angle formulas (tau in (-pi/2, pi/2]: cos >= 0, the
    // sign of sin is the sign of cs0), each branch free of cancellation; no atan2 / sincos on the per-frequency path
    const double s2 = 2.0 * cs0, c2 = cc0 - ss0, hyp = hypot(s2, c2);
    double st, ct;
    if (!(hyp > 0.0)) { ct = 1.0; st = 0.0; }                    // atan2(0, 0) = 0
    else if (c2 >= 0.0) { ct = sqrt(0.5 * (1.0 + c2 / hyp)); st = 0.5 * (s2 / hyp) / ct; }
    else { st = copysign(sqrt(0.5 * (1.0 - c2 / hyp)), s2); ct = 0.5 * (s2 / hyp) / st; }
    const double YCt = ct * dYC + st * dYS, YSt = ct * dYS - st * dYC;
    const double Ct = ct * dC + st * dS, St = ct * dS - st * dC;
    const double CCraw = ct * ct * dCC + 2.0 * ct * st * dCS + st * st * (1.0 - dCC);
    double CCt = CCraw - Ct * Ct, SSt = (1.0 - CCraw) - St * St;
    if (CCt < EPSNEG) CCt = EPSNEG;
    if (SSt < EPSNEG) SSt = EPSNEG;
    const double pw = 2.0 * (YCt * YCt / CCt + YSt * YSt / SSt) * (0.5 / YY);
    psd[sig * max_bins + k] = (float)pw;
    if (spec_f) spec_f[sig * max_bins + k] = (float)ls_freq(k, F, p.min_freq, p.max_freq);
  }
}

// Peak pass: one CTA (128 threads) per signal.  smem doubles: ts[W] | ys[W] | cand_val[max_bins];
// ints: cand_idx[max_bins].
// BAND: the peak is searched over the bins with band.lo <= ls_freq(k) <= band.hi.  Their fp32 maximum and count are taken over
// those bins alone (an out-of-band maximum would set a threshold that excludes every in-band bin).  The bins re-evaluated for the
// unbanded search are still the ones whose float64 values are written back, so the stored spectrum does not depend on the band:
// a candidate carries bit 30 (write back) and bit 29 (in-band candidate) above its bin index.
template <bool BAND>
__global__ void __launch_bounds__(128) ls_peak_kernel(const double* __restrict__ proc_x, const double* __restrict__ proc_y,
                                                      const bpv_window_params p, int max_bins,
                                                      float* __restrict__ spec_f, float* __restrict__ psd,
                                                      int32_t* __restrict__ num_bins, int32_t* __restrict__ peak_idx,
                                                      double* __restrict__ peak_freq, double* __restrict__ peak_mag,
                                                      const PeakBand band) {
  constexpr int WB = 1 << 30, CB = 1 << 29, KM = CB - 1;
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_cnt[4];
  __shared__ double s_d[2];
  __shared__ double s_val[33];
  __shared__ int s_idx[64];
  __shared__ int s_nc;
  const int W = p.window, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  const long long sig = blockIdx.x;
  double* xs = sm;
  double* ys = xs + W;
  double* cval = ys + W;
  int* cidx = reinterpret_cast<int*>(cval + max_bins);
  const SigInfo si = gather_signal(proc_x + sig * W, proc_y + sig * W, W, xs, ys, s_cnt, s_d);
  const int n = si.n;
  if (!(n >= 2 && isfinite(si.fs))) {
    if (tid == 0) { num_bins[sig] = 0; peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
    return;
  }
  const int F = p.ls_num_freqs > 0 ? p.ls_num_freqs : n;
  float* row = psd + sig * max_bins;
  // fp32 maximum over finite bins (BAND: also over the finite in-band bins, bb / cb)
  float bv = -INFINITY; int cnt = 0;
  float bb = -INFINITY; int cb = 0;
  for (int k = tid; k < F; k += blockDim.x) {
    const float v = row[k];
    if (isfinite(v)) {
      ++cnt; bv = fmaxf(bv, v);
      if (BAND && band.in(ls_freq(k, F, p.min_freq, p.max_freq))) { ++cb; bb = fmaxf(bb, v); }
    }
  }
  for (int o = 16; o > 0; o >>= 1) { bv = fmaxf(bv, __shfl_xor_sync(0xffffffffu, bv, o)); cnt += __shfl_xor_sync(0xffffffffu, cnt, o); }
  if (BAND)
    for (int o = 16; o > 0; o >>= 1) { bb = fmaxf(bb, __shfl_xor_sync(0xffffffffu, bb, o)); cb += __shfl_xor_sync(0xffffffffu, cb, o); }
  if (lane == 0) { s_val[wid] = bv; s_idx[wid] = cnt; if (BAND) { s_val[16 + wid] = bb; s_idx[16 + wid] = cb; } }
  if (tid == 0) s_nc = 0;
  __syncthreads();
  bv = s_val[0]; cnt = s_idx[0];
  for (int w2 = 1; w2 < nw; ++w2) { bv = fmaxf(bv, s_val[w2]); cnt += s_idx[w2]; }
  if (BAND) {
    bb = s_val[16]; cb = s_idx[16];
    for (int w2 = 1; w2 < nw; ++w2) { bb = fmaxf(bb, s_val[16 + w2]); cb += s_idx[16 + w2]; }
  }
  __syncthreads();
  // moments for the float64 evaluation (relative time; Y, YY as scipy Eq. 7 / 10)
  const double t0 = xs[0];
  double a = 0.0;
  for (int j = tid; j < n; j += blockDim.x) a += ys[j];
  const double Y = block_sum(a, s_val) / (double)n;
  double q = 0.0;
  for (int j = tid; j < n; j += blockDim.x) { q = fma(ys[j], ys[j], q); }
  double YY = block_sum(q, s_val) / (double)n - Y * Y;
  {  // the centred second moment is better conditioned than YY - Y*Y when DC >> AC
    double q2 = 0.0;
    for (int j = tid; j < n; j += blockDim.x) { const double d = ys[j] - Y; q2 = fma(d, d, q2); }
    YY = block_sum(q2, s_val) / (double)n;
  }
  for (int j = tid; j < n; j += blockDim.x) xs[j] -= t0;
  __syncthreads();
  // candidate list: every bin for small problems, else bins within LS_DELTA of the fp32 maximum
  const bool all = n < LS_SMALL_N || cnt < 2;
  const bool all_b = BAND ? (n < LS_SMALL_N || cb < 2) : all;
  for (int k = tid; k < F; k += blockDim.x) {
    const float v = row[k];
    const bool cw = all || (isfinite(v) && v >= bv - LS_DELTA);
    bool cbd = false;
    if (BAND) cbd = band.in(ls_freq(k, F, p.min_freq, p.max_freq)) && (all_b || (isfinite(v) && v >= bb - LS_DELTA));
    if (cw || cbd) cidx[atomicAdd(&s_nc, 1)] = BAND ? (k | (cw ? WB : 0) | (cbd ? CB : 0)) : k;
  }
  __syncthreads();
  const int nc = s_nc;
  for (int c = wid; c < nc; c += nw) {
    const int k = BAND ? (cidx[c] & KM) : cidx[c];
    const double v = ls_eval_f64(xs, ys, n, ls_freq(k, F, p.min_freq, p.max_freq), Y, YY);
    if (lane == 0) { cval[c] = v; if (!BAND || (cidx[c] & WB)) row[k] = (float)v; }
  }
  __syncthreads();
  if (all_b && tid == 0) {   // recount finite bins from the float64 values
    int c2 = 0;
    for (int c = 0; c < nc; ++c) c2 += isfinite(cval[c]) && (!BAND || (cidx[c] & CB));
    s_idx[0] = c2;
  }
  __syncthreads();
  const int nfinite = all_b ? s_idx[0] : (BAND ? cb : cnt);
  __syncthreads();
  // first-max rule in float64 over the candidates (ties -> smallest bin index)
  double best = -INFINITY; int bi = 0x7fffffff;
  if (tid == 0) {
    for (int c = 0; c < nc; ++c) {
      const double v = cval[c];
      const int k = BAND ? (cidx[c] & KM) : cidx[c];
      if ((!BAND || (cidx[c] & CB)) && isfinite(v) && (v > best || (v == best && k < bi))) { best = v; bi = k; }
    }
    num_bins[sig] = F;
    if (nfinite >= 2 && bi != 0x7fffffff) {
      peak_idx[sig] = bi; peak_freq[sig] = ls_freq(bi, F, p.min_freq, p.max_freq); peak_mag[sig] = best;
    } else { peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
  }
  if (all && spec_f)
    for (int k = tid; k < F; k += blockDim.x) spec_f[sig * max_bins + k] = (float)ls_freq(k, F, p.min_freq, p.max_freq);
}


// Warp-per-signal version of the Lomb-Scargle peak pass (default): the CTA-per-signal kernel above spends most of its time
// in __syncthreads between short phases (gather, three block reductions, candidate list); here every phase is warp-local.
// smem per warp: doubles ts[W] | ys[W].  BAND as ls_peak_kernel.
constexpr int LSP_WPB = 4;
template <bool BAND>
__global__ void __launch_bounds__(32 * LSP_WPB) ls_peak_warp_kernel(const double* __restrict__ proc_x, const double* __restrict__ proc_y,
                                                                    const bpv_window_params p, int max_bins, long long nsig,
                                                                    float* __restrict__ spec_f, float* __restrict__ psd,
                                                                    int32_t* __restrict__ num_bins, int32_t* __restrict__ peak_idx,
                                                                    double* __restrict__ peak_freq, double* __restrict__ peak_mag,
                                                                    const PeakBand band) {
  extern __shared__ __align__(16) double sm[];
  const int W = p.window, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long sig = (long long)blockIdx.x * LSP_WPB + wid;
  if (sig >= nsig) return;
  double* xs = sm + (size_t)wid * 2 * W;
  double* ys = xs + W;
  const double* px = proc_x + sig * W;
  const double* py = proc_y + sig * W;
  for (int k = lane; k < W; k += 32) { xs[k] = px[k]; ys[k] = py[k]; }
  __syncwarp();
  int n = 0, m = 0;
  double xfirst = 0.0, xlast = 0.0;
  const unsigned lt = (1u << lane) - 1u;
  for (int k0 = 0; k0 < W; k0 += 32) {
    const int k = k0 + lane;
    double x = nan_f64(), y = nan_f64();
    if (k < W) { x = xs[k]; y = ys[k]; }
    const bool fx = isfinite(x), fy = isfinite(y);
    const unsigned bx = __ballot_sync(0xffffffffu, fx), by = __ballot_sync(0xffffffffu, fy);
    if (bx) {
      const double xf = shfl_dd(x, __ffs(bx) - 1), xl = shfl_dd(x, 31 - __clz(bx));
      if (m == 0) xfirst = xf;
      xlast = xl;
    }
    __syncwarp();
    if (fy) { const int i = n + __popc(by & lt); ys[i] = y; xs[i] = x; }
    __syncwarp();
    n += __popc(by); m += __popc(bx);
  }
  const double fs = m >= 2 ? 1.0 / ((xlast - xfirst) / (double)(m - 1)) : nan_f64();
  if (!(n >= 2 && isfinite(fs))) {
    if (lane == 0) { num_bins[sig] = 0; peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
    return;
  }
  const int F = p.ls_num_freqs > 0 ? p.ls_num_freqs : n;
  float* row = psd + sig * max_bins;
  float bv = -INFINITY; int cnt = 0;
  float bb = -INFINITY; int cb = 0;              // BAND: over the finite in-band bins
  for (int k = lane; k < F; k += 32) {
    const float v = row[k];
    if (isfinite(v)) {
      ++cnt; bv = fmaxf(bv, v);
      if (BAND && band.in(ls_freq(k, F, p.min_freq, p.max_freq))) { ++cb; bb = fmaxf(bb, v); }
    }
  }
  for (int o = 16; o > 0; o >>= 1) { bv = fmaxf(bv, __shfl_xor_sync(0xffffffffu, bv, o)); cnt += __shfl_xor_sync(0xffffffffu, cnt, o); }
  if (BAND)
    for (int o = 16; o > 0; o >>= 1) { bb = fmaxf(bb, __shfl_xor_sync(0xffffffffu, bb, o)); cb += __shfl_xor_sync(0xffffffffu, cb, o); }
  // moments for the float64 evaluation (relative time; Y, YY as scipy Eq. 7 / 10; centred second moment)
  const double t0 = xs[0];
  double a = 0.0;
  for (int j = lane; j < n; j += 32) a += ys[j];
  const double Y = warp_sum(a) / (double)n;
  double q2 = 0.0;
  for (int j = lane; j < n; j += 32) { const double d = ys[j] - Y; q2 = fma(d, d, q2); }
  const double YY = warp_sum(q2) / (double)n;
  for (int j = lane; j < n; j += 32) xs[j] -= t0;
  __syncwarp();
  const bool all = n < LS_SMALL_N || cnt < 2;
  const bool all_b = BAND ? (n < LS_SMALL_N || cb < 2) : all;
  double best = -INFINITY; int bi = 0x7fffffff, nf64 = 0;
  for (int k0 = 0; k0 < F; k0 += 32) {
    const int k = k0 + lane;
    bool cand = false, cand_b = false;
    if (k < F) {
      const float v = row[k];
      cand = all || (isfinite(v) && v >= bv - LS_DELTA);
      if (BAND) cand_b = band.in(ls_freq(k, F, p.min_freq, p.max_freq)) && (all_b || (isfinite(v) && v >= bb - LS_DELTA));
    }
    // BAND: mw = bins whose float64 value is written back (the unbanded candidates), mb = in-band candidates
    unsigned mk = __ballot_sync(0xffffffffu, cand || cand_b);
    const unsigned mw = BAND ? __ballot_sync(0xffffffffu, cand) : 0u, mb = BAND ? __ballot_sync(0xffffffffu, cand_b) : 0u;
    while (mk) {
      const int b = __ffs(mk) - 1, kc = k0 + b;
      mk &= mk - 1;
      const double v = ls_eval_f64(xs, ys, n, ls_freq(kc, F, p.min_freq, p.max_freq), Y, YY);
      if (lane == 0 && (!BAND || ((mw >> b) & 1u))) row[kc] = (float)v;
      if ((!BAND || ((mb >> b) & 1u)) && isfinite(v)) { ++nf64; if (v > best || (v == best && kc < bi)) { best = v; bi = kc; } }
    }
  }
  const int nfinite = all_b ? nf64 : (BAND ? cb : cnt);
  if (lane == 0) {
    num_bins[sig] = F;
    if (nfinite >= 2 && bi != 0x7fffffff) {
      peak_idx[sig] = bi; peak_freq[sig] = ls_freq(bi, F, p.min_freq, p.max_freq); peak_mag[sig] = best;
    } else { peak_idx[sig] = -1; peak_freq[sig] = nan_f64(); peak_mag[sig] = nan_f64(); }
  }
  if (all && spec_f)
    for (int k = lane; k < F; k += 32) spec_f[sig * max_bins + k] = (float)ls_freq(k, F, p.min_freq, p.max_freq);
}

}  // namespace bpv

// workspace plan: [DFT_RFFT on the tensor cores: the twiddle operand images of dft_tc.cu — persistent across calls,
// zero-initialised once by the caller; FIRST, so that they stay where they were built whatever the launch's job count]
// [coarse magnitudes / LS psd when the spectrum is not stored, rounded up to 256 B] [DFT_RFFT: this launch's split samples]
static int64_t spectrum_coarse_bytes(const bpv_window_params* p, int32_t max_bins) {
  if (p->transform == BPV_PGRAM_WELCH) return 0;
  return ((int64_t)p->S * p->jobs_per_stream * p->R * max_bins * 4 + 255) / 256 * 256;
}
extern "C" int64_t bpv_spectrum_workspace_bytes(const bpv_window_params* p, int32_t max_bins) {
  if (!p) return -1;
  int64_t b = spectrum_coarse_bytes(p, max_bins);
  if (p->transform == BPV_DFT_RFFT && p->window >= 16 && p->window <= 2048)
    b += (bpv::dft_tc_image_bytes(p->window) + 255) / 256 * 256 + bpv::dft_tc_split_bytes(p->window, (long long)p->S * p->jobs_per_stream * p->R);
  return b;
}

extern "C" int bpv_window_spectrum(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                                   int32_t max_bins, void* workspace, int64_t workspace_bytes,
                                   float* spec_f, float* spec_mag, int32_t* num_bins,
                                   int32_t* peak_idx, double* peak_freq, double* peak_mag, void* stream) {
  return bpv_window_spectrum_band(proc_x, proc_y, p, max_bins, workspace, workspace_bytes, spec_f, spec_mag, num_bins, peak_idx, peak_freq,
                                  peak_mag, -INFINITY, INFINITY, stream);
}

extern "C" int bpv_window_spectrum_band(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                                        int32_t max_bins, void* workspace, int64_t workspace_bytes,
                                        float* spec_f, float* spec_mag, int32_t* num_bins,
                                        int32_t* peak_idx, double* peak_freq, double* peak_mag,
                                        double min_freq, double max_freq, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(!isnan(min_freq) && !isnan(max_freq), BPV_E_INVALID, "bpv_window_spectrum: NaN frequency band (%g, %g)", min_freq, max_freq);
  const bool banded = band_limits(min_freq, max_freq);
  const PeakBand band{min_freq, max_freq};
  BPV_REQUIRE(p && proc_x && proc_y && num_bins && peak_idx && peak_freq && peak_mag, BPV_E_INVALID,
              "bpv_window_spectrum: NULL pointer");
  BPV_REQUIRE((spec_f == nullptr) == (spec_mag == nullptr), BPV_E_INVALID, "bpv_window_spectrum: spec_f/spec_mag must both be set or both NULL");
  BPV_REQUIRE(p->transform == BPV_DFT_RFFT || p->transform == BPV_PGRAM_WELCH || p->transform == BPV_PGRAM_LS, BPV_E_UNSUPPORTED,
              "bpv_window_spectrum: unknown spectrum transform %d (NotImplementedError, signal_processor.py:268)", p->transform);
  const int W = p->window;
  const long long nsig = (long long)p->S * p->jobs_per_stream * p->R;
  BPV_REQUIRE(W > 0 && nsig > 0 && max_bins > 0, BPV_E_INVALID, "bpv_window_spectrum: bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  if (p->transform != BPV_PGRAM_LS) {
    const int need = p->transform == BPV_DFT_RFFT ? W / 2 + 1 : (W < 256 ? W : 256) / 2 + 1;
    BPV_REQUIRE(!spec_mag || max_bins >= need, BPV_E_INVALID, "bpv_window_spectrum: max_bins %d < %d", max_bins, need);
    if (p->transform == BPV_PGRAM_WELCH && W <= 512) {   // warp per signal (x staging needs W <= 512 doubles)
      const size_t smw = (size_t)(512 + WELCH_WPB * welch_warp_doubles(W)) * sizeof(double);
      const int only_flagged = 0;
      const unsigned grid = (unsigned)((nsig + WELCH_WPB - 1) / WELCH_WPB);
      const void* kfn = banded ? (const void*)welch_warp_kernel<true> : (const void*)welch_warp_kernel<false>;
      if (int rc = ensure_dyn_smem(kfn, smw)) return rc;
      if (banded)
        welch_warp_kernel<true><<<grid, 32 * WELCH_WPB, smw, st>>>(proc_x, proc_y, *p, max_bins, nsig, only_flagged, spec_f, spec_mag,
                                                                   num_bins, peak_idx, peak_freq, peak_mag, band);
      else
        welch_warp_kernel<false><<<grid, 32 * WELCH_WPB, smw, st>>>(proc_x, proc_y, *p, max_bins, nsig, only_flagged, spec_f, spec_mag,
                                                                    num_bins, peak_idx, peak_freq, peak_mag, band);
      return check_launch("welch_warp_kernel");
    }
    const size_t smem = (size_t)(4 * W + W / 2 + 2 + 256) * sizeof(double);
    BPV_REQUIRE(smem <= 200 * 1024, BPV_E_TOO_LARGE, "bpv_window_spectrum: window %d too large for the dense spectrum kernel", W);
    if (int rc = ensure_dyn_smem(banded ? (const void*)spectrum_dense_kernel<true> : (const void*)spectrum_dense_kernel<false>, smem))
      return rc;
    // DFT_RFFT as one dense contraction on the tensor cores (dft_tc.cu) when the windows of the launch share n = W: by
    // default for pipelines that resample (INTERP_*: valid = block, so every warmed-up window is full), or forced /
    // disabled with BPV_DFT_TC=1 / 0.  Windows with a non-finite sample are flagged and taken by the float64 kernel.
    int only_flagged = 0;
    if (p->transform == BPV_DFT_RFFT && W >= 16 && W <= 2048) {
      bool interp = false;
      for (int i = 0; i < p->num_methods; ++i) interp |= (p->methods[i] == BPV_INTERP_LINEAR || p->methods[i] == BPV_INTERP_CUBIC);
      const char* env = getenv("BPV_DFT_TC");
      const bool use_tc = env ? env[0] == '1' : interp;
      if (use_tc) {
        // the twiddle operand images open the workspace when it has room for them (and for the coarse area, if the spectrum is
        // not stored): their offset must not depend on the launch's job count, or a launch of another J would find a stale
        // header over overwritten images.  Behind them the coarse area, then the hi / lo images of this launch's samples
        // (A operand) when there is room for those too.
        const int64_t cb = spectrum_coarse_bytes(p, max_bins);
        const int64_t ib = (dft_tc_image_bytes(W) + 255) / 256 * 256;
        const int64_t need_coarse = spec_mag ? 0 : cb;
        void* images = (workspace && workspace_bytes >= ib + need_coarse) ? workspace : nullptr;
        unsigned char* rest = (unsigned char*)workspace + (images ? ib : 0);
        float* coarse = spec_mag;
        if (!coarse) {
          BPV_REQUIRE(workspace && workspace_bytes >= cb, BPV_E_INVALID,
                      "bpv_window_spectrum: workspace too small (see bpv_spectrum_workspace_bytes)");
          coarse = (float*)rest;
        }
        void* split = (images && workspace_bytes >= ib + need_coarse + dft_tc_split_bytes(W, nsig)) ? (void*)(rest + need_coarse) : nullptr;
        if (int rc = launch_dft_tc(proc_x, proc_y, W, nsig, max_bins, spec_f, coarse, num_bins, peak_idx, peak_freq, peak_mag, images, split,
                                   banded, band, st))
          return rc;
        only_flagged = 1;
      }
    }
    if (banded)
      spectrum_dense_kernel<true><<<(unsigned)nsig, 128, smem, st>>>(proc_x, proc_y, *p, max_bins, only_flagged, spec_f, spec_mag, num_bins,
                                                                     peak_idx, peak_freq, peak_mag, band);
    else
      spectrum_dense_kernel<false><<<(unsigned)nsig, 128, smem, st>>>(proc_x, proc_y, *p, max_bins, only_flagged, spec_f, spec_mag,
                                                                      num_bins, peak_idx, peak_freq, peak_mag, band);
    return check_launch("spectrum_dense_kernel");
  }
  const int Fmax = p->ls_num_freqs > 0 ? p->ls_num_freqs : W;
  BPV_REQUIRE(max_bins >= Fmax, BPV_E_INVALID, "bpv_window_spectrum: max_bins %d < %d", max_bins, Fmax);
  float* psd = spec_mag;
  if (!psd) {
    BPV_REQUIRE(workspace && workspace_bytes >= spectrum_coarse_bytes(p, max_bins), BPV_E_INVALID,
                "bpv_window_spectrum: workspace too small (see bpv_spectrum_workspace_bytes)");
    psd = (float*)workspace;
  }
  const size_t smem_c = (size_t)W * (2 * sizeof(double) + sizeof(float4) + sizeof(float2));
  const size_t smem_p = (size_t)W * 2 * sizeof(double) + (size_t)max_bins * (sizeof(double) + sizeof(int));
  BPV_REQUIRE(smem_c <= 200 * 1024 && smem_p <= 200 * 1024, BPV_E_TOO_LARGE, "bpv_window_spectrum: window/grid too large for shared memory");
  for (const void* k : {(const void*)ls_coarse_kernel<4>, (const void*)ls_coarse_kernel<5>, (const void*)ls_coarse_kernel<6>,
                        (const void*)ls_coarse_kernel<7>, (const void*)ls_coarse_kernel<8>})
    if (int rc = ensure_dyn_smem(k, smem_c)) return rc;
  // frequencies per thread NF in 4..8 and threads per CTA (multiple of 32, <= 128): the plan with the smallest padded cost
  // tiles * NF * threads * (instructions per (sample, frequency) slot ~ 10 + 12 / NF: one sincos per sample and thread,
  // 6 accumulations per slot, NF - 1 rotations)
  int best_nf = 4, best_bd = 128, best_tiles = 1;
  double best_cost = 1e300;
  for (int nf = 4; nf <= 8; ++nf) {
    int bd = ((Fmax + nf - 1) / nf + 31) / 32 * 32;          // enough threads for Fmax in one tile, up to 128
    if (bd > 128) bd = 128;
    const int tiles = (Fmax + nf * bd - 1) / (nf * bd);
    const double cost = (double)tiles * nf * bd * (10.0 + 12.0 / nf);
    if (cost < best_cost) { best_cost = cost; best_nf = nf; best_bd = bd; best_tiles = tiles; }
  }
  const dim3 grid((unsigned)nsig, best_tiles);
  switch (best_nf) {
    case 4: ls_coarse_kernel<4><<<grid, best_bd, smem_c, st>>>(proc_x, proc_y, *p, max_bins, spec_f, psd); break;
    case 5: ls_coarse_kernel<5><<<grid, best_bd, smem_c, st>>>(proc_x, proc_y, *p, max_bins, spec_f, psd); break;
    case 6: ls_coarse_kernel<6><<<grid, best_bd, smem_c, st>>>(proc_x, proc_y, *p, max_bins, spec_f, psd); break;
    case 7: ls_coarse_kernel<7><<<grid, best_bd, smem_c, st>>>(proc_x, proc_y, *p, max_bins, spec_f, psd); break;
    default: ls_coarse_kernel<8><<<grid, best_bd, smem_c, st>>>(proc_x, proc_y, *p, max_bins, spec_f, psd); break;
  }
  if (int rc = check_launch("ls_coarse_kernel")) return rc;
  const size_t smem_w = (size_t)LSP_WPB * 2 * W * sizeof(double);
  if (smem_w <= 200 * 1024) {          // warp per signal
    const unsigned grid = (unsigned)((nsig + LSP_WPB - 1) / LSP_WPB);
    if (int rc = ensure_dyn_smem(banded ? (const void*)ls_peak_warp_kernel<true> : (const void*)ls_peak_warp_kernel<false>, smem_w))
      return rc;
    if (banded)
      ls_peak_warp_kernel<true><<<grid, 32 * LSP_WPB, smem_w, st>>>(proc_x, proc_y, *p, max_bins, nsig, spec_f, psd, num_bins, peak_idx,
                                                                    peak_freq, peak_mag, band);
    else
      ls_peak_warp_kernel<false><<<grid, 32 * LSP_WPB, smem_w, st>>>(proc_x, proc_y, *p, max_bins, nsig, spec_f, psd, num_bins, peak_idx,
                                                                     peak_freq, peak_mag, band);
    return check_launch("ls_peak_warp_kernel");
  }
  if (int rc = ensure_dyn_smem(banded ? (const void*)ls_peak_kernel<true> : (const void*)ls_peak_kernel<false>, smem_p)) return rc;
  if (banded)
    ls_peak_kernel<true><<<(unsigned)nsig, 128, smem_p, st>>>(proc_x, proc_y, *p, max_bins, spec_f, psd, num_bins, peak_idx, peak_freq,
                                                              peak_mag, band);
  else
    ls_peak_kernel<false><<<(unsigned)nsig, 128, smem_p, st>>>(proc_x, proc_y, *p, max_bins, spec_f, psd, num_bins, peak_idx, peak_freq,
                                                               peak_mag, band);
  return check_launch("ls_peak_kernel");
}
