// F4(b) — pairwise-ROI cross-correlation and PTT lag search (SignalProcessor.correlate_signal_pair /
// correlate_signals and the get_peaks() on sg_corr: signal_processor.py:280-299, 312).
// One CTA per (window job, ROI pair); the jointly valid samples of both signals sit in shared memory;
// each thread owns lags k, k+blockDim, ... of the 2n-1 full-mode lags (float64 dot products, the
// "direct" method scipy.signal.correlate picks for these sizes); normalisation by max(a.a, b.b, a.b);
// first-max argmax over every finite lag fused in.
#include "xcorr_warp.cuh"

namespace bpv {

// BAND: the peak is searched over the lags whose lag in seconds lies in [band.lo, band.hi] (as xcorr_warp_body)
template <bool BAND>
__global__ void __launch_bounds__(128) xcorr_kernel(const double* __restrict__ proc_x, const double* __restrict__ proc_y,
                                                    const bpv_window_params p, float* __restrict__ corr_lag,
                                                    float* __restrict__ corr_val, int32_t* __restrict__ num_lags,
                                                    int32_t* __restrict__ lag_idx, double* __restrict__ lag_sec,
                                                    double* __restrict__ lag_corr, const PeakBand band) {
  extern __shared__ __align__(16) double sm[];
  __shared__ double s_val[33];
  __shared__ int s_idx[64];
  __shared__ int s_n;
  const int W = p.window, R = p.R, P = R * (R - 1) / 2, tid = threadIdx.x, lane = tid & 31;
  const long long jp = blockIdx.x;             // job * P + pair
  const long long job = jp / P;
  int pr = (int)(jp % P), ra = 0, rb = 1;
  for (ra = 0; ra < R - 1; ++ra) {             // itertools.combinations order
    const int cnt = R - 1 - ra;
    if (pr < cnt) { rb = ra + 1 + pr; break; }
    pr -= cnt;
  }
  const double* xa_g = proc_x + (job * R + ra) * W;
  const double* ya_g = proc_y + (job * R + ra) * W;
  const double* yb_g = proc_y + (job * R + rb) * W;
  // shared memory: doubles xa[W] | a64[W] | b64[W] ; floats cv[2W] | c[Kw] reversed b, zero padded | XT[8*LD] a, de-interleaved
  constexpr int RT = 8;
  const int Kw = (W + RT - 1) / RT * RT;
  const int LDw = (Kw + 3 * W + 16) / RT + 1;
  double* xa = sm;             // [W] timestamps of signal a
  double* a64 = xa + W;        // [W] jointly valid samples, float64 (normalisation + refinement)
  double* b64 = a64 + W;       // [W]
  float* cv = reinterpret_cast<float*>(b64 + W);   // [2W] coarse correlation values
  float* c = cv + 2 * W;       // [Kw]
  float* XT = c + Kw;          // [RT * LDw]
  for (int i = tid; i < Kw; i += blockDim.x) c[i] = 0.f;
  for (int i = tid; i < RT * LDw; i += blockDim.x) XT[i] = 0.f;
  __syncthreads();
  // stage the three windows (coalesced), then warp 0 compacts the jointly valid samples in place:
  // valid = a.w & b.w (finite in both)
  for (int k = tid; k < W; k += blockDim.x) { xa[k] = xa_g[k]; a64[k] = ya_g[k]; b64[k] = yb_g[k]; }
  __syncthreads();
  if (tid < 32) {
    int cnt = 0;
    const unsigned lt = (1u << lane) - 1u;
    for (int k0 = 0; k0 < W; k0 += 32) {
      const int k = k0 + lane;
      double va = nan_f64(), vb = nan_f64(), vx = nan_f64();
      if (k < W) { va = a64[k]; vb = b64[k]; vx = xa[k]; }
      const bool ok = isfinite(va) && isfinite(vb);
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      __syncwarp();
      if (ok) {
        const int i = cnt + __popc(bal & lt);
        a64[i] = va; b64[i] = vb; xa[i] = vx;
      }
      __syncwarp();
      cnt += __popc(bal);
    }
    if (lane == 0) s_n = cnt;
  }
  __syncthreads();
  const int n = s_n;
  if (n < 2) {                                  // guard signal_processor.py:284 -> empty
    if (tid == 0) { num_lags[jp] = 0; lag_idx[jp] = -1; lag_sec[jp] = nan_f64(); lag_corr[jp] = nan_f64(); }
    return;
  }
  const int K = (n + RT - 1) / RT * RT;
  double daa = 0, dbb = 0, dab = 0, amax = 0, bmax = 0;
  for (int i = tid; i < n; i += blockDim.x) {
    const double va = a64[i], vb = b64[i];
    daa = fma(va, va, daa); dbb = fma(vb, vb, dbb); dab = fma(va, vb, dab);
    amax = fmax(amax, fabs(va)); bmax = fmax(bmax, fabs(vb));
  }
  daa = block_sum(daa, s_val); dbb = block_sum(dbb, s_val); dab = block_sum(dab, s_val);
  const double den = fmax(fmax(daa, dbb), dab);
  // fp32 operands scaled to O(1) so tiny band-passed signals neither underflow nor lose bits
  for (int o = 16; o > 0; o >>= 1) { amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o)); bmax = fmax(bmax, __shfl_xor_sync(0xffffffffu, bmax, o)); }
  __syncthreads();
  if ((tid & 31) == 0) { s_val[tid >> 5] = amax; s_val[8 + (tid >> 5)] = bmax; }
  __syncthreads();
  for (int w2 = 0; w2 < (int)(blockDim.x >> 5); ++w2) { amax = fmax(amax, s_val[w2]); bmax = fmax(bmax, s_val[8 + w2]); }
  __syncthreads();
  const double sa = amax > 0 ? 1.0 / amax : 1.0, sb = bmax > 0 ? 1.0 / bmax : 1.0;
  for (int i = tid; i < n; i += blockDim.x) {
    XT[xt_index<RT>(i + n - 1 + K, LDw)] = (float)(a64[i] * sa);     // storage index = u + K
    c[n - 1 - i] = (float)(b64[i] * sb);
  }
  __syncthreads();
  const float unscale = (float)(1.0 / (sa * sb * den));
  const int L = 2 * n - 1;
  const long long ob = jp * (2LL * W - 1);
  // COARSE pass in fp32:  corr[li] = sum_l a[l + k] b[l], k = li - (n-1)  ==  sum_m c[m] X[j - m] with j = li + n - 1
  // (corr_tile.cuh); X is non-zero only on u in [n-1, 2n-2], so each tile applies just the taps that can touch it.
  const int jbase = (n - 1 + K) / RT * RT;      // storage index of the tile that holds li = 0
  for (int J0 = jbase + RT * tid; J0 <= (L - 1) + (n - 1) + K; J0 += RT * blockDim.x) {
    float acc[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) acc[r] = 0.f;
    const int u0 = J0 - K;                       // logical index of the tile's first output operand
    int kb_lo = (u0 - (2 * n - 2)) / RT; if (kb_lo < 0) kb_lo = 0;
    int kb_hi = (u0 + RT - 1 - (n - 1)) / RT + 1; if (kb_hi < 0) kb_hi = 0;
    corr_tile<RT, float>(acc, c, K, XT, LDw, J0, kb_lo, kb_hi);
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      const int li = u0 + r - (n - 1);
      if (li >= 0 && li < L) {
        const float cc = acc[r] * unscale;
        cv[li] = cc;
        if (corr_val) {
          const int k = li - (n - 1), ak = k < 0 ? -k : k;
          const double lag = (xa[n - 1] - xa[n - 1 - ak]) * (k > 0 ? 1.0 : (k < 0 ? -1.0 : 0.0));
          corr_lag[ob + li] = (float)lag;
          corr_val[ob + li] = cc;
        }
      }
    }
  }
  __syncthreads();
  // PEAK in float64: every lag whose coarse value is within XC_DELTA of the coarse maximum is re-evaluated as a
  // float64 dot product; the first maximum among those decides (Signal.get_peak after the range reset).
  auto in_band = [&](int li) {
    const int k = li - (n - 1), ak = k < 0 ? -k : k;
    return band.in((xa[n - 1] - xa[n - 1 - ak]) * (k > 0 ? 1.0 : (k < 0 ? -1.0 : 0.0)));
  };
  float cmax = -INFINITY; int cnt = 0, nin = 0;   // BAND: nin = lags inside the band
  for (int li = tid; li < L; li += blockDim.x) {
    const float v = cv[li];
    const bool inb = !BAND || in_band(li);
    if (BAND && inb) ++nin;
    if (isfinite(v) && inb) { ++cnt; cmax = fmaxf(cmax, v); }
  }
  for (int o = 16; o > 0; o >>= 1) { cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o)); cnt += __shfl_xor_sync(0xffffffffu, cnt, o); }
  if (BAND) nin = warp_sum(nin);
  {
    const int wid = tid >> 5, nw = blockDim.x >> 5;
    if (lane == 0) { s_val[wid] = cmax; s_idx[wid] = cnt; if (BAND) s_idx[16 + wid] = nin; }
    __syncthreads();
    cmax = s_val[0]; cnt = s_idx[0];
    if (BAND) nin = s_idx[16];
    for (int w2 = 1; w2 < nw; ++w2) { cmax = fmaxf(cmax, (float)s_val[w2]); cnt += s_idx[w2]; if (BAND) nin += s_idx[16 + w2]; }
    __syncthreads();
  }
  double bv = -INFINITY; int bi = 0x7fffffff;
  for (int li = tid; li < L; li += blockDim.x) {
    const float v = cv[li];
    if ((cnt >= 2 ? (isfinite(v) && v >= cmax - XC_DELTA) : true) && (!BAND || in_band(li))) {
      const int k = li - (n - 1);
      const int l0 = k < 0 ? -k : 0, l1 = k > 0 ? n - k : n;
      double acc = 0.0;
      for (int l = l0; l < l1; ++l) acc = fma(a64[l + k], b64[l], acc);
      const double cc = acc / den;
      if (isfinite(cc) && (cc > bv || (cc == bv && li < bi))) { bv = cc; bi = li; }
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  {
    const int wid = tid >> 5, nw = blockDim.x >> 5;
    if (lane == 0) { s_val[wid] = bv; s_idx[wid] = bi; }
    __syncthreads();
    if (tid == 0) {
      for (int w2 = 1; w2 < nw; ++w2)
        if (s_val[w2] > bv || (s_val[w2] == bv && s_idx[w2] < bi)) { bv = s_val[w2]; bi = s_idx[w2]; }
      // finite-lag count in float64 terms: den == 0 or non-finite makes every lag non-finite (NaN / inf); BAND: of the lags
      // inside the band
      const bool any = isfinite(den) && den != 0.0 && bi != 0x7fffffff;
      num_lags[jp] = L;
      if (any && (BAND ? nin : L) >= 2) {
        const int k = bi - (n - 1), ak = k < 0 ? -k : k;
        lag_idx[jp] = bi;
        lag_sec[jp] = (xa[n - 1] - xa[n - 1 - ak]) * (k > 0 ? 1.0 : (k < 0 ? -1.0 : 0.0));
        lag_corr[jp] = bv;
      } else { lag_idx[jp] = -1; lag_sec[jp] = nan_f64(); lag_corr[jp] = nan_f64(); }
    }
  }
}


// warp-per-pair kernel (default): body in xcorr_warp.cuh
template <int LDC, bool ONE, bool BAND>
__global__ void __launch_bounds__(128, ONE ? 5 : 1) xcorr_warp_kernel(const double* __restrict__ proc_x, const double* __restrict__ proc_y,
                                                         const bpv_window_params p, const XwLayout Lw, long long npairs,
                                                         float* __restrict__ corr_lag, float* __restrict__ corr_val,
                                                         int32_t* __restrict__ num_lags, int32_t* __restrict__ lag_idx,
                                                         double* __restrict__ lag_sec, double* __restrict__ lag_corr,
                                                         const PeakBand band) {
  extern __shared__ __align__(16) unsigned char xsm[];
  xcorr_warp_body<LDC, ONE, BAND>(blockIdx.x, xsm, proc_x, proc_y, p, Lw, npairs, corr_lag, corr_val, num_lags, lag_idx, lag_sec, lag_corr,
                                  band);
}

}  // namespace bpv

extern "C" int bpv_window_xcorr(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                                float* corr_lag, float* corr_val, int32_t* num_lags,
                                int32_t* lag_idx, double* lag_sec, double* lag_corr, void* stream) {
  return bpv_window_xcorr_band(proc_x, proc_y, p, corr_lag, corr_val, num_lags, lag_idx, lag_sec, lag_corr, -INFINITY, INFINITY, stream);
}

extern "C" int bpv_window_xcorr_band(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                                     float* corr_lag, float* corr_val, int32_t* num_lags,
                                     int32_t* lag_idx, double* lag_sec, double* lag_corr,
                                     double min_lag, double max_lag, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(!isnan(min_lag) && !isnan(max_lag), BPV_E_INVALID, "bpv_window_xcorr: NaN lag band (%g, %g)", min_lag, max_lag);
  const bool banded = band_limits(min_lag, max_lag);
  const PeakBand band{min_lag, max_lag};
  BPV_REQUIRE(p && proc_x && proc_y && num_lags && lag_idx && lag_sec && lag_corr, BPV_E_INVALID, "bpv_window_xcorr: NULL pointer");
  BPV_REQUIRE((corr_lag == nullptr) == (corr_val == nullptr), BPV_E_INVALID, "bpv_window_xcorr: corr_lag/corr_val must both be set or both NULL");
  const int W = p->window, P = p->R * (p->R - 1) / 2;
  if (P == 0) return 0;
  const long long n = (long long)p->S * p->jobs_per_stream * P;
  BPV_REQUIRE(W > 0 && n > 0, BPV_E_INVALID, "bpv_window_xcorr: bad sizes");
  {  // warp-per-pair kernel whenever one pair fits the shared memory of a CTA
    const XwLayout Lw = xw_layout(W);
    int wpb = (200 * 1024) / Lw.total;
    if (wpb > 4) wpb = 4;
    if (wpb >= 1) {
      const size_t smw = (size_t)wpb * Lw.total;
      const unsigned grid = (unsigned)((n + wpb - 1) / wpb);
#define BPV_XW1(LDC, ONE, BAND)                                                                                       \
  do {                                                                                                                \
    if (int rc = ensure_dyn_smem((const void*)xcorr_warp_kernel<LDC, ONE, BAND>, smw)) return rc;                     \
    xcorr_warp_kernel<LDC, ONE, BAND><<<grid, wpb * 32, smw, (cudaStream_t)stream>>>(proc_x, proc_y, *p, Lw, n, corr_lag, \
                                                                 corr_val, num_lags, lag_idx, lag_sec, lag_corr, band); \
  } while (0)
#define BPV_XW(LDC, ONE)                                                                                              \
  do {                                                                                                                \
    if (banded) BPV_XW1(LDC, ONE, true);                                                                              \
    else BPV_XW1(LDC, ONE, false);                                                                                    \
  } while (0)
      if (Lw.LD == 63 && Lw.one_round) BPV_XW(63, true);      // windows of 291..300 samples (the 10 s window at 30 fps)
      else if (Lw.LD == 53 && Lw.one_round) BPV_XW(53, true); // 241..250 (the reference's default signal_max_samples)
      else if (Lw.one_round) BPV_XW(0, true);
      else BPV_XW(0, false);
#undef BPV_XW
#undef BPV_XW1
      return check_launch("bpv_window_xcorr");
    }
  }
  const int Kw = (W + 7) / 8 * 8;
  const size_t smem = (size_t)(3 * W) * sizeof(double) + (size_t)(2 * W + Kw + 8 * ((Kw + 3 * W + 16) / 8 + 1)) * sizeof(float);
  BPV_REQUIRE(smem <= 200 * 1024, BPV_E_TOO_LARGE, "bpv_window_xcorr: window %d too large for shared memory", W);
  if (int rc = ensure_dyn_smem(banded ? (const void*)xcorr_kernel<true> : (const void*)xcorr_kernel<false>, smem)) return rc;
  if (banded)
    xcorr_kernel<true><<<(unsigned)n, 128, smem, (cudaStream_t)stream>>>(proc_x, proc_y, *p, corr_lag, corr_val, num_lags, lag_idx, lag_sec,
                                                                         lag_corr, band);
  else
    xcorr_kernel<false><<<(unsigned)n, 128, smem, (cudaStream_t)stream>>>(proc_x, proc_y, *p, corr_lag, corr_val, num_lags, lag_idx, lag_sec,
                                                                          lag_corr, band);
  return check_launch("bpv_window_xcorr");
}
