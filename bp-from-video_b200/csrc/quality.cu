// Per-window signal quality: spectral SNR of the heart-rate peak (de Haan & Jeanne, IEEE TBME 2013) over the spectrum F3
// stored, and the SNR gate of the peaks the running means push (include/bpv.h bpv_window_snr).
//
// One CTA per window job (grid-stride over the jobs), one warp per ROI signal (warps loop when R exceeds them).  The lanes
// stride over the bins with coalesced float32 loads and accumulate S_sig / S_noise in float64; the fixed lane assignment
// and the xor shuffle tree make every result reproducible from run to run.  After a barrier the pairs of the job read the
// accept decisions back from the job's snr_db row.
#include "common.cuh"

namespace bpv {

constexpr int SNR_MAX_WARPS = 8;

__global__ void __launch_bounds__(32 * SNR_MAX_WARPS) window_snr_kernel(
    const float* __restrict__ spec_f, const float* __restrict__ spec_mag, const int32_t* __restrict__ num_bins,
    const int32_t* __restrict__ peak_idx, long long J, int R, int max_bins, int square, double lo, double hi, double hw,
    const double* __restrict__ peak_freq, const double* __restrict__ lag_sec, int P, double min_snr_db, double* snr_db,
    double* __restrict__ gated_freq, double* __restrict__ gated_lag) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (long long j = blockIdx.x; j < J; j += gridDim.x) {
    for (int r = warp; r < R; r += nwarps) {
      const long long sig = j * R + r;
      int nb = num_bins[sig];
      nb = nb < max_bins ? nb : max_bins;
      const int pk = peak_idx[sig];
      double snr = nan_f64();
      if (pk >= 0 && pk < nb) {                      // warp-uniform
        const float* f = spec_f + sig * max_bins;
        const float* m = spec_mag + sig * max_bins;
        const double f0 = (double)f[pk], f1 = 2.0 * f0;
        double s_sig = 0.0, s_noise = 0.0;
        int cnt = 0;
        for (int k = lane; k < nb; k += 32) {
          const double fk = (double)f[k], mk = (double)m[k];
          if (isfinite(mk) && lo <= fk && fk <= hi) {
            const double pw = square ? mk * mk : mk;
            ++cnt;
            if (fabs(fk - f0) <= hw || fabs(fk - f1) <= hw) s_sig += pw;
            else s_noise += pw;
          }
        }
        s_sig = warp_sum(s_sig);
        s_noise = warp_sum(s_noise);
        cnt = warp_sum(cnt);
        if (cnt >= 2) snr = 10.0 * log10(s_sig / s_noise);     // IEEE: 0/x -> -inf, x/0 -> +inf, 0/0 -> NaN
      }
      if (lane == 0) {
        snr_db[sig] = snr;
        if (gated_freq) gated_freq[sig] = snr >= min_snr_db ? peak_freq[sig] : nan_f64();
      }
    }
    if (gated_lag) {
      __syncthreads();                               // the job's snr_db row is written and visible to the CTA
      const double* row = snr_db + j * R;
      for (int a = warp; a < R - 1; a += nwarps) {
        const bool ok_a = row[a] >= min_snr_db;
        const long long q0 = (long long)a * (2LL * R - a - 1) / 2 - (a + 1);   // pair (a, b) is q0 + b
        for (int b = a + 1 + lane; b < R; b += 32) {
          const long long q = j * P + q0 + b;
          gated_lag[q] = ok_a && row[b] >= min_snr_db ? lag_sec[q] : nan_f64();
        }
      }
      __syncthreads();                               // the next job's warps may not run ahead of this one's reads
    }
  }
}

}  // namespace bpv

extern "C" int bpv_window_snr(const float* spec_f, const float* spec_mag, const int32_t* num_bins, const int32_t* peak_idx,
                              int64_t J, int32_t R, int32_t max_bins, int32_t transform, double lo, double hi,
                              double half_width, const double* peak_freq, const double* lag_sec, int32_t P, double min_snr_db,
                              double* snr_db, double* gated_freq, double* gated_lag, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(!isnan(lo) && !isnan(hi), BPV_E_INVALID, "bpv_window_snr: NaN band (%g, %g)", lo, hi);
  BPV_REQUIRE(isfinite(half_width) && half_width >= 0.0, BPV_E_INVALID, "bpv_window_snr: half width %g is not a finite value >= 0",
              half_width);
  BPV_REQUIRE(!isnan(min_snr_db), BPV_E_INVALID, "bpv_window_snr: NaN min_snr_db");
  BPV_REQUIRE(J >= 0 && R >= 1 && max_bins >= 1, BPV_E_INVALID, "bpv_window_snr: bad sizes (J %lld, R %d, max_bins %d)", (long long)J,
              R, max_bins);
  BPV_REQUIRE((long long)P == (long long)R * (R - 1) / 2, BPV_E_INVALID, "bpv_window_snr: P %d != R(R-1)/2 for R = %d", P, R);
  BPV_REQUIRE(transform == BPV_DFT_RFFT || transform == BPV_PGRAM_WELCH || transform == BPV_PGRAM_LS, BPV_E_INVALID,
              "bpv_window_snr: unknown spectrum transform %d", transform);
  BPV_REQUIRE(spec_f && spec_mag && num_bins && peak_idx && snr_db, BPV_E_INVALID, "bpv_window_snr: NULL pointer");
  BPV_REQUIRE(!gated_freq || peak_freq, BPV_E_INVALID, "bpv_window_snr: gated_freq needs peak_freq");
  BPV_REQUIRE(!gated_lag || lag_sec, BPV_E_INVALID, "bpv_window_snr: gated_lag needs lag_sec");
  if (J == 0) return 0;
  const int warps = R < SNR_MAX_WARPS ? R : SNR_MAX_WARPS;
  const unsigned grid = (unsigned)(J < (1LL << 30) ? J : (1LL << 30));
  window_snr_kernel<<<grid, 32 * warps, 0, (cudaStream_t)stream>>>(spec_f, spec_mag, num_bins, peak_idx, (long long)J, R, max_bins,
                                                                   transform == BPV_DFT_RFFT, lo, hi, half_width, peak_freq, lag_sec,
                                                                   P, min_snr_db, snr_db, gated_freq, P > 0 ? gated_lag : nullptr);
  return check_launch("window_snr_kernel");
}
