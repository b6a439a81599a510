// Device-side filter design in float64 (the reference re-designs its filters every frame for every
// signal because fs differs per stream: signal_processor.py:158-173, 226, 232).
#pragma once
#include "common.cuh"

namespace bpv {

constexpr int MAX_SOS = 16;     // butter_order <= 16 -> <= 16 second-order sections
constexpr int MAX_TAPS = 127;   // fir_taps <= 127 (odd)
// design cache (filters.cu): DC_SLOTS entries of [sos 16x6 | taps | zi | merged taps], keyed by the bits of fs
constexpr int DC_SLOTS = 256, DC_PROBES = 8, DC_HDR_BYTES = 16;
constexpr int FIR_MERGED_LEN = 264;  // merged filtfilt taps c[k] = ac[|k - (T-1)|], k = 0 .. 2T-2, zero padded (2T-1 <= 255; tiles read up to 260)
constexpr int FIR_WS_STRIDE = 256 + FIR_MERGED_LEN;   // doubles of filter workspace per window job: taps [128] | lfilter_zi [128] | merged taps [264]
constexpr int DC_STRIDE = MAX_SOS * 6 + FIR_WS_STRIDE;
constexpr long long DC_BYTES = DC_HDR_BYTES + (long long)DC_SLOTS * 8 + (long long)DC_SLOTS * DC_STRIDE * 8;

// status codes written to the per-signal status array
constexpr int ST_OK = 0, ST_GUARD = 1, ST_CUBIC_X = 2, ST_BAD_BANDS = 3;

// Job map of a ragged step (include/bpv.h bpv_stream_jobs): job k reads ring row stream[k], newest sample head[k].  The
// window kernels take it behind a template switch JMAP; the JMAP = false instantiations locate job j of stream s at
// head0 + j * head_step as before and never read the map.  With JMAP the launch's params carry S = number of jobs and
// jobs_per_stream = 1, so every per-job layout is the lockstep one over the job list.
struct JobMap {
  const int32_t* stream;
  const int64_t* head;
};

struct cplx { double re, im; };
__device__ __forceinline__ cplx cmul(cplx a, cplx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ cplx cdiv(cplx a, cplx b) {
  const double d = b.re * b.re + b.im * b.im;
  return {(a.re * b.re + a.im * b.im) / d, (a.im * b.re - a.re * b.im) / d};
}
__device__ __forceinline__ cplx csqrt_(cplx z) {  // principal square root
  const double r = hypot(z.re, z.im);
  if (r == 0.0) return {0.0, 0.0};
  double t = sqrt(0.5 * (r + fabs(z.re)));
  if (z.re >= 0.0) return {t, z.im / (2.0 * t)};
  return {fabs(z.im) / (2.0 * t), z.im >= 0.0 ? t : -t};
}

// Butterworth band-pass, output='sos' — scipy.signal.butter(N, [f1,f2], 'bandpass', output='sos', fs=fs)
// as called at signal_processor.py:160-162: buttap -> lp2bp_zpk -> bilinear_zpk -> zpk2sos('nearest')
// (scipy/signal/_filter_design.py).  sos: [N][6] row-major.  Returns ST_OK or ST_BAD_BANDS (scipy raises).
__device__ inline int butter_bandpass_sos(double fs, int N, double min_freq, double max_freq, double min_bw, double* sos) {
  const double f1 = fmin(min_freq, fs / 2 - 2 * min_bw), f2 = fmin(max_freq, fs / 2 - min_bw);
  const double W1 = f1 / (fs / 2), W2 = f2 / (fs / 2);
  if (!(W1 > 0.0 && W2 < 1.0 && W1 < W2) || N < 1 || N > MAX_SOS) {
    for (int i = 0; i < N * 6; ++i) sos[i] = nan_f64();
    return ST_BAD_BANDS;
  }
  const double PI = 3.141592653589793;
  const double w1 = 4.0 * tan(PI * W1 / 2.0), w2 = 4.0 * tan(PI * W2 / 2.0);
  const double bw = w2 - w1, wo = sqrt(w1 * w2);

  // one digital pole per conjugate pair (or a real pair), with its "distance to the unit circle" key
  double qre[MAX_SOS], qim[MAX_SOS], a1[MAX_SOS], a2[MAX_SOS], key[MAX_SOS];
  int np = 0;
  double kden = 1.0;  // prod over all 2N analog poles of (4 - p)  (real)
  for (int m = -N + 1; m <= N - 1; m += 2) {
    if (m < 0) continue;  // conjugates come for free
    const double th = PI * m / (2.0 * N);
    double s, c;
    sincos(th, &s, &c);
    const cplx plp = {-c * bw / 2.0, -s * bw / 2.0};
    cplx d = cmul(plp, plp);
    d.re -= wo * wo;
    const cplx r = csqrt_(d);
    if (m == 0) {
      // real low-pass pole -> either one conjugate pair or two real poles
      if (d.re < 0.0) {
        const cplx p = {plp.re, sqrt(-d.re)};
        const cplx q = cdiv({4.0 + p.re, p.im}, {4.0 - p.re, -p.im});
        kden *= (4.0 - p.re) * (4.0 - p.re) + p.im * p.im;
        qre[np] = q.re; qim[np] = fabs(q.im);
        a1[np] = -2.0 * q.re; a2[np] = q.re * q.re + q.im * q.im;
        key[np] = fabs(1.0 - sqrt(a2[np]));
      } else {
        const double sr = sqrt(d.re), pa = plp.re + sr, pb = plp.re - sr;
        const double qa = (4.0 + pa) / (4.0 - pa), qb = (4.0 + pb) / (4.0 - pb);
        kden *= (4.0 - pa) * (4.0 - pb);
        const double ka = fabs(1.0 - fabs(qa)), kb = fabs(1.0 - fabs(qb));
        qre[np] = ka <= kb ? qa : qb; qim[np] = 0.0;  // the "worst" of the two picks the zeros
        a1[np] = -(qa + qb); a2[np] = qa * qb;
        key[np] = fmin(ka, kb);
      }
      ++np;
    } else {
      for (int sgn = 0; sgn < 2; ++sgn) {
        const cplx p = sgn == 0 ? cplx{plp.re + r.re, plp.im + r.im} : cplx{plp.re - r.re, plp.im - r.im};
        const cplx q = cdiv({4.0 + p.re, p.im}, {4.0 - p.re, -p.im});
        kden *= (4.0 - p.re) * (4.0 - p.re) + p.im * p.im;  // (4-p)(4-conj p)
        qre[np] = q.re; qim[np] = fabs(q.im);
        a1[np] = -2.0 * q.re; a2[np] = q.re * q.re + q.im * q.im;
        key[np] = fabs(1.0 - sqrt(a2[np]));
        ++np;
      }
    }
  }
  // gain: k = bw^N * real(4^N / prod(4 - p))
  double k = 1.0;
  for (int i = 0; i < N; ++i) k *= bw * 4.0;
  k /= kden;

  // zpk2sos: worst pole (closest to the unit circle) goes to the LAST section; zeros (N at +1, N at -1)
  // are handed out nearest-first to the pole being placed.
  int zp = N, zm = N;
  bool used[MAX_SOS];
  for (int i = 0; i < np; ++i) used[i] = false;
  for (int si = np - 1; si >= 0; --si) {
    int w = -1;
    for (int i = 0; i < np; ++i)
      if (!used[i] && (w < 0 || key[i] < key[w])) w = i;
    used[w] = true;
    const double dp = hypot(qre[w] - 1.0, qim[w]), dm = hypot(qre[w] + 1.0, qim[w]);
    double z[2];
    for (int t = 0; t < 2; ++t) {
      const bool plus = (zp > 0) && (zm == 0 || dp <= dm);
      if (plus) { z[t] = 1.0; --zp; } else { z[t] = -1.0; --zm; }
    }
    double* o = sos + si * 6;
    o[0] = 1.0; o[1] = -(z[0] + z[1]); o[2] = z[0] * z[1];
    o[3] = 1.0; o[4] = a1[w]; o[5] = a2[w];
  }
  sos[0] *= k; sos[1] *= k; sos[2] *= k;
  return ST_OK;
}

// Band edges of the reference's FIR (signal_processor.py:164-169), normalised by Nyquist.  Returns false
// when scipy.signal.firls would raise ValueError (non-monotonic / outside [0, 1]).
__device__ inline bool firls_bands(double fs, double min_freq, double max_freq, double df, double* fb /*[6]*/) {
  const double nyq = fs / 2;
  fb[0] = 0.0;
  fb[1] = fmax(min_freq - df, df) / nyq;
  fb[2] = min_freq / nyq;
  fb[3] = max_freq / nyq;
  fb[4] = fmin(max_freq + df, nyq - df) / nyq;
  fb[5] = nyq / nyq;
  bool ok = isfinite(fs) && fs > 0;
  for (int b = 0; b < 3; ++b) ok = ok && (fb[2 * b + 1] - fb[2 * b] > 0.0);  // width > 0
  ok = ok && fb[1] <= fb[2] && fb[3] <= fb[4];                                // no overlap / ordered
  for (int i = 0; i < 6; ++i) ok = ok && fb[i] >= 0.0 && fb[i] <= 1.0;
  return ok;
}

__device__ __forceinline__ double np_sinc(double x) {  // numpy.sinc
  const double y = 3.141592653589793 * (x == 0.0 ? 1.0e-20 : x);
  return sin(y) / y;
}

}  // namespace bpv
