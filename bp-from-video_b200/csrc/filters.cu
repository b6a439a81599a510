// Filter-design kernels: one Butterworth SOS / one least-squares FIR per window job (the R ROIs of a
// job share the job's timestamps, hence fs, hence the filter).  float64 throughout.
#include "filters.cuh"

namespace bpv {

// ---- job sampling rate: Signal.get_fs (signal_data.py:55-58) over the job's window --------------
// fs = 1 / nanmean(diff(x[finite])) == (m-1) / (x_last - x_first).  After an INTERP_* step the
// reference uses 1/linspace-step, the same quantity up to rounding (signal_processor.py:211,218).
__device__ inline double job_fs(const double* __restrict__ ring_t, int cap, int window, long long head, int* m_out) {
  double first = 0, last = 0;
  int m = 0;
  long long g = head - window + 1;
  int k = 0;
  if (g < 0) { k = (int)(-g < window ? -g : window); g = 0; }     // samples before the stream started read as NaN
  int slot = (int)(g % cap);
  for (; k < window; ++k) {
    const double x = ring_t[slot];
    if (++slot == cap) slot = 0;
    if (isfinite(x)) { if (m == 0) first = x; last = x; ++m; }
  }
  if (m_out) *m_out = m;
  return m >= 2 ? 1.0 / ((last - first) / (double)(m - 1)) : nan_f64();
}

__global__ void butter_from_fs_kernel(const double* __restrict__ fs, int n, int order, double min_freq, double max_freq,
                                      double min_bw, double* __restrict__ sos_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double sos[MAX_SOS * 6];
  butter_bandpass_sos(fs[i], order, min_freq, max_freq, min_bw, sos);
  for (int k = 0; k < order * 6; ++k) sos_out[(long long)i * order * 6 + k] = sos[k];
}

// scipy.signal.firls (_fir_filter_design.py:1130-1171) with desired = [0,0,1,1,0,0], weight = 1 — FIRLS_LPD lanes
// per filter, 32 / FIRLS_LPD filters per warp.
//
// scipy solves Q a = b with Q = toeplitz(q[:M+1]) + hankel(q[:M+1], q[M:]) (Cholesky) and then mirrors a into
// the taps h = [a[M..1], 2 a0, a[1..M]].  Written for h directly, that is the symmetric positive-definite
// TOEPLITZ system  T h = y,  T[u][v] = q[|u-v|] (numtaps x numtaps), y = [b[M..1], b0, b[1..M]]:
// row i >= 0 of T h is 2 q[i] a0 + sum_{j>=1} (q[|i-j|] + q[i+j]) a[j] = (Q a)[i].  T is better conditioned
// than Q (cond 10 at 30 fps, 7e4 at 8.7 fps) and a Toeplitz solve is O(n^2): Levinson-Durbin, 126 steps of
// two dot products + two AXPYs of growing length, instead of a 64^3/3 factorisation.  Agreement with scipy's
// firls: <= 8e-13 relative over fs 8.7..240 Hz (checked against numpy in tests/test_window_gpu.py).
//
// The recursion is a chain of 126 dependent steps whose cost is dominated by per-step overhead (shuffle
// reductions, the reciprocal, warp syncs), not by the FMAs: with a whole warp per filter it issued 22 k warp
// instructions per design.  Here a group of FIRLS_LPD = 8 lanes owns a filter (element i lives on lane i % 8,
// register i / 8), so one warp instruction advances four designs, the reductions are 3 shuffle levels, and the
// band-edge sinc tables are built once per design (five sines per element, advanced by rotation along the lane's
// arithmetic progression of elements).
constexpr int FIRLS_LPD = 8;                        // lanes per design
constexpr int FIRLS_EPL = 128 / FIRLS_LPD;          // elements per lane
constexpr int FIRLS_DPW = 32 / FIRLS_LPD;           // designs per warp
constexpr int FIRLS_WARPS = 2;                      // warps per CTA
constexpr int FIRLS_THREADS = 32 * FIRLS_WARPS;
constexpr int FIRLS_DPB = FIRLS_DPW * FIRLS_WARPS;  // designs per CTA
// doubles of shared memory per design: pad | r [128] | pad | f ping [128] | pad | f pong [128] | b [64].  The zero pads
// (FIRLS_PAD >= 2 * LPD - 1 doubles) make r[k-i] and f_old[k-i] readable as 0 for the lanes whose element i lies
// beyond k, so the element loops carry no per-lane predicate.  Odd designs are shifted by 8 doubles so that the four
// groups of a warp read different bank halves.  Sized so that 7 CTAs (56 designs) fit an SM: 8192 designs = one wave.
constexpr int FIRLS_PAD = 16;
constexpr int FIRLS_WS = 3 * (FIRLS_PAD + 128) + 64;
// design d of the CTA: regions never overlap, bases are 0, 8, 8, 0 (mod 16 doubles) within a warp
__host__ __device__ constexpr int firls_smem_offset(int d) { return d * FIRLS_WS + ((d + 1) >> 1) * 8; }
__device__ __forceinline__ double group_sum_d(double v) {
#pragma unroll
  for (int o = FIRLS_LPD / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// Executed by whole warps: every lane group works on its own design (fs, out, zi_out, smem differ per group);
// `live` = false for padding groups (they compute a shadow design and write nothing).
//
// Step k of Levinson-Durbin on T (f = forward vector of length k, zero extended; x = solution of the leading k x k system):
//   ef = sum_i r[k-i] f[i],  ex = sum_i r[k-i] x[i]                     (two dot products, one shared r load)
//   f'[i]      = (f[i] - ef * f[k-i]) / (1 - ef^2)
//   rev(f')[i] = (f[k-i] - ef * f[i]) / (1 - ef^2)                      (the backward vector, from the same operands)
//   x'[i]      = x[i] + (y[k] - ex) * rev(f')[i]
// so one pass over the elements updates both vectors with a single reversed read of the old f from shared memory.
__device__ void firls_design_group(double fs, bool live, int taps, double min_freq, double max_freq, double df,
                                   double* __restrict__ out, double* __restrict__ zi_out, double* __restrict__ ac_out,
                                   double* smem) {
  const int M = (taps - 1) / 2, n = taps;
  double* r = smem + FIRLS_PAD;                 // [128] first column of T: q[0 .. taps-1]; r[-PAD .. -1] = 0
  double* fA = r + 128 + FIRLS_PAD;             // forward vector, ping (fA[-PAD .. -1] = 0)
  double* fB = fA + 128 + FIRLS_PAD;            // forward vector, pong (fB[-PAD .. -1] = 0)
  double* bt = fB + 128;                        // [64] b[d]; the symmetric right-hand side is y[i] = b[|i - M|]
  const int sub = threadIdx.x & (FIRLS_LPD - 1);
  double fb[6];
  const bool ok = firls_bands(fs, min_freq, max_freq, df, fb);
  if (!ok) firls_bands(30.0, 0.8, 4.0, 0.3, fb);     // keep the group in step with the warp; NaN written at the end
  // q[i] = sum_bands f2 sinc(f2 i) - f1 sinc(f1 i);  b[d] = f3 sinc(f3 d) - f2 sinc(f2 d)  (band edges fb[0..5])
  // the b table is parked in fA / fB until y is in registers
  // The lane's elements i = sub + 8 m are an arithmetic progression, so sin(pi f i) is advanced by the stable rotation
  // s += c * beta - s * alpha, c -= s * beta + c * alpha (alpha = 2 sin^2(4 pi f), beta = sin(8 pi f)) from one exact
  // sincospi at i = sub: 15 trigonometric calls per lane instead of 80, and one reciprocal 1 / (pi i) per element
  // instead of five divisions (the 15 rotations stay within 3e-14 of the exact sines; numpy's own sin(pi * (f * i)) is
  // 6e-14 off through the rounding of its argument — checked against mpmath over the band-edge range).
  double sn[5], cs[5], al[5], be[5];
#pragma unroll
  for (int b = 0; b < 5; ++b) {
    const double f = fb[b + 1];
    sincospi(f * (double)sub, &sn[b], &cs[b]);
    const double sh = sinpi(f * (double)(FIRLS_LPD / 2));
    al[b] = 2.0 * sh * sh;
    be[b] = sinpi(f * (double)FIRLS_LPD);
  }
#pragma unroll 1
  for (int i = sub; i < 128; i += FIRLS_LPD) {
    double acc = 0.0, s2 = 0.0, s3 = 0.0;
    if (i < taps) {
      const double inv = 1.0 / (3.141592653589793 * (double)i);        // unused (inf) for i == 0
      double t[5];
#pragma unroll
      for (int b = 0; b < 5; ++b) t[b] = i == 0 ? fb[b + 1] : sn[b] * inv;   // f sinc(f i) = sin(pi f i) / (pi i)
      s2 = t[1]; s3 = t[2];
      acc = t[0] + (t[2] - t[1]) + (t[4] - t[3]);     // fb[0] = 0 contributes f sinc = 0
    }
    r[i] = acc;
    fA[i] = s2; fB[i] = s3;
#pragma unroll
    for (int b = 0; b < 5; ++b) {
      const double s0 = sn[b], c0 = cs[b];
      sn[b] = s0 + fma(c0, be[b], -s0 * al[b]);
      cs[b] = c0 - fma(s0, be[b], c0 * al[b]);
    }
  }
  for (int i = sub; i < FIRLS_PAD; i += FIRLS_LPD) { r[i - FIRLS_PAD] = 0.0; fA[i - FIRLS_PAD] = 0.0; fB[i - FIRLS_PAD] = 0.0; }
  __syncwarp();
  for (int d = sub; d <= M; d += FIRLS_LPD) bt[d] = fB[d] - fA[d];
  __syncwarp();
  for (int i = sub; i < 128; i += FIRLS_LPD) { fA[i] = 0.0; fB[i] = 0.0; }
  __syncwarp();
  double f[FIRLS_EPL], x[FIRLS_EPL];
#pragma unroll
  for (int m = 0; m < FIRLS_EPL; ++m) { f[m] = 0.0; x[m] = 0.0; }
  double dmin = 1.0;
  const double r0inv = 1.0 / r[0];
  if (sub == 0) { f[0] = r0inv; x[0] = bt[M] * r0inv; fA[0] = r0inv; }
  __syncwarp();
#pragma unroll 1
  for (int k = 1; k < n; ++k) {
    const double* fo = ((k - 1) & 1) ? fB : fA;      // f of step k-1 (length k, zero beyond)
    double* fn = (k & 1) ? fB : fA;                  // f of step k (length k+1)
    const int mmax = k / FIRLS_LPD;                  // last element register that can be non-zero (warp uniform)
    const double* rk = r + (k - sub);                // r[k - i] = rk[-LPD * m]
    const double* fk = fo + (k - sub);               // f_old[k - i]
    double ef0 = 0.0, ef1 = 0.0, ex0 = 0.0, ex1 = 0.0;
    // Duff-style entry into the unrolled element blocks (highest live block first, fall through to block 0): one
    // indexed branch per loop and no exit paths, so f[] / x[] stay pinned in their registers.
#define FIRLS_DOT(m)                                                           \
    { const double ra = rk[-FIRLS_LPD * (m)], rb = rk[-FIRLS_LPD * ((m) + 1)]; \
      ef0 = fma(ra, f[m], ef0); ex0 = fma(ra, x[m], ex0);                      \
      ef1 = fma(rb, f[(m) + 1], ef1); ex1 = fma(rb, x[(m) + 1], ex1); }
    switch (mmax >> 1) {
      case 7: FIRLS_DOT(14)
      case 6: FIRLS_DOT(12)
      case 5: FIRLS_DOT(10)
      case 4: FIRLS_DOT(8)
      case 3: FIRLS_DOT(6)
      case 2: FIRLS_DOT(4)
      case 1: FIRLS_DOT(2)
      default: FIRLS_DOT(0)
    }
#undef FIRLS_DOT
    const int dk = k < M ? M - k : k - M;
    const double ykk = bt[dk];
    const double ef = group_sum_d(ef0 + ef1), ex = group_sum_d(ex0 + ex1);
    const double den2 = 1.0 - ef * ef;               // 1 - (reflection coefficient)^2 = ratio of successive leading minors
    dmin = fmin(dmin, den2);
    const double dinv = 1.0 / den2;
    const double gd = (ykk - ex) * dinv;
    double* fw = fn + sub;
#define FIRLS_UPD(m)                                                           \
    { const double frev = fk[-FIRLS_LPD * (m)], fold = f[m];                   \
      const double fnew = (fold - ef * frev) * dinv;                           \
      x[m] = fma(gd, frev - ef * fold, x[m]);                                  \
      f[m] = fnew; fw[FIRLS_LPD * (m)] = fnew; }
    switch (mmax) {
      case 15: FIRLS_UPD(15)
      case 14: FIRLS_UPD(14)
      case 13: FIRLS_UPD(13)
      case 12: FIRLS_UPD(12)
      case 11: FIRLS_UPD(11)
      case 10: FIRLS_UPD(10)
      case 9: FIRLS_UPD(9)
      case 8: FIRLS_UPD(8)
      case 7: FIRLS_UPD(7)
      case 6: FIRLS_UPD(6)
      case 5: FIRLS_UPD(5)
      case 4: FIRLS_UPD(4)
      case 3: FIRLS_UPD(3)
      case 2: FIRLS_UPD(2)
      case 1: FIRLS_UPD(1)
      default: FIRLS_UPD(0)
    }
#undef FIRLS_UPD
    __syncwarp();
  }
  // scipy solves Q a = b by Cholesky and, when LAPACK reports the matrix rank deficient / ill-conditioned (rcond < eps),
  // falls back to lstsq (_fir_filter_design.py:1156-1168).  The Toeplitz recursion has no such fallback: a leading minor
  // ratio at rounding level is reported as a failed design (NaN taps -> status 3 -> ValueError in the drop-in) instead of
  // returning taps that differ from the reference's.  Unreachable for the reference's band layout (cond(T) <= 7e4, i.e.
  // 1 - ef^2 >= 1e-5, over every valid fs).
  const bool solved = dmin > 1.0e-13;
  // taps out (NaN when scipy would raise), staged through shared memory for lfilter_zi
  double* hs = r;                                                 // [128] taps, zero padded
  __syncwarp();
#pragma unroll
  for (int m = 0; m < FIRLS_EPL; ++m) {
    const int i = sub + FIRLS_LPD * m;
    hs[i] = i < n ? x[m] : 0.0;
    if (live && i < n) out[i] = (ok && solved) ? x[m] : nan_f64();
  }
  __syncwarp();
  if (zi_out && live) {
    // lfilter_zi(b, [1]) = suffix sums of b[1:] (scipy/signal/_signaltools.py:4440-4463): zi[i] = sum_{k>i} b[k].
    // Lane `sub` owns the contiguous block [16 sub, 16 sub + 16): local suffix sums + the totals of higher blocks.
    double tot = 0.0;
#pragma unroll
    for (int e = 0; e < FIRLS_EPL; ++e) tot += hs[FIRLS_EPL * sub + e];
    double above = 0.0;                                           // sum of the blocks of lanes > sub
#pragma unroll
    for (int o = 1; o < FIRLS_LPD; ++o) {
      const double t = __shfl_down_sync(0xffffffffu, tot, o, FIRLS_LPD);
      if (sub + o < FIRLS_LPD) above += t;
    }
    double run = above;
#pragma unroll
    for (int e = FIRLS_EPL - 1; e >= 0; --e) {
      const int i = FIRLS_EPL * sub + e;
      if (i < n - 1) zi_out[i] = ok ? run : nan_f64();
      run += hs[i];
    }
  }
  if (ac_out) {
    // Autocorrelation of the taps, ac[d] = sum_i h[i] h[i+d] (d = 0 .. 127; 0 beyond taps-1): filtfilt's forward and
    // backward passes merged into ONE symmetric filter h * rev(h) of 2*taps-1 coefficients ac[|k|], which the
    // preprocessing kernel applies wherever the padding keeps the initial-condition terms out of the cropped output
    // (window_pre.cu fir_merged).  Lane `sub` owns the 16 consecutive lags [16 sub, 16 sub + 16) as a register-tiled
    // sliding dot product; hs[] is zero beyond the taps (r's pad in front of fA), so no bounds are tested.
    constexpr int E = FIRLS_EPL;
    const int d0 = E * sub;
    double acc[E], wv[E];
#pragma unroll
    for (int e = 0; e < E; ++e) { acc[e] = 0.0; wv[e] = hs[d0 + e]; }
    const int nblk = (128 - d0) / E;                 // h[i + d] == 0 for i >= 128 - d0
#pragma unroll 1
    for (int blk = 0; blk < nblk; ++blk) {
      const double* hc = hs + blk * E;
      const double* hn = hs + blk * E + d0 + E;
#pragma unroll
      for (int ii = 0; ii < E; ++ii) {
        const double ck = hc[ii];
#pragma unroll
        for (int e = 0; e < E; ++e) acc[e] = fma(ck, wv[(e + ii) % E], acc[e]);
        wv[ii] = hn[ii];                             // h[i + d0 + E] replaces h[i + d0]
      }
    }
    if (live) {
      // written out as the symmetric filter itself, c[k] = ac[|k - Mt|] for k = 0 .. 2 Mt (Mt = taps - 1), zero up to
      // FIR_MERGED_LEN: the preprocessing kernel's tiles read c[] straight from here (no per-signal copy into shared memory)
      const int Mt = n - 1;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int d = d0 + e;
        const double v = ok ? acc[e] : nan_f64();
        if (d <= Mt) { ac_out[Mt - d] = v; ac_out[Mt + d] = v; }
      }
      for (int k = 2 * Mt + 1 + sub; k < FIR_MERGED_LEN; k += FIRLS_LPD) ac_out[k] = 0.0;
    }
  }
}

__global__ void __launch_bounds__(FIRLS_THREADS) firls_from_fs_kernel(const double* __restrict__ fs, int n, int taps, double min_freq,
                                                                      double max_freq, double df, double* __restrict__ out) {
  extern __shared__ double smem[];
  const int d = threadIdx.x / FIRLS_LPD, job = blockIdx.x * FIRLS_DPB + d;
  const bool live = job < n;
  firls_design_group(live ? fs[job] : 30.0, live, taps, min_freq, max_freq, df, out + (long long)(live ? job : 0) * taps, nullptr,
                     nullptr, smem + firls_smem_offset(d));
}

// ---- per-job design from the ring timestamps (used by the window pipeline) ----------------------
// JMAP: the job's ring row and newest sample come from the job map (filters.cuh JobMap), else from head0 / head_step
template <bool JMAP>
__global__ void job_butter_kernel(const double* __restrict__ ring_t, bpv_window_params p, double* __restrict__ sos_out,
                                  const JobMap jm) {
  const int job = blockIdx.x * blockDim.x + threadIdx.x;
  const int J = p.S * p.jobs_per_stream;
  if (job >= J) return;
  const int s = JMAP ? jm.stream[job] : job / p.jobs_per_stream, j = JMAP ? 0 : job % p.jobs_per_stream;
  const long long head = JMAP ? (long long)jm.head[job] : p.head0 + (long long)j * p.head_step;
  const double fs = job_fs(ring_t + (long long)s * p.cap, p.cap, p.window, head, nullptr);
  double sos[MAX_SOS * 6];
  if (isfinite(fs)) butter_bandpass_sos(fs, p.butter_order, p.min_freq, p.max_freq, p.butter_min_bw, sos);
  else for (int k = 0; k < p.butter_order * 6; ++k) sos[k] = nan_f64();
  for (int k = 0; k < p.butter_order * 6; ++k) sos_out[(long long)job * (MAX_SOS * 6) + k] = sos[k];   // slot stride 16 x 6 whatever the order
}

// fs of a job's window, cooperative over a group of FIRLS_LPD lanes (first / last finite timestamp and their count); every
// lane of the group returns the same value.  Same arithmetic as job_fs.
template <bool JMAP>
__device__ __forceinline__ double group_job_fs(const double* __restrict__ ring_t, const bpv_window_params& p, int job, int sub,
                                               const JobMap& jm) {
  const int s = JMAP ? jm.stream[job] : job / p.jobs_per_stream, j = JMAP ? 0 : job % p.jobs_per_stream;
  const double* rt = ring_t + (long long)s * p.cap;
  const long long g0 = (JMAP ? (long long)jm.head[job] : p.head0 + (long long)j * p.head_step) - p.window + 1;
  int lo = 0x7fffffff, hi = -1, cnt = 0;
  const int kmin = g0 < 0 ? (int)(-g0 < p.window ? -g0 : p.window) : 0;
  const int slot0 = (int)(((g0 % p.cap) + p.cap) % p.cap);
  for (int k0 = sub; k0 < p.window; k0 += FIRLS_LPD * 8) {     // 8 independent loads in flight per lane
    double tv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int k = k0 + u * FIRLS_LPD;
      int slot = slot0 + k; if (slot >= p.cap) slot -= p.cap;
      tv[u] = (k < p.window && k >= kmin) ? rt[slot] : nan_f64();
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int k = k0 + u * FIRLS_LPD;
      if (isfinite(tv[u])) { lo = lo < k ? lo : k; hi = k; ++cnt; }
    }
  }
  for (int o = FIRLS_LPD / 2; o > 0; o >>= 1) {
    const int l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
    lo = lo < l2 ? lo : l2; hi = hi > h2 ? hi : h2; cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  double fs = nan_f64();
  if (cnt >= 2) fs = 1.0 / ((rt[(slot0 + hi) % p.cap] - rt[(slot0 + lo) % p.cap]) / (double)(cnt - 1));
  return fs;
}

template <bool JMAP>
__global__ void __launch_bounds__(FIRLS_THREADS) job_firls_kernel(const double* __restrict__ ring_t, bpv_window_params p,
                                                                  double* __restrict__ out, const JobMap jm) {
  extern __shared__ double smem[];
  const int d = threadIdx.x / FIRLS_LPD, sub = threadIdx.x & (FIRLS_LPD - 1);
  const int job = blockIdx.x * FIRLS_DPB + d;
  const bool live = job < p.S * p.jobs_per_stream;
  // padding groups shadow job 0 (warp-uniform control flow), write nothing
  const double fs = group_job_fs<JMAP>(ring_t, p, live ? job : 0, sub, jm);
  double* o = out + (long long)(live ? job : 0) * FIR_WS_STRIDE;      // taps [128] | lfilter_zi [128] | merged taps [FIR_MERGED_LEN]
  firls_design_group(fs, live, p.fir_taps, p.min_freq, p.max_freq, p.fir_df, o, o + 128, o + 256, smem + firls_smem_offset(d));
}

// ---------------------------------------------------------------------------------------------
// Design cache.  make_filter is a pure function of the window's sampling rate (the band edges, order and tap count are
// fixed per processor), yet the reference calls it for every signal of every frame (signal_processor.py:226, 232).  A
// stream with a constant frame period — every video file, and the synthetic c2 workload — yields the same fs, bit for
// bit, window after window, and streams that share a clock share it too.  The cache is an open-addressing table in
// device memory keyed by the 64 bits of fs, persistent across launches:
//   probe   (one 8-lane group per window job) computes fs, looks it up and, on a miss, claims a slot with one
//           atomicCAS and appends (destination, fs) to the launch's miss list; a full neighbourhood (DC_PROBES slots)
//           or a non-finite fs falls back to the job's own workspace slot;
//   design  kernels run the Levinson / Butterworth design for the entries of the miss list only (CTAs beyond it exit);
//   filter  (window_pre.cu) reads each job's coefficients through ref[job]: a cache slot, or its own workspace slot.
// Hits return the very bits a fresh design would produce (the design kernels are deterministic in fs), so cached and
// uncached runs are identical.  Jittered timestamps give all-distinct fs: the table fills, later jobs use their own
// slots, and a launch that missed more than half the table clears the keys so stale rates do not squat in it.
// The table is only valid for one set of filter parameters: the owner zeroes it when they change.
// Layout of the cache buffer: hdr [16 B: miss counter] | keys u64 [DC_SLOTS] | vals double [DC_SLOTS][DC_STRIDE].
// ---------------------------------------------------------------------------------------------
struct DesignMiss { int32_t target; int32_t pad; double fs; };     // target >= 0: cache slot; < 0: own slot of job -(target + 1)

__device__ __forceinline__ unsigned dc_hash(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33;
  return (unsigned)k & (DC_SLOTS - 1);
}

template <bool JMAP>
__global__ void __launch_bounds__(256) design_probe_kernel(const double* __restrict__ ring_t, const bpv_window_params p,
                                                           unsigned char* __restrict__ cache, int32_t* __restrict__ ref,
                                                           DesignMiss* __restrict__ miss, const JobMap jm) {
  const int J = p.S * p.jobs_per_stream;
  const int job = (blockIdx.x * blockDim.x + threadIdx.x) / FIRLS_LPD, sub = threadIdx.x & (FIRLS_LPD - 1);
  const bool live = job < J;
  const double fs = group_job_fs<JMAP>(ring_t, p, live ? job : 0, sub, jm);
  if (!live || sub != 0) return;
  unsigned int* counter = reinterpret_cast<unsigned int*>(cache);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(cache + DC_HDR_BYTES);
  int slot = -1;
  bool fresh = false;
  if (isfinite(fs) && fs > 0.0) {
    const unsigned long long key = (unsigned long long)__double_as_longlong(fs);
    unsigned h = dc_hash(key);
    for (int probe = 0; probe < DC_PROBES; ++probe) {
      unsigned long long k = *reinterpret_cast<volatile unsigned long long*>(keys + h);
      if (k == 0ULL) {
        k = atomicCAS(keys + h, 0ULL, key);
        if (k == 0ULL) { slot = (int)h; fresh = true; break; }
      }
      if (k == key) { slot = (int)h; break; }
      h = (h + 1) & (DC_SLOTS - 1);
    }
  }
  ref[job] = slot;
  if (slot < 0 || fresh) {
    const unsigned e = atomicAdd(counter, 1u);
    miss[e].target = slot >= 0 ? slot : -(job + 1);
    miss[e].fs = fs;
  }
}

__device__ __forceinline__ double* dc_dest(int target, unsigned char* cache, double* ws_sos, double* ws_fir, bool fir) {
  if (target >= 0) {
    double* v = reinterpret_cast<double*>(cache + DC_HDR_BYTES + DC_SLOTS * 8) + (long long)target * DC_STRIDE;
    return fir ? v + MAX_SOS * 6 : v;
  }
  const long long job = -(long long)target - 1;
  return fir ? ws_fir + job * FIR_WS_STRIDE : ws_sos + job * (MAX_SOS * 6);
}

__device__ __forceinline__ void dc_maybe_clear(unsigned char* cache, unsigned nmiss) {
  // a launch that missed more than half the table: its rates do not repeat — empty the table for whatever comes next.
  // Nothing reads the keys between this launch's probe and the next one's; the values designed now stay where ref[] says.
  if (blockIdx.x == 0 && nmiss > DC_SLOTS / 2) {
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(cache + DC_HDR_BYTES);
    for (int i = threadIdx.x; i < DC_SLOTS; i += blockDim.x) keys[i] = 0ULL;
  }
}

__global__ void __launch_bounds__(FIRLS_THREADS) miss_firls_kernel(const bpv_window_params p, unsigned char* __restrict__ cache,
                                                                   const DesignMiss* __restrict__ miss, double* __restrict__ ws_sos,
                                                                   double* __restrict__ ws_fir) {
  extern __shared__ double smem[];
  const unsigned nmiss = *reinterpret_cast<const unsigned int*>(cache);
  dc_maybe_clear(cache, nmiss);
  if (blockIdx.x * FIRLS_DPB >= nmiss) return;
  const int d = threadIdx.x / FIRLS_LPD;
  const unsigned e = blockIdx.x * FIRLS_DPB + d;
  const bool live = e < nmiss;
  const DesignMiss m = miss[live ? e : 0];
  double* o = dc_dest(m.target, cache, ws_sos, ws_fir, true);
  firls_design_group(m.fs, live, p.fir_taps, p.min_freq, p.max_freq, p.fir_df, o, o + 128, o + 256, smem + firls_smem_offset(d));
}

__global__ void miss_butter_kernel(const bpv_window_params p, unsigned char* __restrict__ cache, const DesignMiss* __restrict__ miss,
                                   double* __restrict__ ws_sos, double* __restrict__ ws_fir) {
  const unsigned nmiss = *reinterpret_cast<const unsigned int*>(cache);
  dc_maybe_clear(cache, nmiss);
  const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nmiss) return;
  const DesignMiss m = miss[e];
  double sos[MAX_SOS * 6];
  if (isfinite(m.fs)) butter_bandpass_sos(m.fs, p.butter_order, p.min_freq, p.max_freq, p.butter_min_bw, sos);
  else for (int k = 0; k < p.butter_order * 6; ++k) sos[k] = nan_f64();
  double* o = dc_dest(m.target, cache, ws_sos, ws_fir, false);
  for (int k = 0; k < p.butter_order * 6; ++k) o[k] = sos[k];
}

constexpr size_t FIRLS_SMEM = (size_t)(firls_smem_offset(FIRLS_DPB - 1) + FIRLS_WS) * sizeof(double);

// jm = NULL: the lockstep instantiations (head0 / head_step); else the job-map ones
int launch_job_butter(const double* ring_t, const bpv_window_params& p, double* sos_out, cudaStream_t st, const JobMap* jm) {
  const int J = p.S * p.jobs_per_stream;
  if (jm) job_butter_kernel<true><<<(J + 63) / 64, 64, 0, st>>>(ring_t, p, sos_out, *jm);
  else job_butter_kernel<false><<<(J + 63) / 64, 64, 0, st>>>(ring_t, p, sos_out, JobMap{});
  return check_launch("job_butter_kernel");
}

int launch_job_firls(const double* ring_t, const bpv_window_params& p, double* taps_out, cudaStream_t st, const JobMap* jm) {
  const int J = p.S * p.jobs_per_stream;
  if (jm) job_firls_kernel<true><<<(J + FIRLS_DPB - 1) / FIRLS_DPB, FIRLS_THREADS, FIRLS_SMEM, st>>>(ring_t, p, taps_out, *jm);
  else job_firls_kernel<false><<<(J + FIRLS_DPB - 1) / FIRLS_DPB, FIRLS_THREADS, FIRLS_SMEM, st>>>(ring_t, p, taps_out, JobMap{});
  return check_launch("job_firls_kernel");
}

// Cached design of every window job: probe + design of the misses.  ref int32 [J] and the miss list live in the caller's
// workspace (window_pre.cu lays it out); `cache` is the persistent table (zero-initialised by its owner).
int launch_design_cached(const double* ring_t, const bpv_window_params& p, bool butter, bool fir, unsigned char* cache,
                         int32_t* ref, void* miss, double* ws_sos, double* ws_fir, cudaStream_t st, const JobMap* jm) {
  const int J = p.S * p.jobs_per_stream;
  cudaError_t e = cudaMemsetAsync(cache, 0, 4, st);                       // the launch's miss counter
  if (e != cudaSuccess) { set_error("bpv_window_design: cudaMemsetAsync: %s", cudaGetErrorString(e)); return (int)e; }
  const long long threads = (long long)J * FIRLS_LPD;
  const unsigned blocks = (unsigned)((threads + 255) / 256);
  if (jm) design_probe_kernel<true><<<blocks, 256, 0, st>>>(ring_t, p, cache, ref, (DesignMiss*)miss, *jm);
  else design_probe_kernel<false><<<blocks, 256, 0, st>>>(ring_t, p, cache, ref, (DesignMiss*)miss, JobMap{});
  if (int rc = check_launch("design_probe_kernel")) return rc;
  if (butter) {
    miss_butter_kernel<<<(J + 63) / 64, 64, 0, st>>>(p, cache, (const DesignMiss*)miss, ws_sos, ws_fir);
    if (int rc = check_launch("miss_butter_kernel")) return rc;
  }
  if (fir) {
    miss_firls_kernel<<<(J + FIRLS_DPB - 1) / FIRLS_DPB, FIRLS_THREADS, FIRLS_SMEM, st>>>(p, cache, (const DesignMiss*)miss, ws_sos, ws_fir);
    if (int rc = check_launch("miss_firls_kernel")) return rc;
  }
  return 0;
}

int check_filter_params(const bpv_window_params* p, const char* who) {
  BPV_REQUIRE(p, BPV_E_INVALID, "%s: NULL params", who);
  BPV_REQUIRE(p->butter_order >= 1 && p->butter_order <= MAX_SOS, BPV_E_TOO_LARGE, "%s: butter_order must be 1..16", who);
  BPV_REQUIRE(p->fir_taps >= 3 && p->fir_taps <= MAX_TAPS && (p->fir_taps & 1), BPV_E_TOO_LARGE,
              "%s: fir_taps must be odd and <= 127", who);
  return 0;
}

}  // namespace bpv

extern "C" int bpv_butter_sos_design(const double* fs, int32_t n, const bpv_window_params* p, double* sos_out, void* stream) {
  using namespace bpv;
  if (int rc = check_filter_params(p, "bpv_butter_sos_design")) return rc;
  BPV_REQUIRE(fs && sos_out && n >= 0, BPV_E_INVALID, "bpv_butter_sos_design: bad arguments");
  if (n == 0) return 0;
  butter_from_fs_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(fs, n, p->butter_order, p->min_freq, p->max_freq,
                                                                        p->butter_min_bw, sos_out);
  return check_launch("bpv_butter_sos_design");
}

extern "C" int bpv_firls_design(const double* fs, int32_t n, const bpv_window_params* p, double* taps_out, void* stream) {
  using namespace bpv;
  if (int rc = check_filter_params(p, "bpv_firls_design")) return rc;
  BPV_REQUIRE(fs && taps_out && n >= 0, BPV_E_INVALID, "bpv_firls_design: bad arguments");
  if (n == 0) return 0;
  firls_from_fs_kernel<<<(n + FIRLS_DPB - 1) / FIRLS_DPB, FIRLS_THREADS, FIRLS_SMEM, (cudaStream_t)stream>>>(fs, n, p->fir_taps, p->min_freq, p->max_freq, p->fir_df, taps_out);
  return check_launch("bpv_firls_design");
}
