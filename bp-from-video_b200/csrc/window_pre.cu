// F2 — window preprocessing (SignalProcessor.process_signal, signal_processor.py:196-241), batched
// over window jobs.  One warp per signal (job x ROI); the window lives in that warp's slice of shared
// memory; everything is float64 (the reference's dtype; fp32 IIR state loses up to 15 % of the
// peak at 120 fps, SURVEY.md §7).  Filters come from the per-job design kernels (filters.cu).
//
// Work layout inside a warp
//   gather      lanes stride the window, ballot/popc-compact valid samples (NaN-aware masks v, w)
//   diff/detrend lane-strided elementwise + warp-shuffle reductions
//   interp      lane-strided evaluation with per-lane binary search; the not-a-knot spline's
//               tridiagonal solve is a serial Thomas sweep on lane 0 (latency hidden by other warps)
//   sosfiltfilt 16 biquads = 16 lanes of a systolic cascade: lane s owns section s, samples flow
//               lane to lane by __shfl_up (one sample enters per step), forward then backward
//   FIR filtfilt register-tiled sliding dot product (corr_tile.cuh), 8 consecutive outputs per lane; only
//               the part of the padded signal that reaches the cropped output is staged and computed
#include <stdlib.h>
#include "filters.cuh"
#include "corr_tile.cuh"

namespace bpv {

int launch_job_butter(const double* ring_t, const bpv_window_params& p, double* sos_out, cudaStream_t st, const JobMap* jm);
int launch_job_firls(const double* ring_t, const bpv_window_params& p, double* taps_out, cudaStream_t st, const JobMap* jm);
int check_filter_params(const bpv_window_params* p, const char* who);
int launch_design_cached(const double* ring_t, const bpv_window_params& p, bool butter, bool fir, unsigned char* cache,
                         int32_t* ref, void* miss, double* ws_sos, double* ws_fir, cudaStream_t st, const JobMap* jm);

// Where a window job's filter coefficients live: in the design cache (ref[job] = slot) or in the job's own workspace slot.
struct DesignRef {
  const double* sos_ws;            // [J][16*6]
  const double* taps_ws;           // [J][FIR_WS_STRIDE]
  const int32_t* ref;              // [J] cache slot or -1; NULL = no cache in use
  const unsigned char* cache;
  __device__ __forceinline__ const double* slot(long long job) const {
    const int sl = ref ? ref[job] : -1;
    return sl >= 0 ? reinterpret_cast<const double*>(cache + DC_HDR_BYTES + DC_SLOTS * 8) + (long long)sl * DC_STRIDE : nullptr;
  }
  __device__ __forceinline__ const double* sos(long long job) const {
    const double* v = slot(job);
    return v ? v : sos_ws + job * (MAX_SOS * 6);
  }
  __device__ __forceinline__ const double* fir(long long job) const {
    const double* v = slot(job);
    return v ? v + MAX_SOS * 6 : taps_ws + job * FIR_WS_STRIDE;
  }
};

struct PreLayout {        // per-warp shared-memory plan, in bytes
  int yv, xv, posv, posb, buf0, buf1, coef, total;
  int buf_len;            // doubles in buf0
  // FIR sub-plan inside buf0 (doubles): merged path  XT [0, fir_c) | c [fir_c, fir_c + Kmax)
  //                                     two-pass path XT [0, fir_gt) | GT [fir_gt, fir_b)
  int fir_c, fir_gt, fir_b;
};

__host__ __device__ inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
// two-pass FIR (windows shorter than the filter): leading dimensions of the de-interleaved operand buffers
__host__ __device__ inline int fir_ld_fwd(int n, int T) {
  int LD = (round_up(T, 8) + n + T + 15) / 8 + 1;
  LD += (6 - (LD & 3)) & 3;   // LD = 2 (mod 4): the 8 rows of XT start 4 banks apart, the extension stores without conflicts
  return LD;
}
__host__ __device__ inline int fir_ld_bwd(int n, int T) { return (round_up(T, 10) + n + T + 20) / 10 + 1; }
// merged FIR: 2T-1 taps padded to a multiple of the tile, outputs m = 0 .. n-1 at storage index m + K
__host__ __device__ inline int fir_merged_k(int T, int RT) { return round_up(2 * T - 1, RT); }
__host__ __device__ inline int fir_merged_ld(int n, int T, int RT) { return (fir_merged_k(T, RT) / RT + (n + RT - 1) / RT) | 1; }

__host__ __device__ inline PreLayout pre_layout(const bpv_window_params& p) {
  bool interp = false, cubic = false, butter = false, fir = false;
  for (int i = 0; i < p.num_methods; ++i) {
    const int m = p.methods[i];
    interp |= (m == BPV_INTERP_LINEAR || m == BPV_INTERP_CUBIC);
    cubic |= m == BPV_INTERP_CUBIC;
    butter |= m == BPV_FILTER_BUTTER;
    fir |= m == BPV_FILTER_FIR;
  }
  const int W = p.window;
  int pad = 0;
  if (butter) pad = 3 * (2 * p.butter_order + 1);      // sosfiltfilt works on the whole odd-extended signal
  if (pad > W - 1) pad = W - 1 > 0 ? W - 1 : 0;
  PreLayout L;
  L.buf_len = butter ? W + 2 * pad : (interp ? W : 0);
  L.fir_c = L.fir_gt = L.fir_b = 0;
  if (fir) {
    const int T = p.fir_taps, nf = W < T - 1 ? W : T - 1;          // the two-pass path only sees windows of n < T samples
    L.fir_gt = 8 * fir_ld_fwd(nf, T);
    L.fir_b = L.fir_gt + 10 * fir_ld_bwd(nf, T);
    int need = L.fir_b;                                              // taps / zi stay in global memory (fir_filtfilt)
    if (W >= T) {
      const int x8 = 8 * fir_merged_ld(W, T, 8), x10 = 10 * fir_merged_ld(W, T, 10);
      L.fir_c = ((x8 > x10 ? x8 : x10) + 1) & ~1;                    // even: c[] 16-byte aligned inside buf0
      const int k8 = fir_merged_k(T, 8), k10 = fir_merged_k(T, 10);
      const int m = L.fir_c + (k8 > k10 ? k8 : k10);
      if (m > need) need = m;
    }
    if (need > L.buf_len) L.buf_len = need;
  }
  // every section starts on a 16-byte boundary (the merged FIR fetches its taps with 128-bit loads), and so does the next
  // warp's slice
  int o = 0;
  auto sect = [&o](int bytes) { const int at = o; o += (bytes + 15) / 16 * 16; return at; };
  L.yv = sect(W * 8);
  L.xv = sect(interp ? W * 8 : 0);
  L.buf0 = sect(L.buf_len * 8);
  L.buf1 = sect(cubic ? W * 8 : 0);                    // knot slopes of the spline
  L.coef = sect(butter ? 128 * 8 : 0);                 // sos [16][6] | sosfilt_zi [16][2]
  L.posv = sect(W * 2);
  L.posb = sect(interp ? W * 2 : 0);
  L.total = o;
  return L;
}

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ double shfl_up_d(double v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }

// ---------------------------------------------------------------------------------------------
struct Warp {
  int lane;
  double *yv, *xv, *buf0, *buf1, *coef;
  unsigned short *posv, *posb;
  int n, m;            // valid (finite y) / block (finite x) counts
  double xfirst, xlast;
  bool grid;           // x[block] has been replaced by the uniform grid (after an INTERP_*)
  int fir_c, fir_gt, fir_b;   // FIR sub-plan inside buf0 (PreLayout)
  int W;               // window length of the launch (fixes the merged FIR's operand layout for every n <= W)
};

__device__ void diff1(Warp& w) {  // np.diff(y, n=1, prepend=y[0])  (signal_processor.py:203)
  for (int c = (w.n - 1) / 32; c >= 0; --c) {
    const int i = c * 32 + w.lane;
    double v = 0.0;
    if (i < w.n && i > 0) v = w.yv[i] - w.yv[i - 1];
    __syncwarp();
    if (i < w.n) w.yv[i] = v;
    __syncwarp();
  }
}

__device__ void diff2(Warp& w) {  // np.diff(y, n=2, prepend=y[:2])  (signal_processor.py:205)
  const double y0 = w.yv[0], y1 = w.yv[1];
  __syncwarp();
  for (int c = (w.n - 1) / 32; c >= 0; --c) {
    const int i = c * 32 + w.lane;
    double v = 0.0;
    if (i < w.n) {
      // z = [y0, y1, y0, y1, y2, ...];  out[i] = (z[i+2]-z[i+1]) - (z[i+1]-z[i])
      const double z2 = w.yv[i];
      const double z1 = i >= 1 ? w.yv[i - 1] : y1;
      const double z0 = i >= 2 ? w.yv[i - 2] : (i == 1 ? y1 : y0);
      v = (z2 - z1) - (z1 - z0);
    }
    __syncwarp();
    if (i < w.n) w.yv[i] = v;
    __syncwarp();
  }
}

__device__ void detrend_const(Warp& w) {  // scipy.signal.detrend(type='constant')
  double s = 0.0;
  for (int i = w.lane; i < w.n; i += 32) s += w.yv[i];
  const double mean = warp_sum(s) / (double)w.n;
  for (int i = w.lane; i < w.n; i += 32) w.yv[i] -= mean;
  __syncwarp();
}

__device__ void detrend_linear(Warp& w) {
  // scipy.signal.detrend(type='linear'): least squares of y on [i/N, 1], i = 1..N (sample index, not
  // time; scipy/signal/_signaltools.py:4307-4314), solved in centred closed form: with u_i = i/N,
  // du_i = u_i - mean(u), sum(du^2) = (N^2 - 1) / (12 N) exactly, slope = sum(du (y - ybar)) / sum(du^2).
  // Two reductions, no per-element division (u_i = i * (1/N)).
  const double N = (double)w.n, invN = 1.0 / N;
  double s = 0.0;
  for (int i = w.lane; i < w.n; i += 32) s += w.yv[i];
  const double ybar = warp_sum(s) * invN;
  const double ubar = (N + 1.0) * 0.5 * invN;
  double sxy = 0.0;
  for (int i = w.lane; i < w.n; i += 32) {
    const double du = fma((double)(i + 1), invN, -ubar);
    sxy = fma(du, w.yv[i] - ybar, sxy);
  }
  sxy = warp_sum(sxy);
  const double sxx = (N * N - 1.0) / (12.0 * N);
  const double slope = sxx > 0.0 ? sxy / sxx : 0.0;
  for (int i = w.lane; i < w.n; i += 32) {
    const double du = fma((double)(i + 1), invN, -ubar);
    w.yv[i] = (w.yv[i] - ybar) - slope * du;
  }
  __syncwarp();
}

// np.linspace(xfirst, xlast, m)[i] (numpy/_core/function_base.py): i*step + start, last = stop
__device__ __forceinline__ double grid_x(const Warp& w, int i, double step) {
  if (i == w.m - 1 && w.m > 1) return w.xlast;
  return __dadd_rn(__dmul_rn((double)i, step), w.xfirst);
}

// largest j in [0, n-1] with xs[j] <= x (caller guarantees xs[0] <= x)
__device__ __forceinline__ int bsearch_le(const double* xs, int n, double x) {
  int lo = 0, hi = n;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (xs[mid] <= x) lo = mid; else hi = mid;
  }
  return lo;
}

__device__ void finish_interp(Warp& w, double step) {
  // x[block], y[block] = grid, interpolated; valid = block  (signal_processor.py:209-210, 216-217)
  __syncwarp();
  for (int i = w.lane; i < w.m; i += 32) {
    w.yv[i] = w.buf0[i];
    w.xv[i] = grid_x(w, i, step);
    w.posv[i] = w.posb[i];
  }
  w.n = w.m;
  w.grid = true;
  __syncwarp();
}

__device__ void interp_linear(Warp& w) {  // np.interp(linspace(...), x[valid], y[valid])
  const double step = (w.xlast - w.xfirst) / (double)(w.m - 1);
  const int n = w.n;
  for (int i = w.lane; i < w.m; i += 32) {
    const double xi = grid_x(w, i, step);
    double r;
    if (xi > w.xv[n - 1]) r = w.yv[n - 1];
    else if (xi < w.xv[0]) r = w.yv[0];
    else {
      const int j = bsearch_le(w.xv, n, xi);
      if (j == n - 1 || w.xv[j] == xi) r = w.yv[j];
      else {
        const double slope = (w.yv[j + 1] - w.yv[j]) / (w.xv[j + 1] - w.xv[j]);
        r = __dadd_rn(__dmul_rn(slope, xi - w.xv[j]), w.yv[j]);
      }
    }
    w.buf0[i] = r;
  }
  finish_interp(w, step);
}

// scipy.interpolate.CubicSpline(x, y) (not-a-knot, extrapolate) evaluated on the grid
// (scipy/interpolate/_cubic.py:795-963; PPoly evaluation order of _ppoly.evaluate).
// Returns false if x is not strictly increasing (the reference raises ValueError).
__device__ bool interp_cubic(Warp& w) {
  const int n = w.n;
  const double* x = w.xv;
  const double* y = w.yv;
  int bad = 0;
  for (int i = w.lane; i + 1 < n; i += 32) bad |= !(x[i + 1] - x[i] > 0.0);
  if (__any_sync(0xffffffffu, bad)) return false;
  double* cp = w.buf0;   // Thomas scratch, later the evaluation output
  double* s = w.buf1;    // knot slopes
  if (w.lane == 0) {
    if (n == 2) {
      s[0] = s[1] = (y[1] - y[0]) / (x[1] - x[0]);
    } else if (n == 3) {
      const double dx0 = x[1] - x[0], dx1 = x[2] - x[1];
      const double sl0 = (y[1] - y[0]) / dx0, sl1 = (y[2] - y[1]) / dx1;
      const double s1 = (dx0 * sl1 + dx1 * sl0) / (dx0 + dx1);   // parabola through the 3 points
      s[1] = s1; s[0] = 2.0 * sl0 - s1; s[2] = 2.0 * sl1 - s1;
    }
  }
  if (n > 3) {
    // Rows 1..n-2 of the tridiagonal system are independent of each other: every lane builds its share in place —
    // cp[i] <- diagonal 2(dx[i-1]+dx[i]), s[i] <- right-hand side 3(dx[i] sl[i-1] + dx[i-1] sl[i]) — and only the
    // Thomas recurrence itself stays serial on lane 0, with one reciprocal per row on its critical path.
    for (int i = 1 + w.lane; i <= n - 2; i += 32) {
      const double dxp = x[i] - x[i - 1], dxc = x[i + 1] - x[i];
      const double slp = (y[i] - y[i - 1]) / dxp, slc = (y[i + 1] - y[i]) / dxc;
      cp[i] = 2.0 * (dxp + dxc);
      s[i] = 3.0 * (dxc * slp + dxp * slc);
    }
    __syncwarp();
    if (w.lane == 0) {
      double cprev, sprev;
      {  // row 0: dx1*s0 + (x2-x0)*s1 = ((dx0+2d)*dx1*sl0 + dx0^2*sl1)/d
        const double dx0 = x[1] - x[0], dx1 = x[2] - x[1];
        const double sl0 = (y[1] - y[0]) / dx0, sl1 = (y[2] - y[1]) / dx1;
        const double d = x[2] - x[0];
        const double rhs = ((dx0 + 2.0 * d) * dx1 * sl0 + dx0 * dx0 * sl1) / d;
        const double inv = 1.0 / dx1;
        cprev = d * inv; sprev = rhs * inv;
        cp[0] = cprev; s[0] = sprev;
      }
      double xm = x[0], xc = x[1], xn = x[2];                   // x[i-1], x[i], x[i+1]
#pragma unroll 4
      for (int i = 1; i <= n - 2; ++i) {
        // dx[i]*s[i-1] + 2(dx[i-1]+dx[i])*s[i] + dx[i-1]*s[i+1] = rhs[i]
        const double lo = xn - xc, up = xc - xm;
        const double inv = 1.0 / fma(-lo, cprev, cp[i]);
        cprev = up * inv;
        sprev = fma(-lo, sprev, s[i]) * inv;
        cp[i] = cprev; s[i] = sprev;
        xm = xc; xc = xn; xn = x[i + 2 < n ? i + 2 : n - 1];
      }
      {  // last row: (x[n-1]-x[n-3])*s[n-2] + dx[n-3]*s[n-1] = (dx[n-2]^2*sl[n-3] + (2d+dx[n-2])*dx[n-3]*sl[n-2])/d
        const double dxp = x[n - 2] - x[n - 3], dxc = x[n - 1] - x[n - 2];
        const double slp = (y[n - 2] - y[n - 3]) / dxp, slc = (y[n - 1] - y[n - 2]) / dxc;
        const double d = x[n - 1] - x[n - 3];
        const double rhs = (dxc * dxc * slp + (2.0 * d + dxc) * dxp * slc) / d;
        const double den = dxp - d * cprev;
        double sn = (rhs - d * sprev) / den;
        s[n - 1] = sn;
#pragma unroll 4
        for (int i = n - 2; i >= 0; --i) { sn = fma(-cp[i], sn, s[i]); s[i] = sn; }
      }
    }
  }
  __syncwarp();
  const double step = (w.xlast - w.xfirst) / (double)(w.m - 1);
  for (int i = w.lane; i < w.m; i += 32) {
    const double xi = grid_x(w, i, step);
    int j;
    if (xi < x[0]) j = 0;
    else if (xi >= x[n - 1]) j = n - 2;
    else j = bsearch_le(x, n, xi);
    const double dxj = x[j + 1] - x[j];
    const double slj = (y[j + 1] - y[j]) / dxj;
    const double t = (s[j] + s[j + 1] - 2.0 * slj) / dxj;
    const double c0 = t / dxj, c1 = (slj - s[j]) / dxj - t, c2 = s[j], c3 = y[j];
    const double u = xi - x[j];
    double res = c3, z = u;            // sum of c[k]*u^k in increasing powers, as _ppoly.evaluate_poly1
    res = __dadd_rn(res, __dmul_rn(c2, z)); z = __dmul_rn(z, u);
    res = __dadd_rn(res, __dmul_rn(c1, z)); z = __dmul_rn(z, u);
    res = __dadd_rn(res, __dmul_rn(c0, z));
    cp[i] = res;
  }
  finish_interp(w, step);
  return true;
}

// odd extension (scipy.signal._arraytools.odd_ext) of yv[0..n) by p into ext[0..n+2p)
__device__ void odd_ext(const Warp& w, double* ext, int p) {
  const int n = w.n, L = n + 2 * p;
  const double y0 = w.yv[0], yl = w.yv[n - 1];
  for (int i = w.lane; i < L; i += 32) {
    double v;
    if (i < p) v = 2.0 * y0 - w.yv[p - i];
    else if (i < p + n) v = w.yv[i - p];
    else v = 2.0 * yl - w.yv[n - 2 - (i - p - n)];
    ext[i] = v;
  }
  __syncwarp();
}

// scipy.signal.sosfiltfilt(sos, y, padlen) (scipy/signal/_signaltools.py:5091-5203): odd extension,
// sosfilt_zi steady state, forward + backward DF2T cascade (Cython _sosfilt), crop.
__device__ void sos_filtfilt(Warp& w, const double* __restrict__ sos_g, int N) {
  double* sos = w.coef;            // [N*6]
  double* zi = w.coef + 6 * MAX_SOS;  // [N*2]
  for (int i = w.lane; i < N * 6; i += 32) sos[i] = sos_g[i];
  __syncwarp();
  int nb0 = 0, na0 = 0;
  if (w.lane == 0) {
    // sosfilt_zi: zi[s] = scale * lfilter_zi(b, a); scale *= sum(b)/sum(a)   (:4520-4541)
    double scale = 1.0;
    for (int s = 0; s < N; ++s) {
      const double* c = sos + 6 * s;
      const double B0 = c[1] - c[4] * c[0], B1 = c[2] - c[5] * c[0];
      const double z0 = (B0 + B1) / (1.0 + c[4] + c[5]);
      zi[2 * s] = scale * z0;
      zi[2 * s + 1] = scale * (B1 - c[5] * z0);
      scale *= (c[0] + c[1] + c[2]) / (1.0 + c[4] + c[5]);
    }
  }
  for (int s = 0; s < N; ++s) { nb0 += sos[6 * s + 2] == 0.0; na0 += sos[6 * s + 5] == 0.0; }
  __syncwarp();
  // padlen as signal_processor.py:227-228
  const int dpl = 3 * (2 * N + 1 - (nb0 < na0 ? nb0 : na0));
  const int n = w.n, p = n <= dpl ? n - 1 : dpl;
  const int L = n + 2 * p;
  double* ext = w.buf0;
  odd_ext(w, ext, p);

  const int s = w.lane;
  const bool sec = s < N;
  const double b0 = sec ? sos[6 * s] : 0, b1 = sec ? sos[6 * s + 1] : 0, b2 = sec ? sos[6 * s + 2] : 0;
  const double a1 = sec ? sos[6 * s + 4] : 0, a2 = sec ? sos[6 * s + 5] : 0;
  const double zi0 = sec ? zi[2 * s] : 0, zi1 = sec ? zi[2 * s + 1] : 0;

  const double na1 = -a1, na2 = -a2;
  for (int pass = 0; pass < 2; ++pass) {
    // pass 0 runs over ext[0..L), pass 1 over the reversed forward output, both in place.
    // Sample i enters lane 0 at step i and leaves lane N-1 at step i + N - 1 (systolic cascade).
    const double x0 = pass == 0 ? ext[0] : ext[L - 1];
    double z0 = zi0 * x0, z1 = zi1 * x0;
    double prev_out = 0.0;
    const int dir = pass == 0 ? 1 : -1, base = pass == 0 ? 0 : L - 1;   // position of sample i: base + dir*i
    double nxt = ext[base];                                               // software-prefetched input of lane 0
    __syncwarp();
    const int t_steady = N - 1 < L ? N - 1 : L;
    int t = 0;
    // fill: lanes s <= t are live
    for (; t < t_steady; ++t) {
      const double from_prev = shfl_up_d(prev_out, 1);
      const double xc = s == 0 ? nxt : from_prev;
      if (s == 0 && t + 1 < L) nxt = ext[base + dir * (t + 1)];
      if (sec && t >= s) {
        const double xn = fma(b0, xc, z0);
        z0 = fma(b1, xc, fma(na1, xn, z1));
        z1 = fma(b2, xc, na2 * xn);
        prev_out = xn;
      }
    }
    // steady state: every section is live, no per-step liveness tests; lane N-1 emits sample t - (N-1)
    const double* in = ext + base + dir * (t + 1);
    double* out = ext + base + dir * (t - (N - 1));
    for (; t < L - 1; ++t) {
      const double from_prev = shfl_up_d(prev_out, 1);
      const double xc = s == 0 ? nxt : from_prev;
      if (s == 0) nxt = *in;
      in += dir;
      const double xn = fma(b0, xc, z0);
      z0 = fma(b1, xc, fma(na1, xn, z1));
      z1 = fma(b2, xc, na2 * xn);
      prev_out = xn;
      if (s == N - 1) *out = xn;
      out += dir;
    }
    // drain (and the last steady step, which has nothing left to prefetch): lanes with t - s < L are live
    for (; t < L + N - 1; ++t) {
      const double from_prev = shfl_up_d(prev_out, 1);
      const double xc = s == 0 ? nxt : from_prev;
      const int i = t - s;
      if (sec && i >= 0 && i < L) {
        const double xn = fma(b0, xc, z0);
        z0 = fma(b1, xc, fma(na1, xn, z1));
        z1 = fma(b2, xc, na2 * xn);
        prev_out = xn;
        if (s == N - 1) ext[base + dir * i] = xn;
      }
    }
    __syncwarp();
  }
  for (int i = w.lane; i < n; i += 32) w.yv[i] = ext[p + i];
  __syncwarp();
}

// sosfiltfilt for TWO signals per warp: the cascade has at most 16 sections, so the single-signal version above leaves
// half of every warp idle for its 2 x (L + N - 1) serial steps — the longest phase of every Butterworth configuration.
// Here lanes 0-15 run the cascade of signal A and lanes 16-31 that of signal B (their own coefficients: the two signals
// need not belong to the same window job), shuffles are 16 wide, and the arithmetic per lane is exactly that of
// sos_filtfilt, so the results are bit-identical.  The halves may differ in length; the loop without liveness tests runs
// while both are in steady state, the predicated loop finishes the longer one.  la / lb = false parks a half.
__device__ void sos_filtfilt_dual(Warp& wa, Warp& wb, bool la, bool lb, const double* __restrict__ ga,
                                  const double* __restrict__ gb, int N) {
  const int lane = wa.lane, hf = lane >> 4, s = lane & 15;
  const bool live = hf ? lb : la;
  double* yv = hf ? wb.yv : wa.yv;
  double* ext = hf ? wb.buf0 : wa.buf0;
  double* sos = hf ? wb.coef : wa.coef;      // [N*6]
  double* zi = sos + 6 * MAX_SOS;            // [N*2]
  const double* sg = hf ? gb : ga;
  const int n = live ? (hf ? wb.n : wa.n) : 0;
  if (live) for (int i = s; i < N * 6; i += 16) sos[i] = sg[i];
  __syncwarp();
  int nb0 = 0, na0 = 0;
  if (live) {
    if (s == 0) {
      // sosfilt_zi: zi[s] = scale * lfilter_zi(b, a); scale *= sum(b)/sum(a)   (:4520-4541)
      double scale = 1.0;
      for (int k = 0; k < N; ++k) {
        const double* c = sos + 6 * k;
        const double B0 = c[1] - c[4] * c[0], B1 = c[2] - c[5] * c[0];
        const double z0 = (B0 + B1) / (1.0 + c[4] + c[5]);
        zi[2 * k] = scale * z0;
        zi[2 * k + 1] = scale * (B1 - c[5] * z0);
        scale *= (c[0] + c[1] + c[2]) / (1.0 + c[4] + c[5]);
      }
    }
    for (int k = 0; k < N; ++k) { nb0 += sos[6 * k + 2] == 0.0; na0 += sos[6 * k + 5] == 0.0; }
  }
  __syncwarp();
  const int dpl = 3 * (2 * N + 1 - (nb0 < na0 ? nb0 : na0));      // padlen as signal_processor.py:227-228
  const int p = n <= dpl ? n - 1 : dpl;
  const int L = live ? n + 2 * p : 0;
  if (live) {
    const double y0 = yv[0], yl = yv[n - 1];
    for (int i = s; i < L; i += 16) {                             // odd extension
      double v;
      if (i < p) v = 2.0 * y0 - yv[p - i];
      else if (i < p + n) v = yv[i - p];
      else v = 2.0 * yl - yv[n - 2 - (i - p - n)];
      ext[i] = v;
    }
  }
  __syncwarp();
  const int La = __shfl_sync(0xffffffffu, L, 0), Lb = __shfl_sync(0xffffffffu, L, 16);
  const int Lmax = La > Lb ? La : Lb;
  const int Lfast = (La > 0 && Lb > 0) ? (La < Lb ? La : Lb) : Lmax;
  const bool sec = live && s < N;
  const double b0 = sec ? sos[6 * s] : 0, b1 = sec ? sos[6 * s + 1] : 0, b2 = sec ? sos[6 * s + 2] : 0;
  const double a1 = sec ? sos[6 * s + 4] : 0, a2 = sec ? sos[6 * s + 5] : 0;
  const double zi0 = sec ? zi[2 * s] : 0, zi1 = sec ? zi[2 * s + 1] : 0;
  const double na1 = -a1, na2 = -a2;
  const bool first = live && s == 0, last = live && s == N - 1;
  for (int pass = 0; pass < 2; ++pass) {
    const double x0 = L > 0 ? (pass == 0 ? ext[0] : ext[L - 1]) : 0.0;
    double z0 = zi0 * x0, z1 = zi1 * x0;
    double prev_out = 0.0;
    const int dir = pass == 0 ? 1 : -1, base = pass == 0 ? 0 : L - 1;   // position of sample i of this half: base + dir*i
    double nxt = L > 0 ? ext[base] : 0.0;
    __syncwarp();
    const int t_fill = N - 1 < Lmax ? N - 1 : Lmax;
    int t = 0;
    for (; t < t_fill; ++t) {                                     // fill: lanes s <= t are live
      const double from_prev = __shfl_up_sync(0xffffffffu, prev_out, 1, 16);
      const double xc = s == 0 ? nxt : from_prev;
      if (first && t + 1 < L) nxt = ext[base + dir * (t + 1)];
      if (sec && t >= s && t - s < L) {
        const double xn = fma(b0, xc, z0);
        z0 = fma(b1, xc, fma(na1, xn, z1));
        z1 = fma(b2, xc, na2 * xn);
        prev_out = xn;
        if (s == N - 1) ext[base + dir * (t - s)] = xn;           // only when N == 1
      }
    }
    if (Lfast > 0) {
      // steady state of BOTH halves: every section is live, lane N-1 of a half emits its sample t - (N-1)
      const double* in = ext + (L > 0 ? base + dir * (t + 1) : 0);
      double* out = ext + (L > 0 ? base + dir * (t - (N - 1)) : 0);
      for (; t < Lfast - 1; ++t) {
        const double from_prev = __shfl_up_sync(0xffffffffu, prev_out, 1, 16);
        const double xc = s == 0 ? nxt : from_prev;
        if (first) nxt = *in;
        in += dir;
        const double xn = fma(b0, xc, z0);
        z0 = fma(b1, xc, fma(na1, xn, z1));
        z1 = fma(b2, xc, na2 * xn);
        prev_out = xn;
        if (last) *out = xn;
        out += dir;
      }
    }
    for (; t < Lmax + N - 1; ++t) {                               // the longer half, and the drain of both
      const double from_prev = __shfl_up_sync(0xffffffffu, prev_out, 1, 16);
      const double xc = s == 0 ? nxt : from_prev;
      if (first && t + 1 < L) nxt = ext[base + dir * (t + 1)];
      const int i = t - s;
      if (sec && i >= 0 && i < L) {
        const double xn = fma(b0, xc, z0);
        z0 = fma(b1, xc, fma(na1, xn, z1));
        z1 = fma(b2, xc, na2 * xn);
        prev_out = xn;
        if (s == N - 1) ext[base + dir * i] = xn;
      }
    }
    __syncwarp();
  }
  if (live) for (int i = s; i < n; i += 16) yv[i] = ext[p + i];
  __syncwarp();
}

// scipy.signal.filtfilt(b, 1.0, y, padlen) for an FIR b (scipy/signal/_signaltools.py:4893-4924):
// odd extension, zi = lfilter_zi(b, [1]) (suffix sums of b[1:]), forward, backward, crop.
//   F[i] = sum_k b[k] ext[i-k] + (i < T-1 ? zi[i]*ext[0] : 0)          forward over the padded signal
//   B[i] = sum_k b[k] G[i-k]   + (i < T-1 ? zi[i]*F[L-1] : 0),  G[g] = F[L-1-g]   backward
//   out[m] = B[L-1-p-m]
// Only forward outputs that can reach the cropped result are evaluated (F[p .. p+n-1+T-1]).  Both passes
// are the register-tiled sliding dot product of corr_tile.cuh: each lane owns 8 consecutive outputs, the
// operand buffers are de-interleaved by 8 and zero padded in front so no tap needs a bounds check.
constexpr int FIR_RT = 8;     // forward pass: n + T - 1 outputs (426 for n = 300) = 2 rounds of 32 lanes x 8
constexpr int FIR_RTB = 10;   // backward pass: n outputs (300) = ONE round of 30 lanes x 10 instead of 32 + 6 lanes x 8
__device__ void fir_filtfilt(Warp& w, const double* __restrict__ taps_g, int T) {
  const int Kp = (T + FIR_RT - 1) / FIR_RT * FIR_RT;
  const int KpB = (T + FIR_RTB - 1) / FIR_RTB * FIR_RTB;
  // Taps and lfilter_zi are read where the design kernel left them (global memory, L1 / L2 resident): this two-pass form only
  // serves windows shorter than the filter (a stream's first T - 1 frames), and a zero-padded shared-memory copy of both cost
  // every warp of the launch 2 KB — the difference between 18 and 21 resident warps per SM for the steady-state windows.
  const double* __restrict__ b = taps_g;          // [T] (corr_tile supplies the zero padding up to Kp / KpB)
  const double* __restrict__ zi = taps_g + 128;   // [T-1]
  const int n = w.n, dpl = 3 * T, p = n <= dpl ? n - 1 : dpl;  // signal_processor.py:233-234
  const int L = n + 2 * p;
  const int fa = p, fb = (p + n - 1 + T - 1) < (L - 1) ? (p + n - 1 + T - 1) : (L - 1);   // forward outputs needed
  const int ba = p, bb = p + n - 1;                                                      // backward outputs needed
  // Only the operands those outputs can touch are staged: ext[fa-Kp .. fb+7] and G[ba-KpB .. bb+9]
  // (negative logical indices are the zero history of lfilter).  storage index = logical index - base.
  const int xbase = fa - Kp, gbase = ba - KpB;
  int LD = (Kp + n + T + 15) / FIR_RT + 1;
  LD += (6 - (LD & 3)) & 3;   // LD = 2 (mod 4): the 8 rows of XT start 4 banks apart, the extension below stores without conflicts
  const int LDB = (KpB + n + T + 2 * FIR_RTB) / FIR_RTB + 1;
  double* XT = w.buf0;              // ext, de-interleaved by FIR_RT
  double* GT = w.buf0 + w.fir_gt;   // reversed forward output G[g] = F[L-1-g], de-interleaved by FIR_RTB
  const double y_first = w.yv[0], y_last = w.yv[n - 1];
  // odd extension (scipy.signal._arraytools.odd_ext), branch free so that the unrolled iterations overlap their loads:
  // head 2*y[0] - y[p-i], body y[i-p], tail 2*y[n-1] - y[2n-2+p-i], zero outside [0, L)
#pragma unroll 3
  for (int jj = w.lane; jj < FIR_RT * LD; jj += 32) {
    const int i = jj + xbase;
    const bool inside = i >= 0 && i < L, head = i < p, tail = i >= p + n;
    const int src = head ? p - i : (tail ? 2 * n - 2 + p - i : i - p);
    const double y = w.yv[inside ? src : 0];
    const double v = head ? 2.0 * y_first - y : (tail ? 2.0 * y_last - y : y);
    XT[xt_index<FIR_RT>(jj, LD)] = inside ? v : 0.0;
  }
#pragma unroll 4
  for (int jj = w.lane; jj < FIR_RTB * LDB; jj += 32) GT[jj] = 0.0;
  __syncwarp();
  const double x0 = p >= 1 ? 2.0 * y_first - w.yv[p] : y_first;       // ext[0]
  for (int I = Kp; I <= fb - xbase; I += 32 * FIR_RT) {               // storage Kp <-> logical fa
    const int j0 = I + FIR_RT * w.lane, i0 = j0 + xbase;
    if (i0 <= fb) {
      double acc[FIR_RT];
#pragma unroll
      for (int r = 0; r < FIR_RT; ++r) acc[r] = 0.0;
      corr_tile<FIR_RT, double, 0, 0, true>(acc, b, Kp, XT, LD, j0, 0, 0x7fffffff, T);
#pragma unroll
      for (int r = 0; r < FIR_RT; ++r) {
        const int i = i0 + r;
        if (i <= fb) {
          const double v = acc[r] + (i < T - 1 ? zi[i] * x0 : 0.0);
          const int g = L - 1 - i;                                    // >= ba - (T-1) >= gbase
          GT[xt_index<FIR_RTB>(g - gbase, LDB)] = v;
        }
      }
    }
  }
  __syncwarp();
  // F[L-1] = G[0]; only used when p < T-1 (then fb == L-1, so it has been computed)
  const double yend = (0 - gbase >= 0) ? GT[xt_index<FIR_RTB>(0 - gbase, LDB)] : 0.0;
  for (int I = KpB; I <= bb - gbase; I += 32 * FIR_RTB) {
    const int j0 = I + FIR_RTB * w.lane, i0 = j0 + gbase;
    if (i0 <= bb) {
      double acc[FIR_RTB];
#pragma unroll
      for (int r = 0; r < FIR_RTB; ++r) acc[r] = 0.0;
      corr_tile<FIR_RTB, double, 0, 0, true>(acc, b, KpB, GT, LDB, j0, 0, 0x7fffffff, T);
#pragma unroll
      for (int r = 0; r < FIR_RTB; ++r) {
        const int i = i0 + r;
        if (i <= bb) w.yv[L - 1 - p - i] = acc[r] + (i < T - 1 ? zi[i] * yend : 0.0);
      }
    }
  }
  __syncwarp();
}

// filtfilt with both passes merged: wherever the padding is at least T-1 samples (n >= T), neither pass's initial
// condition reaches the cropped output and forward . backward collapses into ONE symmetric FIR of 2T-1 taps,
//   out[m] = sum_{d=-(T-1)}^{T-1} ac[|d|] ext[p + m + d],        ac[d] = sum_i b[i] b[i+d]   (from the design kernel)
// (F[f] = sum_k b[k] ext[f-k] for f >= p >= T-1 has no zi term and no zero history; B[i] for i in [p, p+n-1] likewise.)
// 253 x n multiply-adds instead of 127 x (2n + 126), one staged operand buffer instead of two, no intermediate signal;
// agrees with the two-pass form to rounding (1e-15 relative).  RT consecutive outputs per lane (corr_tile.cuh): RT = 10
// makes a 300-sample window ONE round of 30 lanes, RT = 8 a 250-sample window one round of 32.
// LDC / KC: the operand buffer's leading dimension and the padded tap count as compile-time constants for the common
// (taps, window) pairs (corr_tile.cuh); the leading dimension is the launch's (window length W), not the signal's.
// The merged taps — ready-made by the design kernel, c[k] = ac[|k - M|], zero padded — are copied into the warp's
// shared-memory slice first.  (Tiles reading them from global memory, 2 KB less shared memory per warp, were measured
// slower: 323 against 306 us per 32 768 signals, profiles/r4a — the ring gather streams through L1 and pushes the taps
// out, so the tile loop opens its blocks with L2 round trips.)
template <int RT, int LDC = 0, int KC = 0>
__device__ void fir_merged(Warp& w, const double* __restrict__ c_g, int T) {
  const int M = T - 1;
  const int K = KC ? KC : fir_merged_k(T, RT);
  const int n = w.n, dpl = 3 * T, p = n <= dpl ? n - 1 : dpl;      // signal_processor.py:233-234
  const int L = n + 2 * p;
  const int tiles = (n + RT - 1) / RT;
  const int LD = LDC ? LDC : fir_merged_ld(w.W, T, RT);
  double* XT = w.buf0;              // X[j] = ext[j + xbase], de-interleaved by RT; output m sits at j = m + K
  double* c = w.buf0 + w.fir_c;     // c[k] = ac[|k - M|], k = 0 .. 2M; zero up to FIR_MERGED_LEN >= K
  for (int k = w.lane; k < K; k += 32) c[k] = c_g[k];
  const int xbase = p + M - K;
  const double y_first = w.yv[0], y_last = w.yv[n - 1];
  // odd extension (scipy.signal._arraytools.odd_ext): head 2*y[0] - y[p-i], body y[i-p], tail 2*y[n-1] - y[2n-2+p-i];
  // indices outside [0, L) only meet the zero taps k > 2M
  // storage index jj = i - xbase, written segment by segment (zeros | head | body | tail | zeros): one select-free loop per
  // segment instead of five selects per element (the single loop was 9 % of the kernel's instructions)
  const int total = RT * (K / RT + tiles);
  const int j_h = xbase < 0 ? -xbase : 0;                         // first element of the extension (i = 0)
  const int j_b = p - xbase, j_t = p + n - xbase;                  // body / tail start
  const int j_e = L - xbase < total ? L - xbase : total;           // end of the extension inside the buffer
  for (int jj = w.lane; jj < j_h; jj += 32) XT[xt_index<RT>(jj, LD)] = 0.0;
  for (int jj = j_h + w.lane; jj < j_b; jj += 32) XT[xt_index<RT>(jj, LD)] = 2.0 * y_first - w.yv[j_b - jj];           // p - i
  for (int jj = j_b + w.lane; jj < j_t && jj < total; jj += 32) XT[xt_index<RT>(jj, LD)] = w.yv[jj - j_b];           // i - p
  for (int jj = j_t + w.lane; jj < j_e; jj += 32) XT[xt_index<RT>(jj, LD)] = 2.0 * y_last - w.yv[2 * n - 2 - (jj - j_b)];   // 2n-2+p-i
  for (int jj = (j_e > j_t ? j_e : j_t) + w.lane; jj < total; jj += 32) XT[xt_index<RT>(jj, LD)] = 0.0;
  __syncwarp();
  for (int t = w.lane; t < tiles; t += 32) {
    double acc[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) acc[r] = 0.0;
    // (fetching the staged taps two at a time — corr_tile's C2, LDS.128 — was measured: tile block 125 -> 120 instructions,
    // kernel 306.2 -> 309.5 us per 32 768 signals, profiles/r4d; not used)
    corr_tile<RT, double, LDC, KC>(acc, c, K, XT, LD, K + RT * t);
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      const int m = RT * t + r;
      if (m < n) w.yv[m] = acc[r];          // yv is not an operand of the tiles: no hazard with the other lanes
    }
  }
  __syncwarp();
}

__device__ __forceinline__ void fir_apply(Warp& w, const double* __restrict__ tg, int T) {
  const int n = w.n;
  if (n >= T) {
    // the cheaper tiling for this window length: rounds x RT x padded taps
    const int c8 = ((n + 7) / 8 + 31) / 32 * 8 * fir_merged_k(T, 8);
    const int c10 = ((n + 9) / 10 + 31) / 32 * 10 * fir_merged_k(T, 10);
    const bool t127 = T == 127;                       // the reference's default filter (fir_taps = 127): K = 260 / 256
    if (c10 < c8) {
      if (t127 && w.W == 300) fir_merged<10, 57, 260>(w, tg + 256, T);       // fir_merged_ld(300, 127, 10)
      else fir_merged<10, 0, 0>(w, tg + 256, T);
    } else {
      if (t127 && w.W == 300) fir_merged<8, 71, 256>(w, tg + 256, T);        // fir_merged_ld(300, 127, 8)
      else if (t127 && w.W == 250) fir_merged<8, 65, 256>(w, tg + 256, T);   // fir_merged_ld(250, 127, 8)
      else fir_merged<8, 0, 0>(w, tg + 256, T);
    }
  } else {
    fir_filtfilt(w, tg, T);
  }
}

// ---------------------------------------------------------------------------------------------
// FEAT = which of the heavy stages this instantiation contains (register budget and code size follow the method list):
// bit 0 INTERP_*, bit 1 FILTER_BUTTER, bit 2 FILTER_FIR.  diff / detrend are always present.
constexpr int F_INTERP = 1, F_BUTTER = 2, F_FIR = 4;

// isfinite(fs) for fs = 1 / ((x_last - x_first) / (m - 1)), the guard of signal_processor.py:200 (Signal.get_fs,
// signal_data.py:55-58), m >= 2.  For every spacing a clock can produce the quotient is far from the overflow / underflow
// thresholds and the answer is known without the two float64 divisions (~9 % of the kernel's stall samples sat on them);
// otherwise the reference's expression is evaluated as written.
__device__ __forceinline__ bool fs_is_finite(double xfirst, double xlast, int m) {
  const double d = fabs(xlast - xfirst);
  if (d > 1.0e-290 && d < 1.0e290) return true;          // |d / (m - 1)| in (1e-295, 1e290): 1 / that is finite
  return isfinite(1.0 / ((xlast - xfirst) / (double)(m - 1)));
}

// Stage one signal's window: ring -> shared memory with ballot / popc compaction of the valid samples (Signal.reset_mask:
// v = isfinite(x), w = isfinite(y); signal_data.py:43-45), writing the position-preserving pass-through copy on the way.
// Returns ST_OK, or ST_GUARD when the reference's guard (signal_processor.py:200) leaves the window unprocessed.
// JMAP: the job's ring row and newest sample come from the job map (filters.cuh JobMap).
template <int FEAT, bool JMAP>
__device__ int gather_window(Warp& w, unsigned char* sm, const PreLayout& L, const bpv_window_params& p,
                             const double* __restrict__ ring_t, const double* __restrict__ ring_y, long long sig,
                             double* __restrict__ ox, double* __restrict__ oy, const JobMap& jm) {
  // xv / posb exist in the shared-memory plan only when the method list resamples (an instantiation may serve a subset
  // of its stages)
  bool has_interp = false;
  if (FEAT & F_INTERP)
    for (int i = 0; i < p.num_methods; ++i) has_interp |= (p.methods[i] == BPV_INTERP_LINEAR || p.methods[i] == BPV_INTERP_CUBIC);
  w.yv = reinterpret_cast<double*>(sm + L.yv);
  w.xv = reinterpret_cast<double*>(sm + L.xv);
  w.buf0 = reinterpret_cast<double*>(sm + L.buf0);
  w.buf1 = reinterpret_cast<double*>(sm + L.buf1);
  w.coef = reinterpret_cast<double*>(sm + L.coef);
  w.posv = reinterpret_cast<unsigned short*>(sm + L.posv);
  w.posb = reinterpret_cast<unsigned short*>(sm + L.posb);
  w.grid = false;
  w.W = p.window;
  w.fir_c = L.fir_c; w.fir_gt = L.fir_gt; w.fir_b = L.fir_b;
  const long long job = sig / p.R;
  const int r = (int)(sig % p.R);
  const int s = JMAP ? jm.stream[job] : (int)(job / p.jobs_per_stream), j = JMAP ? 0 : (int)(job % p.jobs_per_stream);
  const long long head = JMAP ? (long long)jm.head[job] : p.head0 + (long long)j * p.head_step;
  const double* rt = ring_t + (long long)s * p.cap;
  const double* ry = ring_y + ((long long)s * p.R + r) * p.cap;
  const int W = p.window;
  int n = 0, m = 0;
  double xfirst = 0.0, xlast = 0.0;
  const unsigned lt = (1u << w.lane) - 1u;
  const long long gfirst = head - W + 1;                      // global index of window position 0
  const int kmin = gfirst < 0 ? (int)(-gfirst < W ? -gfirst : W) : 0;   // positions before the stream started: NaN
  const int slot0 = (int)(((gfirst % p.cap) + p.cap) % p.cap);       // ring slot of position 0 (one 64-bit modulo)
  // stage the window (independent, coalesced loads: no ballot in this loop, so they all overlap); y is staged in yv[]
  // and compacted in place below
  double* xstage = L.buf_len >= W ? w.buf0 : nullptr;
  bool allf = true;
  for (int k = w.lane; k < W; k += 32) {
    double x = nan_f64(), y = nan_f64();
    if (k >= kmin) { int slot = slot0 + k; if (slot >= p.cap) slot -= p.cap; x = rt[slot]; y = ry[slot]; }
    ox[k] = x; oy[k] = y;
    w.yv[k] = y;
    if (xstage) xstage[k] = x;
    allf &= isfinite(x) && isfinite(y);
  }
  __syncwarp();
  // A window without holes (steady state of a stream whose detections never drop) is its own compaction: every position is
  // valid, in place.  One vote replaces the ten ballot / popc / shuffle rounds below and the identity position table.
  if (xstage && !has_interp && __all_sync(0xffffffffu, allf)) {
    for (int k = w.lane; k < W; k += 32) w.posv[k] = (unsigned short)k;
    w.n = w.m = W;
    w.xfirst = xstage[0]; w.xlast = xstage[W - 1];
    __syncwarp();
    return (W >= 2 && fs_is_finite(w.xfirst, w.xlast, W)) ? ST_OK : ST_GUARD;
  }
  for (int k0 = 0; k0 < W; k0 += 32) {
    const int k = k0 + w.lane;
    double x = nan_f64(), y = nan_f64();
    if (k < W) {
      y = w.yv[k];
      if (xstage) x = xstage[k];
      else if (k >= kmin) { int slot = slot0 + k; if (slot >= p.cap) slot -= p.cap; x = rt[slot]; }
    }
    const bool fx = isfinite(x), fy = isfinite(y);
    const unsigned bx = __ballot_sync(0xffffffffu, fx), by = __ballot_sync(0xffffffffu, fy);
    __syncwarp();
    if (fy) {
      const int idx = n + __popc(by & lt);
      w.yv[idx] = y; w.posv[idx] = (unsigned short)k;
      if (has_interp) w.xv[idx] = x;
    }
    if (fx && has_interp) w.posb[m + __popc(bx & lt)] = (unsigned short)k;
    if (bx) {
      if (m == 0) xfirst = shfl_d(x, __ffs(bx) - 1);
      xlast = shfl_d(x, 31 - __clz(bx));
    }
    __syncwarp();
    n += __popc(by); m += __popc(bx);
  }
  __syncwarp();
  w.n = n; w.m = m; w.xfirst = xfirst; w.xlast = xlast;
  return (n >= 2 && m >= 2 && fs_is_finite(xfirst, xlast, m)) ? ST_OK : ST_GUARD;
}

// One processing method that works on a single signal (everything but the two-signal Butterworth cascade).
template <int FEAT>
__device__ int apply_method(Warp& w, int method, const bpv_window_params& p, const DesignRef& dr, long long job) {
  switch (method) {
    case BPV_DIFF_1: diff1(w); break;
    case BPV_DIFF_2: diff2(w); break;
    case BPV_INTERP_LINEAR: if (FEAT & F_INTERP) interp_linear(w); break;
    case BPV_INTERP_CUBIC: if (FEAT & F_INTERP) { if (!interp_cubic(w)) return ST_CUBIC_X; } break;
    case BPV_DETREND_CONST: detrend_const(w); break;
    case BPV_DETREND_LINEAR: detrend_linear(w); break;
    case BPV_FILTER_BUTTER:
      if (FEAT & F_BUTTER) {
        const double* sg = dr.sos(job);
        if (!isfinite(sg[0])) return ST_BAD_BANDS;
        sos_filtfilt(w, sg, p.butter_order);
      }
      break;
    case BPV_FILTER_FIR:
      if (FEAT & F_FIR) {
        const double* tg = dr.fir(job);
        if (!isfinite(tg[0])) return ST_BAD_BANDS;
        fir_apply(w, tg, p.fir_taps);
      }
      break;
    default: break;
  }
  return ST_OK;
}

// scatter back into the position-preserving window (y[valid] = ..., signal_processor.py:202-236)
__device__ void scatter_window(const Warp& w, int st, int W, double* __restrict__ ox, double* __restrict__ oy,
                               int32_t* __restrict__ status, long long sig) {
  if (st == ST_OK) {
    for (int i = w.lane; i < w.n; i += 32) {
      const int k = w.posv[i];
      oy[k] = w.yv[i];
      if (w.grid) ox[k] = w.xv[i];
    }
  } else if (st != ST_GUARD) {
    for (int k = w.lane; k < W; k += 32) oy[k] = nan_f64();
  }
  if (w.lane == 0) status[sig] = st;
}

__device__ __forceinline__ void prefetch_filters(int FEAT, int lane, const bpv_window_params& p, const DesignRef& dr, long long job) {
  // the job's filter coefficients are first needed after the gather and the detrend: start pulling them (taps | zi |
  // merged taps: 33 lines, resp. 768 B of sos) towards the SM now, so that the filter stage does not open with a
  // DRAM round trip
  for (int i = 0; i < p.num_methods; ++i) {
    if ((FEAT & F_FIR) && p.methods[i] == BPV_FILTER_FIR) {
      asm volatile("prefetch.global.L1 [%0];" ::"l"(dr.fir(job) + lane * 16));
      if (lane == 0) asm volatile("prefetch.global.L1 [%0];" ::"l"(dr.fir(job) + 512));
    }
    if ((FEAT & F_BUTTER) && p.methods[i] == BPV_FILTER_BUTTER && lane * 16 < p.butter_order * 6)
      asm volatile("prefetch.global.L1 [%0];" ::"l"(dr.sos(job) + lane * 16));
  }
}

// DUAL = false: one warp per signal.  DUAL = true (every instantiation with FILTER_BUTTER): one warp per PAIR of
// consecutive signals — the single-signal stages run for one and then the other, the Butterworth cascade for both at once
// (sos_filtfilt_dual); the warp's shared-memory slice holds two per-signal plans.
template <int FEAT, int MINB, bool DUAL, bool JMAP>
__global__ void __launch_bounds__(128, MINB) window_preprocess_kernel(const double* __restrict__ ring_t,
                                                                      const double* __restrict__ ring_y,
                                                                      const bpv_window_params p, const PreLayout L,
                                                                      const DesignRef dr,
                                                                      double* __restrict__ proc_x, double* __restrict__ proc_y,
                                                                      int32_t* __restrict__ status, const JobMap jm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const long long unit = (long long)blockIdx.x * wpb + wib;
  const long long nsig = (long long)p.S * p.jobs_per_stream * p.R;
  const int W = p.window;
  const int lane = threadIdx.x & 31;
  if (!DUAL) {
    const long long sig = unit;                                    // job * R + r
    if (sig >= nsig) return;
    Warp w;
    w.lane = lane;
    const long long job = sig / p.R;
    prefetch_filters(FEAT, lane, p, dr, job);
    double* ox = proc_x + sig * W;
    double* oy = proc_y + sig * W;
    int st = gather_window<FEAT, JMAP>(w, smem_raw + (size_t)wib * L.total, L, p, ring_t, ring_y, sig, ox, oy, jm);
    for (int mi = 0; mi < p.num_methods && st == ST_OK; ++mi) st = apply_method<FEAT>(w, p.methods[mi], p, dr, job);
    scatter_window(w, st, W, ox, oy, status, sig);
  } else {
    const long long sa = 2 * unit, sb = sa + 1;
    if (sa >= nsig) return;
    const bool hasb = sb < nsig;
    Warp wa, wb;
    wa.lane = wb.lane = lane;
    const long long ja = sa / p.R, jb = (hasb ? sb : sa) / p.R;
    prefetch_filters(FEAT, lane, p, dr, ja);
    if (jb != ja) prefetch_filters(FEAT, lane, p, dr, jb);
    unsigned char* sm = smem_raw + (size_t)wib * 2 * L.total;
    double* oxa = proc_x + sa * W; double* oya = proc_y + sa * W;
    double* oxb = proc_x + (hasb ? sb : sa) * W; double* oyb = proc_y + (hasb ? sb : sa) * W;
    int sta = gather_window<FEAT, JMAP>(wa, sm, L, p, ring_t, ring_y, sa, oxa, oya, jm);
    int stb = ST_GUARD;
    if (hasb) stb = gather_window<FEAT, JMAP>(wb, sm + L.total, L, p, ring_t, ring_y, sb, oxb, oyb, jm);
    else { wb = wa; }
    for (int mi = 0; mi < p.num_methods && (sta == ST_OK || stb == ST_OK); ++mi) {
      const int m = p.methods[mi];
      if (m == BPV_FILTER_BUTTER) {
        const double* ga = dr.sos(ja);
        const double* gb = dr.sos(jb);
        if (sta == ST_OK && !isfinite(ga[0])) sta = ST_BAD_BANDS;
        if (stb == ST_OK && !isfinite(gb[0])) stb = ST_BAD_BANDS;
        if (sta == ST_OK || stb == ST_OK) sos_filtfilt_dual(wa, wb, sta == ST_OK, stb == ST_OK, ga, gb, p.butter_order);
      } else {
        if (sta == ST_OK) sta = apply_method<FEAT & ~F_BUTTER>(wa, m, p, dr, ja);
        if (stb == ST_OK) stb = apply_method<FEAT & ~F_BUTTER>(wb, m, p, dr, jb);
      }
    }
    scatter_window(wa, sta, W, oxa, oya, status, sa);
    if (hasb) scatter_window(wb, stb, W, oxb, oyb, status, sb);
  }
}

template <int FEAT, int MINB, bool DUAL>
static int launch_preprocess(const double* ring_t, const double* ring_y, const bpv_window_params& p, const PreLayout& L,
                             const DesignRef& dr, double* proc_x, double* proc_y, int32_t* status, cudaStream_t st,
                             const JobMap* jm) {
  const int max_smem = 200 * 1024;
  const int per_warp = (DUAL ? 2 : 1) * L.total;                 // a warp holds one signal, or a pair of them
  BPV_REQUIRE(per_warp <= max_smem, BPV_E_TOO_LARGE, "bpv_window_preprocess: window %d needs %d B of shared memory per signal",
              p.window, L.total);
  // warps per CTA: the value in 1..4 (__launch_bounds__(128)) that keeps the most warps resident per SM
  // what the register budget of this instantiation allows: 4 MINB warps by the launch bound; one-warp CTAs of a 96-register
  // instantiation fit 21 (65536 / (96 * 32)), of an 80-register one 25
  const int reg_warps = MINB >= 6 ? 25 : (MINB == 5 ? 21 : 4 * MINB);   // 80 / 96 registers
  int wpb = 1, best = 0;
  for (int c = 1; c <= 4; ++c) {
    const int per_block = c * per_warp + 1024;                   // + per-CTA reservation
    if (per_block > max_smem) break;
    int blocks = (227 * 1024) / per_block;
    if (blocks > 32) blocks = 32;
    int warps = blocks * c;
    if (warps > reg_warps) warps = reg_warps;
    if (warps > best || (warps == best && c < wpb)) { best = warps; wpb = c; }
  }
  const size_t smem = (size_t)wpb * per_warp;
  auto kern = jm ? window_preprocess_kernel<FEAT, MINB, DUAL, true> : window_preprocess_kernel<FEAT, MINB, DUAL, false>;
  if (int rc = ensure_dyn_smem((const void*)kern, smem)) return rc;
  const long long nsig = (long long)p.S * p.jobs_per_stream * p.R;
  const long long units = DUAL ? (nsig + 1) / 2 : nsig;
  kern<<<(unsigned)((units + wpb - 1) / wpb), wpb * 32, smem, st>>>(ring_t, ring_y, p, L, dr, proc_x, proc_y, status,
                                                                    jm ? *jm : JobMap{});
  return check_launch("bpv_window_preprocess");
}

static int parse_methods(const bpv_window_params* p, const char* who, bool& butter, bool& fir, bool& interp) {
  butter = fir = interp = false;
  BPV_REQUIRE(p->num_methods >= 0 && p->num_methods <= BPV_MAX_METHODS, BPV_E_INVALID, "%s: bad sizes", who);
  for (int i = 0; i < p->num_methods; ++i) {
    const int m = p->methods[i];
    BPV_REQUIRE(m >= BPV_DIFF_1 && m <= BPV_FILTER_FIR, BPV_E_UNSUPPORTED,
                "%s: unknown processing method %d (NotImplementedError, signal_processor.py:238)", who, m);
    butter |= m == BPV_FILTER_BUTTER;
    fir |= m == BPV_FILTER_FIR;
    interp |= m == BPV_INTERP_LINEAR || m == BPV_INTERP_CUBIC;
  }
  return 0;
}

}  // namespace bpv

// workspace of a launch: sos [J][16*6] | fir [J][FIR_WS_STRIDE] | ref int32 [J] (padded to 8 B) | miss list [J] x 16 B
namespace bpv {
struct WsPlan { long long sos, fir, ref, miss, total; };
static WsPlan ws_plan(const bpv_window_params* p) {
  const long long J = (long long)p->S * p->jobs_per_stream;
  WsPlan w;
  w.sos = 0;
  w.fir = w.sos + J * MAX_SOS * 6 * 8;
  w.ref = w.fir + J * FIR_WS_STRIDE * 8;
  w.miss = w.ref + (J * 4 + 7) / 8 * 8;
  w.total = w.miss + J * 16;
  return w;
}
}  // namespace bpv

extern "C" int64_t bpv_window_workspace_bytes(const bpv_window_params* p) {
  if (!p) return -1;
  return bpv::ws_plan(p).total;
}

extern "C" int64_t bpv_design_cache_bytes(void) { return bpv::DC_BYTES; }

namespace bpv {
static int window_design(const double* ring_t, const bpv_window_params* p, void* workspace, int64_t workspace_bytes,
                         void* cache, int64_t cache_bytes, void* stream, const JobMap* jm) {
  if (int rc = check_filter_params(p, "bpv_window_design")) return rc;
  BPV_REQUIRE(ring_t, BPV_E_INVALID, "bpv_window_design: NULL pointer");
  BPV_REQUIRE(p->S > 0 && p->window > 0 && p->window <= p->cap && p->jobs_per_stream > 0, BPV_E_INVALID, "bpv_window_design: bad sizes");
  bool butter, fir, interp;
  if (int rc = parse_methods(p, "bpv_window_design", butter, fir, interp)) return rc;
  if (!butter && !fir) return 0;
  const WsPlan wp = ws_plan(p);
  BPV_REQUIRE(workspace && workspace_bytes >= wp.total, BPV_E_INVALID,
              "bpv_window_design: workspace too small (see bpv_window_workspace_bytes)");
  BPV_REQUIRE(!cache || cache_bytes >= DC_BYTES, BPV_E_INVALID, "bpv_window_design: design cache too small (see bpv_design_cache_bytes)");
  unsigned char* ws = (unsigned char*)workspace;
  double* sos_ws = (double*)(ws + wp.sos);
  double* taps_ws = (double*)(ws + wp.fir);
  cudaStream_t st = (cudaStream_t)stream;
  if (cache)
    return launch_design_cached(ring_t, *p, butter, fir, (unsigned char*)cache, (int32_t*)(ws + wp.ref), ws + wp.miss, sos_ws, taps_ws, st, jm);
  if (butter) if (int rc = launch_job_butter(ring_t, *p, sos_ws, st, jm)) return rc;
  if (fir) if (int rc = launch_job_firls(ring_t, *p, taps_ws, st, jm)) return rc;
  return 0;
}

static int window_filter(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                         const void* workspace, int64_t workspace_bytes, const void* cache, int64_t cache_bytes,
                         double* proc_x, double* proc_y, int32_t* status, void* stream, const JobMap* jm) {
  if (int rc = check_filter_params(p, "bpv_window_preprocess")) return rc;
  BPV_REQUIRE(ring_t && ring_y && proc_x && proc_y && status, BPV_E_INVALID, "bpv_window_preprocess: NULL pointer");
  BPV_REQUIRE(p->S > 0 && p->R > 0 && p->window > 0 && p->window <= p->cap && p->jobs_per_stream > 0, BPV_E_INVALID,
              "bpv_window_preprocess: bad sizes");
  BPV_REQUIRE(p->window <= 65535, BPV_E_TOO_LARGE, "bpv_window_preprocess: window > 65535");
  bool butter, fir, interp;
  if (int rc = parse_methods(p, "bpv_window_preprocess", butter, fir, interp)) return rc;
  const WsPlan wp = ws_plan(p);
  if (butter || fir) {
    BPV_REQUIRE(workspace && workspace_bytes >= wp.total, BPV_E_INVALID,
                "bpv_window_preprocess: workspace too small (see bpv_window_workspace_bytes)");
    BPV_REQUIRE(!cache || cache_bytes >= DC_BYTES, BPV_E_INVALID, "bpv_window_preprocess: design cache too small (see bpv_design_cache_bytes)");
  }
  const unsigned char* ws = (const unsigned char*)workspace;
  DesignRef dr;
  dr.sos_ws = ws ? (const double*)(ws + wp.sos) : nullptr;
  dr.taps_ws = ws ? (const double*)(ws + wp.fir) : nullptr;
  dr.ref = (ws && cache && (butter || fir)) ? (const int32_t*)(ws + wp.ref) : nullptr;
  dr.cache = (const unsigned char*)cache;
  const bool fir_only = !interp && !butter && fir;
  const PreLayout L = pre_layout(*p);
  cudaStream_t st = (cudaStream_t)stream;
#define BPV_PRE(feat, minb, dual) return launch_preprocess<feat, minb, dual>(ring_t, ring_y, *p, L, dr, proc_x, proc_y, status, st, jm)
  // Two signals per warp pay off while enough warps stay resident to hide the stages that run for one signal after the
  // other (the spline's serial Thomas sweep above all): with the 46 KB per signal of a 1200-sample cubic + Butterworth
  // window only two such warps fit an SM and the pair is slower than two single-signal warps (measured on config 4:
  // 3.57 ms against 2.86 ms per step), so large plans keep one signal per warp.  BPV_SOS_SINGLE = test switch.
  const bool single_sos = getenv("BPV_SOS_SINGLE") != nullptr || (227 * 1024) / (2 * L.total + 1024) < 8;
  if (!interp && !butter && !fir) BPV_PRE(0, 6, false);
  if (fir_only) BPV_PRE(F_FIR, 5, false);
  if (single_sos) {
    if (!interp && !fir) BPV_PRE(F_BUTTER, 4, false);
    BPV_PRE(F_INTERP | F_BUTTER | F_FIR, 4, false);
  }
  if (!interp && !fir) BPV_PRE(F_BUTTER, 4, true);
  if (!fir) BPV_PRE(F_INTERP | F_BUTTER, 4, true);
  BPV_PRE(F_INTERP | F_BUTTER | F_FIR, 4, true);
#undef BPV_PRE
}

// The params of a job-map launch: the window kernels see the job list as S = num_jobs streams of one job each (their
// per-job layouts, workspace plan and grid are then those of the lockstep path over J jobs); the map supplies each job's
// ring row and newest sample.  Validates what the lockstep checks cannot see.
static int jobs_params(const bpv_window_params* p, const int32_t* job_stream, const int64_t* job_head, int64_t num_jobs,
                       const char* who, bpv_window_params& q) {
  BPV_REQUIRE(p, BPV_E_INVALID, "%s: NULL params", who);
  BPV_REQUIRE(job_stream && job_head, BPV_E_INVALID, "%s: NULL job map", who);
  BPV_REQUIRE(p->S > 0 && num_jobs > 0 && num_jobs <= INT32_MAX / 32, BPV_E_INVALID, "%s: bad sizes", who);
  q = *p;
  q.S = (int32_t)num_jobs;
  q.jobs_per_stream = 1;
  q.head0 = 0;
  q.head_step = 0;
  return 0;
}
}  // namespace bpv

extern "C" int bpv_window_design(const double* ring_t, const bpv_window_params* p, void* workspace, int64_t workspace_bytes,
                                 void* cache, int64_t cache_bytes, void* stream) {
  return bpv::window_design(ring_t, p, workspace, workspace_bytes, cache, cache_bytes, stream, nullptr);
}

extern "C" int bpv_window_filter(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                                 const void* workspace, int64_t workspace_bytes, const void* cache, int64_t cache_bytes,
                                 double* proc_x, double* proc_y, int32_t* status, void* stream) {
  return bpv::window_filter(ring_t, ring_y, p, workspace, workspace_bytes, cache, cache_bytes, proc_x, proc_y, status, stream,
                            nullptr);
}

extern "C" int bpv_window_design_jobs(const double* ring_t, const bpv_window_params* p, void* workspace, int64_t workspace_bytes,
                                      void* cache, int64_t cache_bytes, const int32_t* job_stream, const int64_t* job_head,
                                      int64_t num_jobs, void* stream) {
  using namespace bpv;
  if (num_jobs == 0 && p) return 0;
  bpv_window_params q;
  if (int rc = jobs_params(p, job_stream, job_head, num_jobs, "bpv_window_design_jobs", q)) return rc;
  const JobMap jm{job_stream, job_head};
  return window_design(ring_t, &q, workspace, workspace_bytes, cache, cache_bytes, stream, &jm);
}

extern "C" int bpv_window_filter_jobs(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                                      const void* workspace, int64_t workspace_bytes, const void* cache, int64_t cache_bytes,
                                      double* proc_x, double* proc_y, int32_t* status, const int32_t* job_stream,
                                      const int64_t* job_head, int64_t num_jobs, void* stream) {
  using namespace bpv;
  if (num_jobs == 0 && p) return 0;
  bpv_window_params q;
  if (int rc = jobs_params(p, job_stream, job_head, num_jobs, "bpv_window_filter_jobs", q)) return rc;
  const JobMap jm{job_stream, job_head};
  return window_filter(ring_t, ring_y, &q, workspace, workspace_bytes, cache, cache_bytes, proc_x, proc_y, status, stream, &jm);
}

extern "C" int bpv_window_preprocess_jobs(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                                          void* workspace, int64_t workspace_bytes, double* proc_x, double* proc_y,
                                          int32_t* status, const int32_t* job_stream, const int64_t* job_head, int64_t num_jobs,
                                          void* stream) {
  if (int rc = bpv_window_design_jobs(ring_t, p, workspace, workspace_bytes, nullptr, 0, job_stream, job_head, num_jobs, stream))
    return rc;
  return bpv_window_filter_jobs(ring_t, ring_y, p, workspace, workspace_bytes, nullptr, 0, proc_x, proc_y, status, job_stream,
                                job_head, num_jobs, stream);
}

extern "C" int bpv_window_preprocess(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                                     void* workspace, int64_t workspace_bytes,
                                     double* proc_x, double* proc_y, int32_t* status, void* stream) {
  if (int rc = bpv_window_design(ring_t, p, workspace, workspace_bytes, nullptr, 0, stream)) return rc;
  return bpv_window_filter(ring_t, ring_y, p, workspace, workspace_bytes, nullptr, 0, proc_x, proc_y, status, stream);
}
