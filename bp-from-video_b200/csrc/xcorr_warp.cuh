// Pairwise-ROI cross-correlation, warp-per-pair kernel body (moved out of xcorr.cu so that a second translation unit can
// instantiate it).
#pragma once
#include "filters.cuh"
#include "corr_tile.cuh"

namespace bpv {

constexpr float XC_DELTA = 2.0e-4f;   // candidate band below the fp32 maximum (normalised correlation, |c| <~ 1)

// ---------------------------------------------------------------------------------------------
// Warp-per-pair version (default): the CTA-per-pair kernel above spends most of its time in __syncthreads between short
// phases (staging, single-warp compaction, five block reductions, peak search: the tile phase is 18 % of its samples).
// Here one warp owns a (job, pair): every phase is warp-local (ballot compaction, shuffle reductions), each lane owns the
// XW_RT = 10 lag pairs (li, li + n) of one tile, so a 300-sample window (599 lags) is a single round of the register-tiled
// circular sliding dot product (2 LDS + 2 predicated moves per 10 FFMA, n taps per lane), and the float64 re-evaluation of
// the candidate lags is a warp-cooperative dot product.
// smem per warp: doubles a64[W] | b64[W]; u16 pos[W]; floats cv[2W] (only when a lane owns more than one tile, W > 320) | c[K] | XT[RT * LD]
// ---------------------------------------------------------------------------------------------
constexpr int XW_RT = 10;
struct XwLayout { int b64, pos, cv, c, xt, total, K, LD, one_round; };
__host__ __device__ inline XwLayout xw_layout(int W) {
  XwLayout L;
  L.K = (W + XW_RT - 1) / XW_RT * XW_RT;                 // taps, padded to the tile
  L.LD = (2 * (L.K / XW_RT) + 2) | 1;                    // columns of the de-interleaved periodic operand (odd: no bank conflicts)
  int o = W * 8;
  L.b64 = o; o += W * 8;
  L.pos = o; o += (W * 2 + 15) / 16 * 16;
  L.one_round = L.K / XW_RT <= 32;                       // every lane owns at most one tile: coarse values stay in registers
  L.cv = o; o += L.one_round ? 0 : 2 * W * 4;
  L.c = o; o += L.K * 4;
  L.xt = o; o += XW_RT * L.LD * 4;
  L.total = (o + 15) / 16 * 16;
  return L;
}

// COARSE pass layout (corr_tile.cuh, corr_tile_wrap):  corr[li] = sum_m c[m] a[li - m]  (c[m] = b[n-1-m], 0 <= li - m < n).
// Lags li and li + n use complementary tap ranges, so a lane owns the lag PAIRS li = RT*tile - 1 + r, r = 0..RT-1 and sweeps the
// K taps once over the periodic extension AA[t] = a[t mod n], t in [-n, n), stored at X[t + K + RT + 1]: n multiply-adds per
// output pair for every lane (a 300-sample window: 30 lanes x 10 pairs, one round), where one tile of consecutive lags per
// lane made the warp wait for the centre lanes' n taps per lag.
// LDC = the operand buffer's leading dimension when it is one of the specialised window sizes (0 = run-time value)
// ONE = every lane owns at most one tile (windows up to 320 samples): the 2 x RT coarse values of a lane never leave its
// registers — the candidate lags are flagged from them as a 20-bit mask per lane — so the plan has no cv[] array (9.1 instead of
// 11.5 KB per warp at W = 300) and the peak search does not re-read 2n - 1 values from shared memory.  Launch bound 5 CTAs per SM:
// 88 registers keep the packed tile loop free of spills (ptxas settles on 72 without it and pays 60 register moves per 10 taps).
// The kernel's body as a device function of (CTA index, shared memory): xcorr_warp_kernel (xcorr.cu) is a CTA of up to four
// such warps; welch_xcorr_kernel (welch_xcorr.cu) interleaves CTAs of this role with Welch CTAs in one grid.
// BAND: the peak is searched over the lags whose lag in seconds (the float64 value reported as lag_sec) lies in [band.lo, band.hi],
// evaluated lag by lag (the timestamps need not be monotone); the coarse maximum and the finite count are taken over those lags
// alone, so that an out-of-band maximum cannot set a threshold that excludes every in-band lag.
template <int LDC, bool ONE, bool BAND = false>
__device__ __forceinline__ void xcorr_warp_body(unsigned blk, unsigned char* __restrict__ xsm, const double* __restrict__ proc_x,
                                                const double* __restrict__ proc_y, const bpv_window_params& p, const XwLayout& Lw,
                                                long long npairs, float* __restrict__ corr_lag, float* __restrict__ corr_val,
                                                int32_t* __restrict__ num_lags, int32_t* __restrict__ lag_idx,
                                                double* __restrict__ lag_sec, double* __restrict__ lag_corr,
                                                const PeakBand band = PeakBand{}) {
  constexpr int RT = XW_RT;
  const int W = p.window, R = p.R, P = R * (R - 1) / 2, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long jp = (long long)blk * (blockDim.x >> 5) + wid;          // job * P + pair
  if (jp >= npairs) return;
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
  unsigned char* sm = xsm + (size_t)wid * Lw.total;
  double* a64 = reinterpret_cast<double*>(sm);
  double* b64 = reinterpret_cast<double*>(sm + Lw.b64);
  unsigned short* pos = reinterpret_cast<unsigned short*>(sm + Lw.pos);
  float* cv = reinterpret_cast<float*>(sm + Lw.cv);
  float* c = reinterpret_cast<float*>(sm + Lw.c);
  float* XT = reinterpret_cast<float*>(sm + Lw.xt);
  const int LD = LDC ? LDC : Lw.LD;
  // stage both windows (independent coalesced loads)
  bool allf = true;
  for (int k = lane; k < W; k += 32) {
    const double va = ya_g[k], vb = yb_g[k];
    a64[k] = va; b64[k] = vb; pos[k] = (unsigned short)k;
    allf &= isfinite(va) && isfinite(vb);
  }
  __syncwarp();
  // jointly valid samples (valid = a.w & b.w), compacted in place; a pair of windows without holes already is (one vote
  // instead of W / 32 ballot rounds, positions = identity)
  int n = 0;
  if (__all_sync(0xffffffffu, allf)) {
    n = W;
  } else {
    const unsigned lt = (1u << lane) - 1u;
    for (int k0 = 0; k0 < W; k0 += 32) {
      const int k = k0 + lane;
      double va = nan_f64(), vb = nan_f64();
      if (k < W) { va = a64[k]; vb = b64[k]; }
      const bool ok = isfinite(va) && isfinite(vb);
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      __syncwarp();
      if (ok) { const int i = n + __popc(bal & lt); a64[i] = va; b64[i] = vb; pos[i] = (unsigned short)k; }
      __syncwarp();
      n += __popc(bal);
    }
  }
  if (n < 2) {                                  // guard signal_processor.py:284 -> empty
    if (lane == 0) { num_lags[jp] = 0; lag_idx[jp] = -1; lag_sec[jp] = nan_f64(); lag_corr[jp] = nan_f64(); }
    return;
  }
  const int K = (n + RT - 1) / RT * RT;         // <= Lw.K
  const int OFF = K + RT + 1;                   // storage index of AA[0]
  double daa = 0, dbb = 0, dab = 0, amax = 0, bmax = 0;
  for (int i = lane; i < n; i += 32) {
    const double va = a64[i], vb = b64[i];
    daa = fma(va, va, daa); dbb = fma(vb, vb, dbb); dab = fma(va, vb, dab);
    amax = fmax(amax, fabs(va)); bmax = fmax(bmax, fabs(vb));
  }
  daa = warp_sum(daa); dbb = warp_sum(dbb); dab = warp_sum(dab);
  for (int o = 16; o > 0; o >>= 1) { amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o)); bmax = fmax(bmax, __shfl_xor_sync(0xffffffffu, bmax, o)); }
  const double den = fmax(fmax(daa, dbb), dab);
  // fp32 operands scaled to O(1) so tiny band-passed signals neither underflow nor lose bits.  The operand buffer is
  // written completely (every storage index a tile can touch): periodic extension inside [-n, n), zeros outside.
  const double sa = amax > 0 ? 1.0 / amax : 1.0, sb = bmax > 0 ? 1.0 / bmax : 1.0;
  const int jtot = 2 * K + 2 * RT;              // storage indices [0, jtot): t = j - OFF in [-K - RT - 1, K + RT - 2]
  // each sample is converted once and stored at its two periods (t = i and t = i - n); the few slots outside [-n, n) are zeroed
  for (int i = lane; i < n; i += 32) {
    const float v = (float)(a64[i] * sa);
    XT[xt_index<RT>(i + OFF, LD)] = v;
    XT[xt_index<RT>(i + OFF - n, LD)] = v;
  }
  for (int j = lane; j < OFF - n; j += 32) XT[xt_index<RT>(j, LD)] = 0.f;
  for (int j = OFF + n + lane; j < jtot; j += 32) XT[xt_index<RT>(j, LD)] = 0.f;
  for (int m = lane; m < K; m += 32) c[m] = m < n ? (float)(b64[n - 1 - m] * sb) : 0.f;
  __syncwarp();
  const float unscale = (float)(1.0 / (sa * sb * den));
  const int L = 2 * n - 1;
  const long long ob = jp * (2LL * W - 1);
  const double x_last = xa_g[pos[n - 1]];
  auto in_band = [&](int li) {                  // BAND: lag index li -> is its lag in seconds inside the band
    const int k = li - (n - 1), ak = k < 0 ? -k : k;
    return band.in((x_last - xa_g[pos[n - 1 - ak]]) * (k > 0 ? 1.0 : (k < 0 ? -1.0 : 0.0)));
  };
  float cmax = -INFINITY; int cnt = 0;          // coarse maximum / finite count, gathered while the tiles are written
  int nin = 0;                                  // BAND, cv[] path: lags inside the band (ONE: the bits of okm)
  const int tiles = K / RT;
  unsigned okm = 0;                             // ONE: bit r = first lag of pair r is a lag of this window (BAND: in band), bit RT + r = second lag
  float acc[RT], first[RT];                     // ONE: after the tile, the lane's scaled coarse values (second | first lags)
  for (int tile = lane; tile < tiles; tile += 32) {
#pragma unroll
    for (int r = 0; r < RT; ++r) { acc[r] = 0.f; first[r] = 0.f; }
    corr_tile_wrap_f32x2<RT, LDC>(acc, first, c, K, XT, LD, RT * tile + K + RT, tile);
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      const int la = RT * tile - 1 + r;          // first lag of the pair; the second is la + n
      first[r] *= unscale; acc[r] *= unscale;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int li = h ? la + n : la;
        const bool ok = h ? (la <= n - 2) : (la >= 0 && la <= n - 2);
        if (ok) {
          const float cc = h ? acc[r] : first[r];
          bool inb = true;
          if (BAND) inb = in_band(li);
          if (ONE) { if (inb) okm |= 1u << (h * RT + r); } else { cv[li] = cc; if (BAND && inb) ++nin; }
          if (isfinite(cc) && inb) { ++cnt; cmax = fmaxf(cmax, cc); }
          if (corr_val) {
            const int k = li - (n - 1), ak = k < 0 ? -k : k;
            const double lag = (x_last - xa_g[pos[n - 1 - ak]]) * (k > 0 ? 1.0 : (k < 0 ? -1.0 : 0.0));
            corr_lag[ob + li] = (float)lag;
            corr_val[ob + li] = cc;
          }
        }
      }
    }
    if (ONE) break;                             // tiles <= 32: one tile per lane
  }
  __syncwarp();
  // PEAK in float64: every lag whose coarse value is within XC_DELTA of the coarse maximum is re-evaluated as a
  // float64 dot product (warp cooperative); the first maximum among those decides (Signal.get_peak after the range reset).
  for (int o = 16; o > 0; o >>= 1) { cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o)); cnt += __shfl_xor_sync(0xffffffffu, cnt, o); }
  double bv = -INFINITY; int bi = 0x7fffffff;
  const float thr = cmax - XC_DELTA;
  auto refine = [&](int lc) {                    // whole warp: lag index lc -> float64 correlation, first-max update
    const int k = lc - (n - 1);
    const int l0 = k < 0 ? -k : 0, l1 = k > 0 ? n - k : n;
    double acc = 0.0;
    for (int l = l0 + lane; l < l1; l += 32) acc = fma(a64[l + k], b64[l], acc);
    acc = warp_sum(acc);
    const double cc = acc / den;
    if (isfinite(cc) && (cc > bv || (cc == bv && lc < bi))) { bv = cc; bi = lc; }
  };
  if (ONE) {
    unsigned cand = 0;
#pragma unroll
    for (int b = 0; b < 2 * RT; ++b) {
      const float v = b < RT ? first[b] : acc[b - RT];
      if (((okm >> b) & 1u) && (cnt >= 2 ? (isfinite(v) && v >= thr) : true)) cand |= 1u << b;
    }
    unsigned m = __ballot_sync(0xffffffffu, cand != 0);
    while (m) {                                  // any order: the update keeps the largest value, ties to the smallest lag
      const int src = __ffs(m) - 1;
      m &= m - 1;
      unsigned f = __shfl_sync(0xffffffffu, cand, src);
      while (f) {
        const int b = __ffs(f) - 1;
        f &= f - 1;
        const int la = RT * src - 1 + (b < RT ? b : b - RT);
        refine(b < RT ? la : la + n);
      }
    }
  } else {
    for (int li0 = 0; li0 < L; li0 += 128) {       // 4 consecutive lags per lane per step
      const int lb = li0 + 4 * lane;
      unsigned flags = 0;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int li = lb + e;
        if (li < L) {
          const float v = cv[li];
          if ((cnt >= 2 ? (isfinite(v) && v >= thr) : true) && (!BAND || in_band(li))) flags |= 1u << e;
        }
      }
      unsigned m = __ballot_sync(0xffffffffu, flags != 0);
      while (m) {                                  // lanes in increasing lag order, lags of a lane in increasing order
        const int src = __ffs(m) - 1;
        m &= m - 1;
        unsigned f = __shfl_sync(0xffffffffu, flags, src);
        while (f) {
          const int lc = li0 + 4 * src + __ffs(f) - 1;
          f &= f - 1;
          refine(lc);
        }
      }
    }
  }
  // eligible lags (BAND: inside the band) in float64 terms: den == 0 or non-finite makes every lag non-finite (NaN / inf),
  // any other den every lag finite
  int neligible = L;
  if (BAND) neligible = warp_sum(ONE ? __popc(okm) : nin);
  if (lane == 0) {
    const bool any = isfinite(den) && den != 0.0 && bi != 0x7fffffff;
    num_lags[jp] = L;
    if (any && neligible >= 2) {
      const int k = bi - (n - 1), ak = k < 0 ? -k : k;
      lag_idx[jp] = bi;
      lag_sec[jp] = (x_last - xa_g[pos[n - 1 - ak]]) * (k > 0 ? 1.0 : (k < 0 ? -1.0 : 0.0));
      lag_corr[jp] = bv;
    } else { lag_idx[jp] = -1; lag_sec[jp] = nan_f64(); lag_corr[jp] = nan_f64(); }
  }
}

}  // namespace bpv
