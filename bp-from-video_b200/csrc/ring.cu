// Device ring buffers of raw samples (sg_raw): the batched twin of Signal.add_sample /
// SignalGroup.add_samples (signal_data.py:31-35, 94-98).  deque(maxlen) semantics are a ring
// addressed by the global sample index; the NaN prefill (signal_data.py:18-19) is the caller's
// initial fill plus the "negative global index reads NaN" rule of the window kernels.
#include "common.cuh"

namespace bpv {
// RAGGED (bpv_ring_push_ragged): stream s appends its first n[s] rows at global indices g0s[s] ...; the other rows of its T are
// not read.  The ragged parameters follow the lockstep ones, so the lockstep instantiation keeps its parameter layout.
template <bool RAGGED>
__global__ void ring_push_kernel(double* __restrict__ ring_t, double* __restrict__ ring_y, int S, int R, int cap,
                                 long long g0, int T, const double* __restrict__ ts, const double* __restrict__ values,
                                 const int64_t* __restrict__ g0s, const int32_t* __restrict__ n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over S*T*(R+1)
  const long long total = (long long)S * T * (R + 1);
  if (i >= total) return;
  const int c = (int)(i % (R + 1));
  const long long st = i / (R + 1);
  const int t = (int)(st % T);
  const long long s = st / T;
  if (RAGGED && t >= n[s]) return;
  const int slot = (int)(((RAGGED ? g0s[s] : g0) + t) % cap);
  if (c == R) { if (ts) ring_t[s * cap + slot] = ts[s * T + t]; }
  else if (values) ring_y[(s * R + c) * cap + slot] = values[(s * T + t) * R + c];
}
}  // namespace bpv

extern "C" int bpv_ring_push(double* ring_t, double* ring_y, int32_t S, int32_t R, int32_t cap,
                             int64_t g0, int32_t T, const double* ts, const double* values, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(ring_t && ring_y && (ts || values), BPV_E_INVALID, "bpv_ring_push: NULL pointer");
  BPV_REQUIRE(S > 0 && R > 0 && cap > 0 && T > 0 && T <= cap && g0 >= 0, BPV_E_INVALID, "bpv_ring_push: bad sizes");
  const long long total = (long long)S * T * (R + 1);
  ring_push_kernel<false><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ring_t, ring_y, S, R, cap, g0, T, ts, values,
                                                                                            nullptr, nullptr);
  return check_launch("bpv_ring_push");
}

namespace bpv {
// Job map of a ragged step: CTA b owns streams [1024 b, 1024 b + 1024), one per thread.  Every CTA sums the job counts of
// ALL streams (coalesced, L2-resident after the first CTA: 256 KB at S = 65 536) to get its chunk's first job and the total,
// so one launch needs no inter-CTA scratch; a warp-shuffle block scan places the chunk's streams.  The map entries are then
// written job-parallel (thread per job, coalesced stores; the job's stream by a binary search over the chunk's offsets in
// shared memory): a stream's up to T entries written by one thread would make every store of a warp touch 32 lines.
// STRIDED (bpv_stream_jobs_strided): stream s evaluates its window after its m-th sample exactly when (m + phase) % stride
// == 0, so of a step's n frames from count c it takes q = (c + n + phase) / stride - (c + phase) / stride jobs, job i with its
// newest sample at ((c + phase) / stride + 1 + i) * stride - phase - 1.  The !STRIDED instantiation is bpv_stream_jobs's.
constexpr int STREAM_JOBS_THREADS = 1024;
__device__ __forceinline__ long long block_sum_ll(long long v, long long* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  v = lane < (int)(blockDim.x >> 5) ? red[lane] : 0;
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// A stream's cadence: a stride below 1 reads as 1, a phase as its remainder modulo the stride (in [0, stride)); NULL arrays
// read as stride 1 / phase 0.  Whatever the entries hold, a stream then takes between 0 and n of its step's jobs.
__device__ __forceinline__ void stream_cadence(const int32_t* __restrict__ stride, const int32_t* __restrict__ phase, int s,
                                               long long& k, long long& ph) {
  k = stride ? max(stride[s], 1) : 1;
  ph = phase ? ((long long)phase[s] % k + k) % k : 0;
}
__device__ __forceinline__ int strided_jobs(const int64_t* __restrict__ g0, const int32_t* __restrict__ stride,
                                            const int32_t* __restrict__ phase, int s, int n) {
  long long k, ph;
  stream_cadence(stride, phase, s, k, ph);
  const long long c = g0[s] + ph;                            // 64-bit: counts grow without bound on long-running streams
  return (int)((c + n) / k - c / k);
}
template <bool STRIDED>
__global__ void __launch_bounds__(STREAM_JOBS_THREADS) stream_jobs_kernel(int S, const int64_t* __restrict__ g0,
                                                                          const int32_t* __restrict__ n, int last_only,
                                                                          long long num_jobs, int32_t* __restrict__ job_stream,
                                                                          int64_t* __restrict__ job_head,
                                                                          int32_t* __restrict__ stream_job0,
                                                                          int64_t* __restrict__ g0_next,
                                                                          const int32_t* __restrict__ stride,
                                                                          const int32_t* __restrict__ phase) {
  __shared__ long long red[32];
  __shared__ int first[STREAM_JOBS_THREADS];                  // first job of each of the chunk's streams, chunk-relative
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int s0 = blockIdx.x * STREAM_JOBS_THREADS;
  long long all = 0, before = 0;
  for (int s = tid; s < S; s += STREAM_JOBS_THREADS) {
    const int k = max(n[s], 0);
    const int jk = STRIDED ? strided_jobs(g0, stride, phase, s, k) : last_only ? (k > 0) : k;
    all += jk;
    if (s < s0) before += jk;
  }
  all = block_sum_ll(all, red);
  before = block_sum_ll(before, red);
  const int s = s0 + tid;
  const int k = s < S ? max(n[s], 0) : 0;
  const int jk = STRIDED ? (s < S ? strided_jobs(g0, stride, phase, s, k) : 0) : last_only ? (k > 0) : k;
  long long inc = jk;                                          // inclusive scan of the chunk's job counts
  for (int o = 1; o < 32; o <<= 1) {
    const long long v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  __syncthreads();
  if (lane == 31) red[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    long long w = red[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const long long v = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += v;
    }
    red[lane] = w;                                             // inclusive over the warps
  }
  __syncthreads();
  const int rel = (int)((wid ? red[wid - 1] : 0) + inc - jk);
  const int chunk_jobs = (int)red[31];
  first[tid] = rel;
  const bool ok = all == num_jobs;
  if (s < S) {
    stream_job0[s] = (int32_t)(before + rel);
    if (ok) g0_next[s] = g0[s] + k;
  }
  if (blockIdx.x == gridDim.x - 1 && tid == 0) stream_job0[S] = (int32_t)all;
  __syncthreads();
  if (!ok) return;
  const int nst = min(STREAM_JOBS_THREADS, S - s0);
  for (int q = tid; q < chunk_jobs; q += STREAM_JOBS_THREADS) {
    int lo = 0, hi = nst - 1;                                  // the last stream whose first job is <= q owns job q
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (first[mid] <= q) lo = mid; else hi = mid - 1;
    }
    const int ss = s0 + lo;
    const long long base = g0[ss];
    job_stream[before + q] = ss;
    if (STRIDED) {
      long long k, ph;
      stream_cadence(stride, phase, ss, k, ph);
      job_head[before + q] = ((base + ph) / k + 1 + (q - first[lo])) * k - ph - 1;
    } else {
      job_head[before + q] = last_only ? base + max(n[ss], 0) - 1 : base + (q - first[lo]);
    }
  }
}
}  // namespace bpv

extern "C" int bpv_ring_push_ragged(double* ring_t, double* ring_y, int32_t S, int32_t R, int32_t cap, const int64_t* g0,
                                    const int32_t* n, int32_t T, const double* ts, const double* values, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(ring_t && ring_y && g0 && n && (ts || values), BPV_E_INVALID, "bpv_ring_push_ragged: NULL pointer");
  BPV_REQUIRE(S > 0 && R > 0 && cap > 0 && T > 0 && T <= cap, BPV_E_INVALID, "bpv_ring_push_ragged: bad sizes");
  const long long total = (long long)S * T * (R + 1);
  ring_push_kernel<true><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ring_t, ring_y, S, R, cap, 0, T, ts, values,
                                                                                           g0, n);
  return check_launch("bpv_ring_push_ragged");
}

namespace bpv {
static int stream_jobs(const char* who, int32_t S, const int64_t* g0, const int32_t* n, int32_t last_only, const int32_t* stride,
                       const int32_t* phase, int64_t num_jobs, int32_t* job_stream, int64_t* job_head, int32_t* stream_job0,
                       int64_t* g0_next, void* stream) {
  BPV_REQUIRE(g0 && n && stream_job0 && g0_next && (num_jobs == 0 || (job_stream && job_head)), BPV_E_INVALID,
              "%s: NULL pointer", who);
  BPV_REQUIRE(S > 0 && S <= 65536 && num_jobs >= 0 && num_jobs <= INT32_MAX, BPV_E_INVALID,
              "%s: bad sizes (1 <= S <= 65536, 0 <= num_jobs < 2^31)", who);
  const unsigned grid = (unsigned)((S + STREAM_JOBS_THREADS - 1) / STREAM_JOBS_THREADS);
  if (stride || phase)
    stream_jobs_kernel<true><<<grid, STREAM_JOBS_THREADS, 0, (cudaStream_t)stream>>>(S, g0, n, 0, num_jobs, job_stream, job_head,
                                                                                     stream_job0, g0_next, stride, phase);
  else
    stream_jobs_kernel<false><<<grid, STREAM_JOBS_THREADS, 0, (cudaStream_t)stream>>>(S, g0, n, last_only != 0, num_jobs, job_stream,
                                                                                      job_head, stream_job0, g0_next, nullptr, nullptr);
  return check_launch(who);
}
}  // namespace bpv

extern "C" int bpv_stream_jobs(int32_t S, const int64_t* g0, const int32_t* n, int32_t last_only, int64_t num_jobs,
                               int32_t* job_stream, int64_t* job_head, int32_t* stream_job0, int64_t* g0_next, void* stream) {
  return bpv::stream_jobs("bpv_stream_jobs", S, g0, n, last_only, nullptr, nullptr, num_jobs, job_stream, job_head, stream_job0,
                          g0_next, stream);
}

extern "C" int bpv_stream_jobs_strided(int32_t S, const int64_t* g0, const int32_t* n, const int32_t* stride, const int32_t* phase,
                                       int64_t num_jobs, int32_t* job_stream, int64_t* job_head, int32_t* stream_job0,
                                       int64_t* g0_next, void* stream) {
  return bpv::stream_jobs("bpv_stream_jobs_strided", S, g0, n, 0, stride, phase, num_jobs, job_stream, job_head, stream_job0,
                          g0_next, stream);
}

// ---------------------------------------------------------------------------------------------
// Running means of the per-frame results — SURVEY.md §8(f) row 3: sg_bpm / sg_ptt (deque(maxlen =
// peak_max_samples), signal_processor.py:49, 83-84, 310, 312) and what the drawer shows,
// sg_bpm.get_means(as_int=True) (drawer.py:134-135; Signal.get_mean, signal_data.py:60-63).
// One thread per (stream, column) pushes the T new values of the step in order and emits, after each
// push, nanmean over the history with numpy's summation order (pairwise_sum for a contiguous 1-D array:
// 8 interleaved accumulators for n >= 8, numpy/_core/src/umath/loops_utils.h.src) and its half-to-even round.
namespace bpv {
__device__ inline double np_sum_small(const double* a, int n) {   // numpy pairwise sum, n <= 128
  if (n < 8) {
    double r = 0.0;          // numpy starts from -0.0; identical for every finite input except an all -0.0 array
    for (int i = 0; i < n; ++i) r += a[i];
    return r;
  }
  double r[8];
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] += a[i + j];
  double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) res += a[i];
  return res;
}

constexpr int MAX_MEAN_HIST = 128;

// Push v into the history rg [H] at slot `newest` and write the nanmean over the history, oldest slot first (deque order;
// NaN -> 0 as np.nanmean does), and its rounded value to element e of mean / mean_int.
__device__ __forceinline__ void push_nanmean(double* __restrict__ rg, int H, int newest, double v, long long e,
                                             double* __restrict__ mean, double* __restrict__ mean_int) {
  double tmp[MAX_MEAN_HIST];
  rg[newest] = v;
  int cnt = 0;
  for (int h = 0; h < H; ++h) {
    int slot = newest + 1 + h; if (slot >= H) slot -= H;
    const double x = rg[slot];
    const bool ok = isfinite(x);
    tmp[h] = ok ? x : 0.0;
    cnt += ok;
  }
  double m = nan_f64();
  if (cnt) m = np_sum_small(tmp, H) / (double)cnt;
  if (mean) mean[e] = m;
  if (mean_int) mean_int[e] = cnt ? rint(m) : nan_f64();
}

__global__ void running_mean_kernel(double* __restrict__ ring, int S, int C, int H, long long g0, int T,
                                    const double* __restrict__ values, double scale,
                                    double* __restrict__ mean, double* __restrict__ mean_int) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;     // s * C + c
  if (idx >= S * C) return;
  const int s = idx / C, c = idx % C;
  double* rg = ring + (long long)idx * H;
  for (int t = 0; t < T; ++t) {
    const long long e = ((long long)s * T + t) * C + c;
    const double v = values[e] * scale;                        // f * 60 / t * 1000 (signal_processor.py:310, 312)
    push_nanmean(rg, H, (int)((g0 + t) % H), v, e, mean, mean_int);
  }
}
}  // namespace bpv

extern "C" int bpv_running_mean(double* ring, int32_t S, int32_t C, int32_t H, int64_t g0, int32_t T,
                                const double* values, double scale, double* mean, double* mean_int, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(ring && values && (mean || mean_int), BPV_E_INVALID, "bpv_running_mean: NULL pointer");
  BPV_REQUIRE(S > 0 && C > 0 && H > 0 && H <= MAX_MEAN_HIST && T > 0 && g0 >= 0, BPV_E_INVALID, "bpv_running_mean: bad sizes (history <= 128)");
  const int n = S * C;
  running_mean_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(ring, S, C, H, g0, T, values, scale, mean, mean_int);
  return check_launch("bpv_running_mean");
}

// The same pushes over a job map: stream s pushes the values of its jobs stream_job0[s] .. stream_job0[s+1] - 1, in order,
// starting at its own history count g0[s].
namespace bpv {
__global__ void running_mean_jobs_kernel(double* __restrict__ ring, int S, int C, int H, const int64_t* __restrict__ g0,
                                         const int32_t* __restrict__ stream_job0, const double* __restrict__ values,
                                         double scale, double* __restrict__ mean, double* __restrict__ mean_int) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;     // s * C + c
  if (idx >= S * C) return;
  const int s = idx / C, c = idx % C;
  double* rg = ring + (long long)idx * H;
  const long long gs = g0[s];
  const int j0 = stream_job0[s], j1 = stream_job0[s + 1];
  for (int j = j0; j < j1; ++j) {
    const long long e = (long long)j * C + c;
    push_nanmean(rg, H, (int)((gs + (j - j0)) % H), values[e] * scale, e, mean, mean_int);
  }
}
}  // namespace bpv

extern "C" int bpv_running_mean_jobs(double* ring, int32_t S, int32_t C, int32_t H, const int64_t* g0, const int32_t* stream_job0,
                                     const double* values, double scale, double* mean, double* mean_int, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(ring && g0 && stream_job0 && values && (mean || mean_int), BPV_E_INVALID, "bpv_running_mean_jobs: NULL pointer");
  BPV_REQUIRE(S > 0 && C > 0 && H > 0 && H <= MAX_MEAN_HIST, BPV_E_INVALID, "bpv_running_mean_jobs: bad sizes (history <= 128)");
  const int n = S * C;
  running_mean_jobs_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(ring, S, C, H, g0, stream_job0, values, scale, mean,
                                                                           mean_int);
  return check_launch("bpv_running_mean_jobs");
}

// ---------------------------------------------------------------------------------------------
// Result record of a step: [J, 2R + 2P] float64 = (bpm[R], ptt_ms[P], peak_idx[R], lag_idx[P]) per window job —
// what SignalProcessor.process appends to sg_bpm / sg_ptt (signal_processor.py:310, 312: f * 60, t * 1000) plus the
// bit-exact bins; the record the multi-GPU gather and the host read-back move.
namespace bpv {
__global__ void pack_records_kernel(const double* __restrict__ peak_freq, const double* __restrict__ lag_sec,
                                    const int32_t* __restrict__ peak_idx, const int32_t* __restrict__ lag_idx,
                                    long long J, int R, int P, double* __restrict__ out) {
  const int C = 2 * R + 2 * P;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= J * C) return;
  const long long j = i / C;
  const int c = (int)(i % C);
  double v;
  if (c < R) v = peak_freq[j * R + c] * 60;
  else if (c < R + P) v = lag_sec[j * P + (c - R)] * 1000;
  else if (c < 2 * R + P) v = (double)peak_idx[j * R + (c - R - P)];
  else v = (double)lag_idx[j * P + (c - 2 * R - P)];
  out[i] = v;
}
}  // namespace bpv

extern "C" int bpv_pack_records(const double* peak_freq, const double* lag_sec, const int32_t* peak_idx,
                                const int32_t* lag_idx, int64_t J, int32_t R, int32_t P, double* out, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(peak_freq && peak_idx && out && (P == 0 || (lag_sec && lag_idx)), BPV_E_INVALID, "bpv_pack_records: NULL pointer");
  BPV_REQUIRE(J >= 0 && R > 0 && P >= 0, BPV_E_INVALID, "bpv_pack_records: bad sizes");
  if (J == 0) return 0;
  const long long n = J * (2 * R + 2 * P);
  pack_records_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(peak_freq, lag_sec, peak_idx, lag_idx, J, R, P, out);
  return check_launch("bpv_pack_records");
}


// Compact form of the same record, SURVEY.md 8(e): 4-byte words (bpm f32 [R], ptt_ms f32 [P], peak_idx i32 [R],
// lag_idx i32 [P]) = 24 B per window job at R = 2 — what the per-step NCCL gather moves.  bpm / ptt are rounded from
// the float64 result once, here; the bins travel exactly.
namespace bpv {
__global__ void pack_records32_kernel(const double* __restrict__ peak_freq, const double* __restrict__ lag_sec,
                                      const int32_t* __restrict__ peak_idx, const int32_t* __restrict__ lag_idx,
                                      long long J, int R, int P, int32_t* __restrict__ out) {
  const int C = 2 * R + 2 * P;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= J * C) return;
  const long long j = i / C;
  const int c = (int)(i % C);
  int32_t v;
  if (c < R) v = __float_as_int((float)(peak_freq[j * R + c] * 60));
  else if (c < R + P) v = __float_as_int((float)(lag_sec[j * P + (c - R)] * 1000));
  else if (c < 2 * R + P) v = peak_idx[j * R + (c - R - P)];
  else v = lag_idx[j * P + (c - 2 * R - P)];
  out[i] = v;
}
}  // namespace bpv

extern "C" int bpv_pack_records32(const double* peak_freq, const double* lag_sec, const int32_t* peak_idx,
                                  const int32_t* lag_idx, int64_t J, int32_t R, int32_t P, int32_t* out, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(peak_freq && peak_idx && out && (P == 0 || (lag_sec && lag_idx)), BPV_E_INVALID, "bpv_pack_records32: NULL pointer");
  BPV_REQUIRE(J >= 0 && R > 0 && P >= 0, BPV_E_INVALID, "bpv_pack_records32: bad sizes");
  if (J == 0) return 0;
  const long long n = J * (2 * R + 2 * P);
  pack_records32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(peak_freq, lag_sec, peak_idx, lag_idx, J, R, P, out);
  return check_launch("bpv_pack_records32");
}
