/* libbpv — C ABI of the B200-native signal path of bp-from-video.
 *
 * The reference has no FFI: its boundary is three Python modules (roi.py, signal_data.py,
 * signal_processor.py).  Our drop-in modules of the same names (bp-from-video_b200/) keep that
 * Python surface and bind THIS library through ctypes; each entry point below names the reference
 * code it replaces (file:line under /root/reference).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - every function returns int: 0 = OK, <0 = bpv error (BPV_E_*), >0 = cudaError_t.
 *     bpv_last_error() returns a thread-local message for the last non-zero return.
 *   - no allocation, no ownership transfer: every buffer is caller-owned, device-accessible memory
 *     (device memory, or pinned/mapped host memory for the zero-copy ROI path).
 *   - every call enqueues work on the caller's cudaStream_t (passed as void*; NULL = default stream)
 *     and returns without synchronising.
 *   - "signal" = one (stream, ROI) time series; "window job" = one evaluation of the sliding window
 *     of one stream (all R ROIs + C(R,2) pairs), i.e. one SignalProcessor.process() call.
 */
#ifndef BPV_H
#define BPV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BPV_VERSION 100

/* error codes (negative) */
#define BPV_E_INVALID   (-1)   /* bad argument */
#define BPV_E_UNSUPPORTED (-2) /* NotImplementedError in the reference (unknown enum value) */
#define BPV_E_TOO_LARGE (-3)   /* window does not fit the kernel's shared-memory plan */

/* SignalColorChannel (signal_processor.py:23-25) */
#define BPV_GREEN       0
#define BPV_CHROM_GREEN 1

/* SignalProcessingMethod (signal_processor.py:28-36) */
#define BPV_DIFF_1         1
#define BPV_DIFF_2         2
#define BPV_INTERP_LINEAR  3
#define BPV_INTERP_CUBIC   4
#define BPV_DETREND_CONST  5
#define BPV_DETREND_LINEAR 6
#define BPV_FILTER_BUTTER  7
#define BPV_FILTER_FIR     8
#define BPV_MAX_METHODS    8

/* SignalSpectrumTransform (signal_processor.py:39-42) */
#define BPV_DFT_RFFT    1
#define BPV_PGRAM_WELCH 2
#define BPV_PGRAM_LS    3

/* x0 sentinel for "no detection": the reference's (nan,)*6 Location (signal_processor.py:154) */
#define BPV_NO_BOX INT32_MIN

int bpv_version(void);
const char* bpv_last_error(void);

/* L2->DRAM fetch granularity hint of the device (32 / 64 / 128 bytes).  ROI rows are short unaligned
 * spans, so a smaller granularity trims the DRAM over-fetch around each row.  get returns bytes or -1. */
int bpv_set_l2_fetch_granularity(int bytes);
int bpv_get_l2_fetch_granularity(void);

/* ---------------------------------------------------------------------------------------------
 * F1  ROI sampling — replaces SignalProcessor.sample_signal / sample_signals
 *     (signal_processor.py:176-193).
 *
 * frames      uint8 HWC BGR images.  Image f starts at frames + f*frame_stride_bytes (dense batch),
 *             or at frame_ptrs[f] when frame_ptrs != NULL (then frames may be NULL).  Rows are
 *             row_stride_bytes apart (>= 3*W; supports the reference's cropped views,
 *             video_reader.py:101).  No alignment requirement.
 * boxes       int32 [num_frames, R, 4] = (x0, y0, x1, y1) exactly as the reference slices them:
 *             frame[y0:y1, x0:x1] with Python slice semantics (negative indices wrap, stops clamp,
 *             empty -> NaN).  x0 == BPV_NO_BOX -> NaN sample.
 * mode        BPV_GREEN: mean(G).  BPV_CHROM_GREEN: mean(G/2 - B/4 - R/4 + 0.5).
 * out_sums    uint64 [num_frames, R, 4] = (sumB, sumG, sumR, N) exact integers; may be NULL.
 * out_value   float64 [num_frames, R]: bit-identical to the reference's np.mean.
 * roi_pixels_hint  typical ROI area in pixels (0 = unknown); only selects threads-per-ROI.
 */
int bpv_roi_sample_u8(const uint8_t* frames, const uint8_t* const* frame_ptrs,
                      int64_t frame_stride_bytes, int64_t row_stride_bytes,
                      int32_t H, int32_t W, int64_t num_frames,
                      const int32_t* boxes, int32_t R, int32_t mode,
                      uint64_t* out_sums, double* out_value,
                      int64_t roi_pixels_hint, void* stream);

/* F1 on NV12 frames (decoder output: Y plane [H, pitch] followed by the interleaved half-resolution UV plane
 * [H/2, pitch]; frame f at frames + f*frame_stride_bytes).  The reference only ever sees the BGR frame
 * cv2.VideoCapture makes of such a buffer (video_reader.py:93); this samples the ROI from the planes directly with
 * OpenCV's integer BT.601 conversion (cvtColor COLOR_YUV2BGR_NV12), so sums and values equal those of that BGR
 * frame bit for bit.  boxes / mode / out_sums / out_value as bpv_roi_sample_u8.  H and W even. */
int bpv_roi_sample_nv12(const uint8_t* frames, int64_t frame_stride_bytes, int64_t pitch_bytes,
                        int32_t H, int32_t W, int64_t num_frames, const int32_t* boxes, int32_t R, int32_t mode,
                        uint64_t* out_sums, double* out_value, void* stream);

/* F1 on a frame the reference would first have resized: VideoReader applies cv2.resize(frame, target_res[::-1])
 * (INTER_LINEAR) to file input (video_reader.py:95-96) and boxes are expressed in the resized dst_h x dst_w frame.
 * The resized frame is never materialised: each ROI pixel is produced with OpenCV's integer bilinear arithmetic
 * (11-bit coefficients; exact 2x decimation = area fast path), so sums and values equal those of cv2.resize's output
 * bit for bit.  frames uint8 HWC BGR [num_frames] of src_h x src_w; other arguments as bpv_roi_sample_u8. */
int bpv_roi_sample_resized_u8(const uint8_t* frames, int64_t frame_stride_bytes, int64_t row_stride_bytes,
                              int32_t src_h, int32_t src_w, int32_t dst_h, int32_t dst_w, int64_t num_frames,
                              const int32_t* boxes, int32_t R, int32_t mode,
                              uint64_t* out_sums, double* out_value, void* stream);

/* F1 through a segmentation mask (SURVEY.md 8f row 4).  masks uint8 [num_frames] of H x W per-pixel categories — the
 * category_mask the reference's person segmenter returns for every frame (inference_runner.py:154-166; used there only for
 * drawing, drawer.py:95-99).  A ROI is sampled only over the pixels whose category equals categories[r] (int32 [R], device
 * memory; e.g. 3 = face skin, 2 = body skin): sums = (sumB, sumG, sumR, N) over those pixels, value = the float64
 * np.mean(channel(frame[y0:y1, x0:x1])[mask[y0:y1, x0:x1] == category]) gives; no selected pixel -> NaN.  Other arguments
 * as bpv_roi_sample_u8. */
int bpv_roi_sample_masked_u8(const uint8_t* frames, int64_t frame_stride_bytes, int64_t row_stride_bytes,
                             const uint8_t* masks, int64_t mask_frame_stride_bytes, int64_t mask_row_stride_bytes,
                             int32_t H, int32_t W, int64_t num_frames, const int32_t* boxes, int32_t R,
                             const int32_t* categories, int32_t mode, uint64_t* out_sums, double* out_value, void* stream);

/* ---------------------------------------------------------------------------------------------
 * ROI geometry for batched landmark tensors — replaces SignalProcessor.calc_rois and the ROI smoothing
 *     sg_roi.add_samples + get_means(as_int=True) (signal_processor.py:133-155, 304-305; signal_data.py:60-63).
 *
 * Per (stream, frame, ROI): present uint8 [S,T,R] (0 = no detection of the ROI's model), bbox int32 [S,T,R,4]
 * of the largest detection, points int32 [S,T,R,K,2] = the landmark points the ROI config selects (first
 * num_points[r] <= K used), rel_bbox float64 [R,4] = (left, top, right, bottom).
 * hist float64 [S,R,H,6] is the smoothing state (H = roi_max_samples; fill with NaN before the first call), g0 =
 * frames pushed so far.  Outputs: locations / smoothed float64 [S,T,R,6] (x, y, x0, y0, x1, y1; NaN rows; may be
 * NULL) and boxes int32 [S,T,R,4] ready for bpv_roi_sample_u8 (x0 == BPV_NO_BOX when no box).
 */
int bpv_calc_rois(const uint8_t* present, const int32_t* bbox, const int32_t* points,
                  const int32_t* num_points, const double* rel_bbox,
                  int32_t S, int32_t T, int32_t R, int32_t K, int32_t H, int64_t g0,
                  double* hist, double* locations, double* smoothed, int32_t* boxes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * VideoReader view in front of F1 — the reference crops the decoded frame to a centred portrait window
 *     (frame[:, left:right], video_reader.py:97-101) and mirrors it (cv2.flip(frame, 1), :103) before the signal
 *     path sees it; boxes are expressed in that view.  Maps boxes int32 [num_boxes, 4] (x0, y0, x1, y1; Python slice
 *     semantics against the view_w x view_h VIEW) onto the decoded frame in HBM: out = in-range boxes of the source
 *     frame whose ROI means equal the view's (a mean is invariant under mirroring the ROI).  No pixel is copied.
 */
int bpv_view_boxes(const int32_t* boxes, int64_t num_boxes, int32_t view_w, int32_t view_h, int32_t left,
                   int32_t flip_horizontally, int32_t* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Ring buffers — replaces Signal.add_sample / SignalGroup.add_samples for sg_raw
 *     (signal_data.py:31-35, 94-98; deque(maxlen) prefilled with NaN, signal_data.py:18-19).
 *
 * ring_t float64 [S, cap], ring_y float64 [S, R, cap]: sample with global index g (0-based count
 * since the stream started) lives at slot g % cap.  Pushes T samples per stream with global
 * indices g0 .. g0+T-1.  ts float64 [S, T]; values float64 [S, T, R] (F1's out_value).  Either of ts / values may be
 * NULL: the timestamps of a batch can be pushed ahead of its samples (they are all bpv_window_design needs).
 */
int bpv_ring_push(double* ring_t, double* ring_y, int32_t S, int32_t R, int32_t cap,
                  int64_t g0, int32_t T, const double* ts, const double* values, void* stream);

/* Ragged steps — streams that advance at their own pace (cameras that join, leave, run at other frame rates or drop
 * frames).  Stream s of a ragged step takes n[s] frames, 0 <= n[s] <= T, and behaves exactly like its own one-stream
 * pipeline fed only those frames: one reference SignalProcessor per camera.
 *
 * bpv_ring_push_ragged: stream s appends its first n[s] rows of ts [S, T] / values [S, T, R] at global indices
 *   g0[s] .. g0[s]+n[s]-1 (g0 int64 [S], n int32 [S], device memory); its other rows are not read.  Either of ts /
 *   values may be NULL, as in bpv_ring_push.  g0 is not advanced (bpv_stream_jobs writes the advanced counts). */
int bpv_ring_push_ragged(double* ring_t, double* ring_y, int32_t S, int32_t R, int32_t cap, const int64_t* g0,
                         const int32_t* n, int32_t T, const double* ts, const double* values, void* stream);

/* bpv_stream_jobs: the job map of a ragged step, built on the device (a scan over the counts, one launch; S <= 65 536).
 *   Stream s contributes n[s] window jobs (last_only = 0: one per pushed frame, as windows='every_frame') or one job when
 *   n[s] > 0 (last_only = 1: the window after its newest frame).  Jobs are laid out stream-major and, within a stream,
 *   in frame order; with every n[s] = T this is the lockstep layout job = s*T + t.  Outputs: job_stream int32 [num_jobs]
 *   (the job's stream), job_head int64 [num_jobs] (global index of the job's newest sample), stream_job0 int32 [S+1]
 *   (the jobs of stream s are stream_job0[s] .. stream_job0[s+1]-1) and g0_next int64 [S] = g0 + n (a buffer other than g0).
 *   num_jobs is the caller's sum of the job counts: the kernel always writes stream_job0 (so stream_job0[S] is the
 *   device's sum) and writes the job map and g0_next only when the two agree.  stream_job0[S] != num_jobs is the error
 *   status of a mismatch; nothing is written out of bounds.  Counts are expected in 0..T (a negative count reads as 0). */
int bpv_stream_jobs(int32_t S, const int64_t* g0, const int32_t* n, int32_t last_only, int64_t num_jobs,
                    int32_t* job_stream, int64_t* job_head, int32_t* stream_job0, int64_t* g0_next, void* stream);
/* bpv_stream_jobs_strided: the job map of a step with a window cadence (windows evaluated every stride[s]-th sample of
 *   stream s).  Stream s evaluates its window after its m-th sample (m = 1, 2, ...; global index m - 1) exactly when
 *   (m + phase[s]) % stride[s] == 0; the phase is tied to the stream's own count, so it carries across steps.  Of a step in
 *   which it holds c = g0[s] samples and takes n[s] frames it contributes q = floor((c + n + phase) / stride) -
 *   floor((c + phase) / stride) jobs, job i (0 <= i < q) with its newest sample at (floor((c + phase) / stride) + 1 + i) *
 *   stride - phase - 1.  stride = phase = 1 / 0 everywhere is bpv_stream_jobs with last_only = 0.  stride, phase: int32 [S]
 *   in device memory; NULL reads as 1 / 0 for every stream.  A stride below 1 reads as 1 and a phase as its remainder
 *   modulo the stride, in [0, stride), so whatever the entries hold a stream takes between 0 and n[s] jobs.  The
 *   arithmetic is 64-bit.  Outputs, num_jobs, the mismatch status and the bounds are those of bpv_stream_jobs; one launch
 *   for up to 65 536 streams. */
int bpv_stream_jobs_strided(int32_t S, const int64_t* g0, const int32_t* n, const int32_t* stride, const int32_t* phase,
                            int64_t num_jobs, int32_t* job_stream, int64_t* job_head, int32_t* stream_job0, int64_t* g0_next,
                            void* stream);

/* Running means of the per-frame results — replaces sg_bpm / sg_ptt (deque(maxlen=peak_max_samples)) and
 * their get_means() (signal_processor.py:49, 83-84, 310, 312; signal_data.py:60-63; read by drawer.py:134-135).
 * ring float64 [S, C, H] (NaN-initialised state, H = peak_max_samples <= 128), values float64 [S, T, C] (e.g.
 * peak_freq of the step's S*T jobs), scale = 60 (bpm) or 1000 (ptt ms).  After each of the T pushes:
 * mean float64 [S, T, C] = np.nanmean of the history (numpy's summation order), mean_int = its half-to-even
 * round (NaN when the history holds no finite value).  Either output may be NULL.
 */
int bpv_running_mean(double* ring, int32_t S, int32_t C, int32_t H, int64_t g0, int32_t T,
                     const double* values, double scale, double* mean, double* mean_int, void* stream);
/* The running means of a ragged step: stream s pushes the values of its jobs stream_job0[s] .. stream_job0[s+1]-1 (the
 * map of bpv_stream_jobs) in order, from its own history count g0[s] (int64 [S], device memory; not advanced: it grows
 * by the stream's job count).  values, mean, mean_int float64 [J, C] over the step's jobs; otherwise as bpv_running_mean. */
int bpv_running_mean_jobs(double* ring, int32_t S, int32_t C, int32_t H, const int64_t* g0, const int32_t* stream_job0,
                          const double* values, double scale, double* mean, double* mean_int, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Window jobs.  A window job j of stream s looks at the `window` samples whose newest global
 * index is head(j) = head0 + j*head_step (samples with negative global index read as NaN,
 * exactly the NaN prefill of the reference's deque).  J = S * jobs_per_stream jobs in all, job id
 * = s*jobs_per_stream + j.  All per-job outputs are laid out [J, R, ...] / [J, P, ...].
 */
typedef struct bpv_window_params {
  int32_t S, R, cap, window;        /* ring geometry; window = signal_max_samples (<= cap)        */
  int64_t head0;                    /* global index of the newest sample of job 0 of each stream  */
  int32_t head_step;                /* global-index step between consecutive jobs of a stream     */
  int32_t jobs_per_stream;
  int32_t num_methods;              /* processing_methods, applied in order                       */
  int32_t methods[BPV_MAX_METHODS];
  int32_t transform;                /* BPV_DFT_RFFT / BPV_PGRAM_WELCH / BPV_PGRAM_LS              */
  int32_t butter_order;             /* signal_processor.py:57 (even, <= 16)                       */
  int32_t fir_taps;                 /* signal_processor.py:59 (odd, <= 127)                       */
  int32_t ls_num_freqs;             /* 0 = reference behaviour (F = n valid); >0 fixed grid       */
  double butter_min_bw, fir_df, min_freq, max_freq;   /* signal_processor.py:58,60,64,65          */
} bpv_window_params;
int bpv_sizeof_window_params(void);   /* lets a binding verify its struct layout */

/* F2 preprocessing — replaces SignalProcessor.process_signal(s) + make_filter
 *     (signal_processor.py:158-173, 196-245).
 * proc_x, proc_y float64 [J, R, window]: the processed window, position-preserving (NaN where the
 * reference's arrays hold NaN).  status int32 [J, R]: 0 ok, 1 = guard failed (copied through
 * unprocessed, signal_processor.py:200), 2 = INTERP_CUBIC saw non-increasing x (the reference
 * raises ValueError there), 3 = filter band edges invalid for this fs (scipy raises ValueError).
 * workspace: caller-owned device scratch of bpv_window_workspace_bytes(p) bytes holding the per-job
 * filters (needed only when a FILTER_* method is listed).
 */
int64_t bpv_window_workspace_bytes(const bpv_window_params* p);
int bpv_window_preprocess(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                          void* workspace, int64_t workspace_bytes,
                          double* proc_x, double* proc_y, int32_t* status, void* stream);
/* The two halves of bpv_window_preprocess, for callers that overlap them or keep a design cache:
 * bpv_window_design — make_filter for every window job (signal_processor.py:158-173, called per frame and signal at
 *   :226, :232): needs only the timestamps (ring_t), so it can run on another stream as soon as they are pushed, beside
 *   the ROI sampling of the same frames.  Fills `workspace` (per job: Butterworth sos | FIR taps | lfilter_zi | the
 *   2T-1 taps of the merged forward.backward filter, i.e. the tap autocorrelation laid out symmetrically).
 * bpv_window_filter — process_signal given the designs (same stream, or after an event on the design).
 * cache (optional, may be NULL): caller-owned device memory of bpv_design_cache_bytes() bytes, zero-initialised, kept
 *   across calls.  make_filter is a pure function of the window's sampling rate; the cache is a table keyed by the 64 bits
 *   of fs, so a rate that has been designed before (constant-fps streams: every window, every stream on the same clock)
 *   costs a lookup instead of a design.  Hits return the very bits a fresh design produces.  The table belongs to ONE
 *   set of filter parameters (orders, taps, band edges): zero it when they change.  Pass the same cache to both calls. */
int64_t bpv_design_cache_bytes(void);
int bpv_window_design(const double* ring_t, const bpv_window_params* p, void* workspace, int64_t workspace_bytes,
                      void* cache, int64_t cache_bytes, void* stream);
int bpv_window_filter(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                      const void* workspace, int64_t workspace_bytes, const void* cache, int64_t cache_bytes,
                      double* proc_x, double* proc_y, int32_t* status, void* stream);
/* F2 over a job map (ragged steps, bpv_stream_jobs): the same calls with job k reading ring row job_stream[k] and the
 * window whose newest sample has global index job_head[k].  p->S / R / cap / window describe the rings; head0 /
 * head_step / jobs_per_stream are ignored.  Outputs (proc_x, proc_y, status, and the per-job filter designs) are laid
 * out over the num_jobs jobs as the lockstep calls lay them out over J = num_jobs.  The workspace must hold
 * bpv_window_workspace_bytes() of params with S * jobs_per_stream >= num_jobs (e.g. the engine's largest lockstep step).
 * job_stream entries must lie in [0, p->S).  num_jobs = 0 enqueues nothing; num_jobs < 0 or a NULL map is BPV_E_INVALID.
 * The kernels are the lockstep ones compiled with a job-map switch: the results of a job equal those of the lockstep job
 * with the same stream and head bit for bit. */
int bpv_window_design_jobs(const double* ring_t, const bpv_window_params* p, void* workspace, int64_t workspace_bytes,
                           void* cache, int64_t cache_bytes, const int32_t* job_stream, const int64_t* job_head,
                           int64_t num_jobs, void* stream);
int bpv_window_filter_jobs(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                           const void* workspace, int64_t workspace_bytes, const void* cache, int64_t cache_bytes,
                           double* proc_x, double* proc_y, int32_t* status, const int32_t* job_stream,
                           const int64_t* job_head, int64_t num_jobs, void* stream);
int bpv_window_preprocess_jobs(const double* ring_t, const double* ring_y, const bpv_window_params* p,
                               void* workspace, int64_t workspace_bytes, double* proc_x, double* proc_y, int32_t* status,
                               const int32_t* job_stream, const int64_t* job_head, int64_t num_jobs, void* stream);

/* F3 + F4(a) spectrum and HR peak — replaces transform_signal(s) + SignalGroup.get_peaks on
 *     sg_spec (signal_processor.py:248-277, 310; signal_data.py:65-70 with the range reset of
 *     signal_data.py:82-86 => search over every finite bin).
 * spec_f, spec_mag float32 [J, R, max_bins] (first num_bins[j,r] entries valid; may be NULL to skip
 * storing the spectrum); num_bins int32 [J, R]; peak_idx int32 [J, R] (-1 = none);
 * peak_freq, peak_mag float64 [J, R] (NaN = none).  The peak is decided in float64.
 * workspace: device memory of bpv_spectrum_workspace_bytes() bytes: for DFT_RFFT first the twiddle operand images of the
 * tensor-core kernel (at offset 0 whatever the job count of the call), then scratch for the coarse spectrum of PGRAM_LS /
 * DFT_RFFT when it is not stored (spec_mag == NULL).  Zero it once and pass the SAME buffer on every call: the images are
 * built on first use and reused while the window length stays the same, by calls of any job count.  Without it (NULL / too small) DFT_RFFT generates its operands inside the kernel.
 */
/* F3 and F4 only ever use the J = S * jobs_per_stream processed windows, never p->S or a head on its own: the jobs of a
 * ragged step are passed as params with S = num_jobs, jobs_per_stream = 1. */
int64_t bpv_spectrum_workspace_bytes(const bpv_window_params* p, int32_t max_bins);
int bpv_window_spectrum(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                        int32_t max_bins, void* workspace, int64_t workspace_bytes,
                        float* spec_f, float* spec_mag, int32_t* num_bins,
                        int32_t* peak_idx, double* peak_freq, double* peak_mag, void* stream);
/* Band-limited HR peak — what a single transform_signal(s).get_peak() searches (signal_processor.py:272 sets the range to
 *     (min_freq, max_freq); signal_data.py:65-70), where process() searches every bin.  Same arguments and spectra as
 * bpv_window_spectrum; the peak is the first maximum over the bins k with a finite magnitude and
 * min_freq <= x_k <= max_freq, x_k being the float64 frequency the kernel reports for the bin (k * fval for DFT_RFFT /
 * PGRAM_WELCH, the linspace value for PGRAM_LS).  Fewer than two such bins: no peak (-1 / NaN).  peak_idx still indexes
 * the full spectrum, and spec_f / spec_mag / num_bins do not depend on the band.  (-INFINITY, INFINITY) is
 * bpv_window_spectrum bit for bit (which forwards here); min_freq > max_freq gives no peak; a NaN bound returns
 * BPV_E_INVALID before anything is enqueued. */
int bpv_window_spectrum_band(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                             int32_t max_bins, void* workspace, int64_t workspace_bytes,
                             float* spec_f, float* spec_mag, int32_t* num_bins,
                             int32_t* peak_idx, double* peak_freq, double* peak_mag,
                             double min_freq, double max_freq, void* stream);

/* F4(b) pairwise cross-correlation lag search — replaces correlate_signal_pair / correlate_signals
 *     + get_peaks on sg_corr (signal_processor.py:280-299, 312).  Pairs in
 *     itertools.combinations order, P = R*(R-1)/2.
 * corr_lag, corr_val float32 [J, P, 2*window-1] (first num_lags[j,p] valid; may be NULL);
 * lag_idx int32 [J, P] index into the 2n-1 lags (-1 = none); lag_sec, lag_corr float64 [J, P].
 */
int bpv_window_xcorr(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                     float* corr_lag, float* corr_val, int32_t* num_lags,
                     int32_t* lag_idx, double* lag_sec, double* lag_corr, void* stream);
/* Band-limited PTT lag — what a single correlate_signal_pair(a, b).get_peak() searches (signal_processor.py:294 sets the
 *     range to (min_lag, max_lag) = (-0.5, 0.5) s).  Same arguments and correlations as bpv_window_xcorr; the peak is the
 * first maximum over the lags with a finite correlation and min_lag <= x_k <= max_lag, x_k = (x_last - x[pos[n-1-|k|]]) *
 * sign(k) being the float64 lag in seconds reported as lag_sec, evaluated lag by lag (timestamps need not be monotone).
 * Fewer than two such lags: no peak.  lag_idx still indexes the 2n-1 lags.  (-INFINITY, INFINITY) is bpv_window_xcorr bit
 * for bit (which forwards here); min_lag > max_lag gives no peak; a NaN bound returns BPV_E_INVALID before anything is
 * enqueued. */
int bpv_window_xcorr_band(const double* proc_x, const double* proc_y, const bpv_window_params* p,
                          float* corr_lag, float* corr_val, int32_t* num_lags,
                          int32_t* lag_idx, double* lag_sec, double* lag_corr,
                          double min_lag, double max_lag, void* stream);

/* F3 + F4 of the same window jobs in ONE grid (PGRAM_WELCH only; unbanded peaks): CTAs of the Welch kernel and of the cross-correlation
 *     kernel interleaved in the ratio of their counts, so that every SM holds both for the whole launch (the two are bound
 *     by different things — shared-memory wavefronts vs FP32 issue — and mix poorly when launched as two kernels).
 *     Same arguments and results, bit for bit, as bpv_window_spectrum followed by bpv_window_xcorr; shapes the fused grid
 *     does not cover (windows over 320 samples, R = 1) run as those two launches on `stream`.
 *     MEASURED SLOWER on B200 than the two kernels on two streams (272.9 against 227.5 us per 16 384 window jobs,
 *     profiles/r4g_*): an experiment kept for reference — the engine does not use it unless asked (overlap bit 4). */
int bpv_window_welch_xcorr(const double* proc_x, const double* proc_y, const bpv_window_params* p, int32_t max_bins,
                           float* spec_f, float* spec_mag, int32_t* num_bins, int32_t* peak_idx, double* peak_freq,
                           double* peak_mag, float* corr_lag, float* corr_val, int32_t* num_lags, int32_t* lag_idx,
                           double* lag_sec, double* lag_corr, void* stream);

/* Per-window signal quality: spectral SNR of the heart-rate peak (de Haan & Jeanne, IEEE TBME 2013) over the spectrum
 *     F3 stored, and the SNR gate of the values the running means push.  No reference counterpart: process() reports a
 *     peak for every window, whether the ROI held a pulse or not.
 * Inputs: spec_f, spec_mag float32 [J, R, max_bins], num_bins, peak_idx int32 [J, R] as bpv_window_spectrum(_band) wrote
 * them.  For signal (j, r), in float64 arithmetic on the stored float32 values f_k, m_k widened to float64:
 *   - bin power P_k = m_k^2 for BPV_DFT_RFFT (the stored spectrum is the amplitude 2|X|/n), m_k for PGRAM_WELCH / PGRAM_LS;
 *   - B = the bins k < num_bins with a finite m_k and lo <= f_k <= hi;
 *   - f0 = f_{peak_idx}; a bin is in the template when |f_k - f0| <= half_width or |f_k - 2 f0| <= half_width (Hz);
 *   - S_sig = sum of P_k over B within the template, S_noise = over B outside it;
 *   - snr_db = 10 log10(S_sig / S_noise) with IEEE semantics (0/x -> -inf, x/0 -> +inf, 0/0 -> NaN); NaN when
 *     peak_idx < 0 or |B| < 2.  A DC peak of the unbanded search puts no template bin in a band above 0 Hz: -inf.
 * B is decided on the stored float32 frequencies, so it can differ from the band of bpv_window_spectrum_band (which decides
 * on float64 frequencies) in a bin that lies within float32 rounding of lo or hi.  The sums are float64 in a fixed lane
 * order and shuffle tree: reproducible from run to run.
 * Gate (optional outputs, NULL to skip): a heart rate is accepted when snr_db >= min_snr_db (NaN is rejected); the PTT of
 * pair (a, b), itertools.combinations order, when both a and b are.  gated_freq [J, R] = peak_freq where accepted, else
 * NaN; gated_lag [J, P] = lag_sec likewise.  snr_db float64 [J, R] is always written.  P must be R(R-1)/2.
 * BPV_E_INVALID before anything is enqueued: a NaN bound, a negative or non-finite half_width, a NaN min_snr_db (-inf is
 * allowed), J < 0, R < 1, max_bins < 1, a bad P or transform, a NULL input / snr_db, gated_freq without peak_freq,
 * gated_lag without lag_sec.  J = 0 enqueues nothing.  lo > hi leaves B empty (NaN). */
int bpv_window_snr(const float* spec_f, const float* spec_mag, const int32_t* num_bins, const int32_t* peak_idx,
                   int64_t J, int32_t R, int32_t max_bins, int32_t transform, double lo, double hi, double half_width,
                   const double* peak_freq, const double* lag_sec, int32_t P, double min_snr_db,
                   double* snr_db, double* gated_freq, double* gated_lag, void* stream);

/* Filter design alone (debug / parity of make_filter, signal_processor.py:158-173).
 * fs float64 [n]; sos_out float64 [n, order, 6]; taps_out float64 [n, fir_taps]. */
int bpv_butter_sos_design(const double* fs, int32_t n, const bpv_window_params* p, double* sos_out, void* stream);
int bpv_firls_design(const double* fs, int32_t n, const bpv_window_params* p, double* taps_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Result record of a step — what SignalProcessor.process appends to sg_bpm / sg_ptt
 *     (signal_processor.py:310, 312: f * 60, t * 1000) plus the bit-exact bins.
 * out float64 [J, 2R + 2P] = (bpm[R], ptt_ms[P], peak_idx[R], lag_idx[P]) per window job: the record the multi-GPU
 * gather and the host read-back move.
 */
int bpv_pack_records(const double* peak_freq, const double* lag_sec, const int32_t* peak_idx, const int32_t* lag_idx,
                     int64_t J, int32_t R, int32_t P, double* out, void* stream);
/* Compact record, SURVEY.md 8(e): out int32 [J, 2R + 2P] 4-byte words = (bpm f32 [R], ptt_ms f32 [P], peak_idx i32 [R],
 * lag_idx i32 [P]) — 24 B per window job at R = 2; the payload of the per-step multi-GPU gather. */
int bpv_pack_records32(const double* peak_freq, const double* lag_sec, const int32_t* peak_idx, const int32_t* lag_idx,
                       int64_t J, int32_t R, int32_t P, int32_t* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Scratch hygiene (no reference counterpart: the reference's intermediate arrays die in the CPU cache).  Drops the
 * 128-byte L2 lines that lie entirely inside [ptr, ptr + bytes) WITHOUT writing them back to DRAM (discard.global.L2);
 * the contents of the range are undefined afterwards.  The engine calls it on the processed windows once F3 and F4 have
 * consumed them, so that ~80 MB of dead dirty lines per step do not compete with the next step's ROI sampling for DRAM.
 */
int bpv_scratch_discard(void* ptr, int64_t bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core building block of the spectra: 256-point DFT of `rows` real segments as one dense contraction on the
 * 5th-generation tensor cores (tcgen05.mma kind::tf32 with hi/lo split operands, fp32 accumulators in TMEM) — the
 * transform inside scipy.signal.welch(y, fs) as the reference calls it (signal_processor.py:260, nperseg = 256).
 * z float32 [rows, 256]; d float32 [rows, 256]: d[:, 0..128] = Re X[0..128], d[:, 129..255] = -Im X[1..127].
 */
int bpv_dft256_tc(const float* z, int32_t rows, float* d, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Measurement aid (bench.py roofline of the FP64 / FP32 bound families; not part of the reference path): a grid of
 * `blocks` x 256 threads, each running `iters` rounds of 8 independent dependent-chain fused multiply-adds in
 * float64 (dtype 1) or float32 (dtype 0).  Returns the number of FMAs enqueued (2 flop each) or a negative error;
 * sink = >= 8 bytes of device memory (written only if a result is non-finite, so the loop is not optimised away). */
int64_t bpv_probe_fma(int32_t dtype, int64_t iters, int32_t blocks, void* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BPV_H */
