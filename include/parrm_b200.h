/*
 * parrm_b200.h -- C ABI of libparrm_b200.so: the PARRM hot path on NVIDIA B200 (sm_100a).
 *
 * The reference (neuromodulation/PyPARRM) is pure Python and has no FFI of its
 * own; its boundary for this path is the private seams of `pyparrm.PARRM`
 * (src/pyparrm/parrm.py).  Each entry point below replaces one of those seams
 * and cites it.  The Python host (`pyparrm_b200/parrm.py`) binds these with
 * ctypes (`pyparrm_b200/_native.py`); INTEGRATION.md shows the same stub as a
 * maintainer of the reference would add it.
 *
 * Conventions
 *   - Every function returns a parrm_status_t (0 = success).  On failure a
 *     thread-local message is available from parrm_last_error().
 *   - Pointers named d_* are DEVICE pointers owned by the caller (PyTorch tensors
 *     in the shipped host); h_* are host pointers.  The library never allocates or
 *     frees device memory and never synchronises the device: work is enqueued on
 *     `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).
 *     Scratch space is passed in as (d_workspace, workspace_bytes); sizes come
 *     from the *_workspace_bytes functions.
 *   - Recordings are row-major [n_chans, n_samples] with a row stride `ld`
 *     counted in elements.  dtype selects float64 (reference arithmetic,
 *     rel. err <= 1e-9) or float32 storage (<= 1e-4).
 *   - No global mutable state apart from the thread-local error string.
 */
#ifndef PARRM_B200_H
#define PARRM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PARRM_B200_ABI_VERSION 9

typedef enum {
  PARRM_OK = 0,
  PARRM_ERR_INVALID_ARGUMENT = 1,
  PARRM_ERR_CUDA = 2,           /* a CUDA runtime call failed (no device, launch error, ...) */
  PARRM_ERR_WORKSPACE = 3,      /* workspace too small */
  PARRM_ERR_UNSUPPORTED = 4     /* e.g. bandwidth above PARRM_MAX_BANDWIDTH */
} parrm_status_t;

typedef enum { PARRM_F64 = 0, PARRM_F32 = 1 } parrm_dtype_t;
/* what a recording may be stored as on its way in (parrm_convert widens it on the device) */
typedef enum { PARRM_I16 = 2, PARRM_I32 = 3 } parrm_storage_t;

/* filter_direction strings of PARRM.create_filter (parrm.py:710-714, 817-820) */
typedef enum { PARRM_DIR_BOTH = 0, PARRM_DIR_PAST = 1, PARRM_DIR_FUTURE = 2 } parrm_direction_t;

/* how parrm_filter_plan() may re-associate the tap sum (the result is the same tap set) */
typedef enum {
  PARRM_PLAN_AUTO = 0,    /* comb boxes when the tap set has progressions, else plain gather */
  PARRM_PLAN_GATHER = 1,  /* one load per tap */
  PARRM_PLAN_COMB = 2     /* comb boxes; PARRM_ERR_UNSUPPORTED if the tap set has none */
} parrm_plan_strategy_t;

#define PARRM_MAX_BANDWIDTH 23  /* harmonics per candidate; the reference uses 5/10/20 (parrm.py:295) */

int         parrm_abi_version(void);
const char* parrm_last_error(void);
/* Number of visible CUDA devices (0 on a CPU-only host; never fails). */
int         parrm_device_count(void);
/* 1 if the host pointer lies in page-locked (pinned / registered) memory, else 0.  The host
 * pipeline uses it to choose between direct async copies and staged ones. */
int         parrm_host_is_pinned(const void* h_ptr);
/* cudaMemcpyAsync wrappers for the host pipeline (pageable pointers are legal but make the
 * copy synchronous with respect to the host, as CUDA defines). */
int         parrm_copy_h2d_async(void* d_dst, const void* h_src, size_t bytes, void* stream);
int         parrm_copy_d2h_async(void* h_dst, const void* d_src, size_t bytes, void* stream);
/* cudaMemcpy2DAsync wrappers: `height` rows of `width` bytes, source rows src_pitch bytes apart,
 * destination rows dst_pitch bytes apart (both >= width).  They move one time window of a
 * recording between its place in a larger host array ([C, T] rows, or the [T, ld] rows of a
 * time-major array) and a dense device buffer, without touching the bytes between the rows. */
int         parrm_copy_h2d_2d_async(void* d_dst, size_t dst_pitch, const void* h_src,
                                    size_t src_pitch, size_t width, size_t height, void* stream);
int         parrm_copy_d2h_2d_async(void* h_dst, size_t dst_pitch, const void* d_src,
                                    size_t src_pitch, size_t width, size_t height, void* stream);
/* Page-lock / release a host range in place (cudaHostRegister): a caller that filters or
 * searches the same NumPy array repeatedly registers it once instead of having every call
 * staged through pinned buffers (PARRM holds `data` by reference, parrm.py:124). */
int         parrm_host_register(void* h_ptr, size_t bytes);
int         parrm_host_unregister(void* h_ptr);
/* Host-to-host copy on up to n_threads threads of a persistent pool, streaming stores for
 * large pieces: the staged leg of the host pipeline, where a pageable recording (the
 * reference takes any ndarray, parrm.py:877-886, 120-124) is moved through page-locked
 * staging buffers.  Blocks until the copy is complete; ranges must not overlap. */
int         parrm_host_copy(void* h_dst, const void* h_src, size_t bytes, int n_threads);

/* ------------------------------------------------------------------------
 * Standardisation: PARRM._standardise_data (parrm.py:272-280)
 *   d[c,t] = x[c,t+1]-x[c,t];  s_c = mean_t |d[c,t]|;  z = clip(d/s_c, -ob, +ob)
 * Only the columns the search fits are ever consumed (parrm.py:589-591), so the
 * device path computes s_c in one streaming pass and gathers z at `indices`.
 * ---------------------------------------------------------------------- */
size_t parrm_channel_scales_workspace_bytes(int64_t n_chans, int64_t n_samples);
/* d_scale[c] = mean |diff| of channel c (float64 regardless of dtype). */
int parrm_channel_scales(const void* d_x, int64_t n_chans, int64_t n_samples, int64_t ld,
                         double* d_scale, void* d_workspace, size_t workspace_bytes,
                         int dtype, void* stream);
/* d_y[c, j] = clip((x[c, idx_j + 1] - x[c, idx_j]) / scale[c]); also d_sumsq[c] = sum_j y^2
 * (float64; may be NULL).  d_y is float64, SAMPLE-MAJOR: d_y[j * ld_y + c], ld_y >= n_chans
 * (the layout the evaluator's shared-memory tiles want). */
int parrm_standardise_gather(const void* d_x, int64_t n_chans, int64_t n_samples, int64_t ld,
                             const int64_t* d_indices, int64_t n_indices,
                             const double* d_scale, double outlier_boundary,
                             double* d_y, int64_t ld_y, double* d_sumsq,
                             int dtype, void* stream);
/* d_sumsq[c] = sum_j d_y[j * ld_y + c]^2 for a tile the caller standardised itself (the
 * `_optimise_local(period, data, indices, ...)` seam, parrm.py:552-559). */
int parrm_channel_sumsq(const void* d_y, int y_dtype, int64_t ld_y, int64_t n_chans,
                        int64_t n_indices, double* d_sumsq, void* stream);
/* Full z[c, 0..n_samples-2] (the `_standard_data` attribute), same dtype as x. */
int parrm_standardise_full(const void* d_x, int64_t n_chans, int64_t n_samples, int64_t ld,
                           const double* d_scale, double outlier_boundary,
                           void* d_z, int64_t ld_z, int dtype, void* stream);

/* ------------------------------------------------------------------------
 * Period-candidate evaluator: PARRM._optimise_local + _fit_waves_to_data
 * (parrm.py:552-632), batched over candidates (the pqdm map of parrm.py:445-454
 * and the Nelder-Mead evaluations of parrm.py:499-517, 545-550).
 *
 * For every candidate p:  a_i = (idx_i + 1) * (2 pi / p);  W = [1, sin k a, cos k a]_{k<=bw};
 * per channel beta = solve(W'W, W'y);  e_c = mean (y - W beta)^2 + sum_j lambda*j/sum(1..M) beta_j^2;
 * fit_error[p] = sum_c e_c / n_chans_divisor;  +inf when the factorisation meets a zero pivot
 * (the reference's LinAlgError -> inf, parrm.py:592-593, 627-628).
 * ---------------------------------------------------------------------- */
size_t parrm_eval_workspace_bytes(int64_t n_chans, int64_t n_indices, int64_t n_periods,
                                  int bandwidth);
/* Kernels one parrm_eval_periods call with these arguments enqueues (accumulate + solve, plus
 * the column-sum pair, the dense copy of y and the partial sums where the shape needs them);
 * 0 for an empty or invalid shape.  For launch accounting (bench.py's gpu_launches). */
int parrm_eval_launch_count(const double* d_y, int64_t ld_y, int64_t n_chans, int64_t n_indices,
                            int64_t n_periods, int bandwidth);
int parrm_eval_periods(const double* d_y, int64_t ld_y, const double* d_sumsq,
                       const int64_t* d_indices, int64_t n_chans, int64_t n_indices,
                       const double* d_periods, int64_t n_periods,
                       int bandwidth, double lambda, int64_t n_chans_divisor,
                       double* d_fit_error,
                       void* d_workspace, size_t workspace_bytes, void* stream);
/* The same with the tile's storage type given: y_dtype = PARRM_F64 (as above) or PARRM_F32,
 * the search's "fp32" mode (SURVEY 8(b) proposed `dtype` here; BASELINE north_star: period
 * within 1e-4).  Policy: float32 STORAGE of the standardised tile -- what is resident in L2,
 * what parrm_standardise_gather's consumers keep and what the sharded search all-gathers --
 * widened once per call; the fit itself stays on the FP64 tensor path (DMMA).  An FP32
 * CUDA-core accumulate was rejected on measurement grounds: B200's FP32 FMA peak is only 2x
 * its DMMA rate, a register-tiled FFMA GEMM of this shape (40 x 64 x N) reaches well under
 * half of it, and sums over 25 000 samples in float32 cost the objective ~1e-4 of its value;
 * TF32 tensor cores (10-bit mantissa) are not used anywhere. */
size_t parrm_eval_workspace_bytes_typed(int64_t n_chans, int64_t n_indices, int64_t n_periods,
                                        int bandwidth, int y_dtype);
int parrm_eval_periods_typed(const void* d_y, int y_dtype, int64_t ld_y, const double* d_sumsq,
                             const int64_t* d_indices, int64_t n_chans, int64_t n_indices,
                             const double* d_periods, int64_t n_periods,
                             int bandwidth, double lambda, int64_t n_chans_divisor,
                             double* d_fit_error,
                             void* d_workspace, size_t workspace_bytes, void* stream);
/* First index of the smallest non-NaN value (NaN entries are skipped; all-NaN -> index 0). */
int parrm_argmin(const double* d_values, int64_t n, double* d_min_value, int64_t* d_min_index,
                 void* stream);

/* ------------------------------------------------------------------------
 * Tap builder: PARRM._generate_filter (parrm.py:803-833), integer-exact.
 *   w in [-hw, hw] is a tap iff (mod(w, period) <= phw or >= period - phw) and |w| > omit,
 *   "past" drops w > 0, "future" drops w <= 0.  mod is NumPy's (fmod + sign fix-up).
 * d_taps (capacity 2*hw+1) receives the signed offsets ascending; *d_n_taps their count
 * (0 = the reference's RuntimeError "A suitable filter cannot be created").
 * ---------------------------------------------------------------------- */
int parrm_build_taps(double period, double period_half_width, int64_t filter_half_width,
                     int64_t omit_n_samples, int direction,
                     int32_t* d_taps, int32_t* d_n_taps, void* stream);

/* ------------------------------------------------------------------------
 * Filter application: body of PARRM.filter_data (parrm.py:861-869).
 *   y[c,t] = x[c,t] - (1/n_in(t)) * sum_{w in taps, 0 <= t-w < T} x[c,t-w];  y = 0 where n_in(t) = 0
 * (all tap weights are -1/n_taps, parrm.py:829, so the edge renormalisation of
 *  parrm.py:861-866 reduces to the mean over the in-range taps).
 *
 * Time-chunk form (for halo'd shards, SURVEY 8(e)): the output covers global times
 * [t0, t0 + n_out) of a recording of n_samples_total samples; d_x holds global times
 * [x_t0, x_t0 + n_x) and must contain every in-range sample the outputs touch, i.e.
 * [max(0, t0 - w_max), min(T, t0 + n_out - w_min)).  For a whole recording pass
 * x_t0 = t0 = 0 and n_x = n_out = n_samples_total.
 *
 * The tap list is passed as a "plan": an opaque relocatable blob that
 * parrm_filter_plan() builds on the host from the ascending tap offsets (as produced by
 * parrm_build_taps) and that the caller uploads verbatim; parrm_filter_apply() takes both
 * the host copy (launch geometry) and the device copy (read by the kernels).
 *
 * Every tap has the same weight (parrm.py:829), so the planner may regroup the tap set into
 * windowed stride-d sums ("comb boxes") plus single taps -- an exact identity over which
 * offsets are summed, pyparrm_b200/csrc/filter_plan.h -- which the run-time specialised kernel
 * evaluates with ~10x fewer shared-memory loads than one load per tap.
 * parrm_filter_plan_info() exposes the decomposition (tests expand it back into the tap set).
 * ---------------------------------------------------------------------- */
size_t parrm_filter_plan_bytes(const int32_t* h_taps, int32_t n_taps);
int parrm_filter_plan(const int32_t* h_taps, int32_t n_taps, int dtype, int strategy,
                      void* h_plan, size_t plan_bytes);
/* info[0..15] = kind, stride, n_kinds, window0, window1, n_box0, n_box1, n_plus, n_minus,
 * centre, cost_milli, n_taps, w_min, w_max, n_terms, 0;  terms (capacity >= n_terms, may be
 * NULL) = box offsets of length 0, of length 1, +1 taps, -1 taps. */
int parrm_filter_plan_info(const void* h_plan, int32_t* info, int32_t* terms, int32_t capacity);
int parrm_filter_apply(const void* d_x, int64_t ld_x, int64_t x_t0, int64_t n_x,
                       void* d_out, int64_t ld_out, int64_t t0, int64_t n_out,
                       int64_t n_samples_total, int64_t n_chans,
                       const void* d_plan, const void* h_plan,
                       int dtype, void* stream);

/* Which kernel evaluates the plan.  AUTO picks, for comb plans, a kernel SPECIALISED for the
 * plan at run time (NVRTC, sm_100a: stride, box lengths and tap offsets are immediates; built
 * once per plan and device, about a second) when the call is large enough (2^24
 * channel-samples) to be worth it or the kernel already exists, else the pre-built GATHER
 * (one shared-memory load per tap).  Both compute the same tap sum; they differ in
 * floating-point association only.  (Value 2 was the round-1 strip kernel, removed.) */
typedef enum {
  PARRM_FILTER_KERNEL_AUTO = 0,
  PARRM_FILTER_KERNEL_GATHER = 1,
  PARRM_FILTER_KERNEL_SPECIALISED = 3
} parrm_filter_kernel_t;

/* Launch options of parrm_filter_apply_ex (all zero = library defaults; NULL allowed). */
typedef struct {
  int32_t kernel;           /* parrm_filter_kernel_t */
  int32_t steps_per_chunk;  /* specialised kernel: comb steps per TMA chunk */
  int32_t prefetch_chunks;  /* specialised kernel: chunks in flight beyond the tap window */
  int32_t ctas_per_sm;      /* specialised kernel: resident CTAs per SM (1 or 2) */
  int32_t variant;          /* specialised kernel, measurement aids (0 = default): 2 = record the
                             * per-CTA timeline, 4 = strips of equal length instead of equal cost */
  int32_t reserved;
  uint64_t timeline;        /* profiling aid, 0 = off: device pointer to 4 uint64 per CTA (SM id,
                             * start ns, end ns, pieces); written only with variant & 2 */
} parrm_filter_options_t;

int parrm_filter_apply_ex(const void* d_x, int64_t ld_x, int64_t x_t0, int64_t n_x,
                          void* d_out, int64_t ld_out, int64_t t0, int64_t n_out,
                          int64_t n_samples_total, int64_t n_chans,
                          const void* d_plan, const void* h_plan,
                          int dtype, const parrm_filter_options_t* options, void* stream);
/* Name of the kernel the calling thread's last parrm_filter_apply* enqueued ("" before the
 * first call): tests and bench.py assert on it so that a fallback is never silent. */
const char* parrm_filter_last_kernel(void);
/* Builds the specialised kernel for a plan WITHOUT loading or launching it (works on a host
 * with no GPU): the build check of the run-time compiled path.  shape[0..11] (may be NULL) =
 * stride, box kinds, M0, M1, boxes of M0, boxes of M1, single taps, steps per chunk, chunks
 * in flight, CTAs per SM, dynamic shared memory bytes, threads per CTA.  With cubin_bytes
 * NULL only the shape is worked out (is the plan inside the kernel's range?) and nothing is
 * compiled; otherwise *cubin_bytes receives the size of the compiled image.
 * PARRM_ERR_UNSUPPORTED: plan outside the kernel's range, or NVRTC not available. */
int parrm_filter_specialise_check(const void* h_plan, int dtype,
                                  const parrm_filter_options_t* options, int32_t* shape,
                                  size_t* cubin_bytes);

/* Element-wise precision conversion for the float32 storage mode of the filter (the recording
 * crosses PCIe as float64, as the reference's API hands it over, parrm.py:866-875). */
int parrm_convert_f64_to_f32(const double* d_src, float* d_dst, int64_t n, void* stream);
int parrm_convert_f32_to_f64(const float* d_src, double* d_dst, int64_t n, void* stream);
/* General form: src_type in {PARRM_F64, PARRM_F32, PARRM_I16, PARRM_I32}, dst_type in
 * {PARRM_F64, PARRM_F32}.  The reference accepts any 2-D ndarray and widens it on the host
 * (parrm.py:861-866, 877-886); here float32 / int16 / int32 recordings cross PCIe in their
 * own width and are widened on the device. */
int parrm_convert(const void* d_src, int src_type, void* d_dst, int dst_type, int64_t n,
                  void* stream);
/* Transposing convert (csrc/transpose.cu), for time-major recordings -- [times, channels] with
 * the channels of each sample interleaved, as SpikeGLX / Open Ephys / Intan files and
 * acquisition APIs deliver them:
 *     d_dst[c * dst_ld + r] = (dst_type) d_src[r * src_ld + c],  r < rows, c < cols
 * in one pass through shared-memory tiles.  src_type in {PARRM_F64, PARRM_F32, PARRM_I16,
 * PARRM_I32}; dst_type is src_type itself, PARRM_F64 or PARRM_F32; each element is converted
 * with static_cast exactly as parrm_convert does.  Requires src_ld >= cols, dst_ld >= rows and
 * non-null pointers (else PARRM_ERR_INVALID_ARGUMENT, checked before anything is enqueued); the
 * source base needs no alignment beyond its element size.  rows or cols 0: nothing to do. */
int parrm_transpose(const void* d_src, int src_type, int64_t rows, int64_t cols, int64_t src_ld,
                    void* d_dst, int dst_type, int64_t dst_ld, void* stream);

/* ------------------------------------------------------------------------
 * Streaming filter: filter_data applied block by block as the recording is acquired (an
 * online caller runs find_period / create_filter on a calibration segment, then filters every
 * block the acquisition system delivers).  Concatenating every push's outputs and the closing
 * push's gives exactly parrm_filter_apply with a PARRM_PLAN_GATHER plan on the concatenated
 * recording, bit for bit: recording start and end edges and the non-finite rule included.
 *
 * Caller-owned state: d_ring of parrm_stream_ring_bytes() (the last span + max_chunk samples
 * of every channel in the compute type, span = max(w_max, 0) - min(w_min, 0)), the ascending
 * taps on the device (d_taps, n_taps, w_min = taps[0], w_max = taps[n_taps - 1]) and the
 * position `pos`, the number of samples pushed before this block.
 *
 * parrm_stream_push enqueues ONE kernel that widens the block [n_chans, n] (storage type
 * block_type, row stride ld_block, n <= max_chunk) into the ring and writes the outputs that
 * are now final to d_out [n_chans, ld_out] in out_type:
 *     open   (close = 0): outputs [max(0, pos - L), max(that, pos + n - L))
 *     closing (close = 1): outputs [max(0, pos - L), pos + n), the recording ending at pos + n
 * where L = max(0, -w_min) is the stream's latency: output t is final once sample t + L has
 * arrived.  Under the reference's convolution y[t] reads x[t - w], so a "future" filter (w > 0)
 * reads only earlier samples and has L = 0 -- it is the causal one -- while "past" and "both"
 * need filter_half_width samples of look-ahead.  Work per push is O(n_chans * (n + span)).
 * d_pos (may be NULL): device int64 the kernel reads the position from instead of `pos`, so
 * that a push captured in a CUDA graph (H2D of a header + block -> kernel -> D2H) replays with
 * a new position; the output count must then stay that of `pos` (it does for an open stream
 * once pos >= L).  Errors: block longer than max_chunk, negative position, bad types.
 * ---------------------------------------------------------------------- */
size_t parrm_stream_ring_bytes(int64_t n_chans, const int32_t* h_taps, int32_t n_taps,
                               int64_t max_chunk, int dtype);
int parrm_stream_push(void* d_ring, int64_t n_chans, int64_t max_chunk, const int32_t* d_taps,
                      int32_t n_taps, int32_t w_min, int32_t w_max, const void* d_block,
                      int block_type, int64_t ld_block, int64_t n, void* d_out, int out_type,
                      int64_t ld_out, int64_t pos, const int64_t* d_pos, int close, int dtype,
                      void* stream);

/* parrm_stream_push_at: the same kernel with the ring length and the first output passed
 * explicitly, for a stream whose taps were switched while it was open (a re-calibrated
 * filter).  d_ring holds the last ring_len samples of every channel ([n_chans, ring_len], any
 * ring_len the caller allocated); the push writes outputs [out_lo, out_hi) to d_out, with
 *     out_hi = close ? pos + n : max(out_lo, pos + n - L),   L = max(0, -w_min),
 * so after a switch to a smaller latency a push can emit more than n outputs, and after a
 * switch to a larger one none.  With one tap set, out_lo = max(0, pos - L) and
 * ring_len = span + max_chunk give exactly parrm_stream_push.  Requirements (else
 * PARRM_ERR_INVALID_ARGUMENT): 0 <= out_lo <= pos, n >= 0, and the ring invariant
 *     pos + n - max(0, out_lo - max(w_max, 0)) <= ring_len:
 * every sample the launch reads is still in the ring, and no slot it writes is read in it.
 * d_hdr (may be NULL): device int64 {pos, out_lo} read instead of the host values, so that a
 * captured CUDA graph replays with new positions; the output count must stay the one the host
 * arguments give.  Same arithmetic, bit for bit, as parrm_stream_push. */
int parrm_stream_push_at(void* d_ring, int64_t ring_len, int64_t n_chans, const int32_t* d_taps,
                         int32_t n_taps, int32_t w_min, int32_t w_max, const void* d_block,
                         int block_type, int64_t ld_block, int64_t n, void* d_out, int out_type,
                         int64_t ld_out, int64_t pos, int64_t out_lo, const int64_t* d_hdr,
                         int close, int dtype, void* stream);

/* parrm_stream_window: copy the last n samples of a stream's ring (ring_len slots per channel,
 * pos samples pushed) to d_dst: d_dst[c * ld_dst + i] = sample pos - n + i of channel c, in the
 * ring's compute type.  Requires 1 <= n <= min(pos, ring_len) and ld_dst >= n.  At most two
 * strided device-to-device copies on `stream` (the window wraps the ring at most once). */
int parrm_stream_window(const void* d_ring, int64_t ring_len, int64_t n_chans, int64_t pos,
                        int64_t n, void* d_dst, int64_t ld_dst, int dtype, void* stream);

/* ------------------------------------------------------------------------
 * Device-resident Nelder-Mead: the scipy.optimize.fmin refinements of find_period
 * (parrm.py:499-517, 545-550; SciPy 1.18 _minimize_neldermead, N = 1, defaults) as a state
 * machine on the device.  A round is
 *     parrm_eval_periods(d_points[5 * n_chains] -> d_values[5 * n_chains]);  parrm_nm_step(...)
 * with no host involvement, so rounds can be captured into a CUDA graph; *d_n_active (written
 * by every step) is the number of chains still running.  d_state holds n_chains records of
 * PARRM_NM_STATE_BYTES: { double sim[2], fsim[2], points[5]; int32 fcalls, iterations, done,
 * started } -- x = sim[0], fval = min(fsim), as fmin(..., full_output=True) reports them.
 * parrm_nm_init writes the initial simplex {x0, 1.05 x0} to d_points slots 0 and 1 of each
 * chain (slots 2-4 repeat x0); the first parrm_nm_step consumes those two values.
 * ---------------------------------------------------------------------- */
#define PARRM_NM_STATE_BYTES 88
int parrm_nm_init(const double* d_starts, int32_t n_chains, void* d_state, double* d_points,
                  void* stream);
int parrm_nm_step(void* d_state, int32_t n_chains, const double* d_values, double* d_points,
                  double xtol, double ftol, int32_t maxiter, int32_t maxfun, int32_t* d_n_active,
                  void* stream);

/* ------------------------------------------------------------------------
 * Parameter sweeps (the explorer's loop, _utils/_plotting.py:568-584; SURVEY 8(f).4): many
 * (period, period_half_width, filter_half_width, omit_n_samples, direction) sets at once.
 *   parrm_default_half_width  -- PARRM._get_filter_half_width (parrm.py:788-801) per set:
 *       d_limit[s] = (n_samples - 1) // 2; result int64 per set.
 *   parrm_build_taps_batch    -- parrm_build_taps per set, ONE launch; row s of d_taps
 *       (stride >= 2 * max half-width + 1) holds d_n_taps[s] ascending offsets.
 *   parrm_filter_apply_batch  -- filter the same [n_chans, n_samples] recording with every
 *       set in ONE launch, taking taps and counts straight from the device buffers above:
 *       d_out[s * set_stride + c * ld_out + t].  Direct gather; for the short recordings a
 *       sweep looks at (max_half_width bounded by shared memory: ~10^4 samples).
 * All parameter arrays are device arrays of n_sets entries.
 * ---------------------------------------------------------------------- */
int parrm_default_half_width(const double* d_period, const double* d_period_half_width,
                             const int64_t* d_omit_n_samples, const int64_t* d_limit,
                             int64_t n_sets, int64_t* d_half_width, void* stream);
int parrm_build_taps_batch(const double* d_period, const double* d_period_half_width,
                           const int64_t* d_filter_half_width, const int64_t* d_omit_n_samples,
                           const int32_t* d_direction, int64_t n_sets, int32_t* d_taps,
                           int64_t stride, int32_t* d_n_taps, void* stream);
int parrm_filter_apply_batch(const void* d_x, int64_t ld_x, int64_t n_samples, int64_t n_chans,
                             const int32_t* d_taps, int64_t tap_stride, const int32_t* d_n_taps,
                             int64_t n_sets, int64_t max_half_width, void* d_out, int64_t ld_out,
                             int64_t set_stride, int dtype, void* stream);

/* ------------------------------------------------------------------------
 * Periodogram: compute_psd (src/pyparrm/_utils/_power.py:10-68), the spectrum the parameter
 * explorer draws after every re-filter (_utils/_plotting.py:568-584, 637-642).
 *   X = fft(float32(x[c, :n_points]), n_points)   (cropped or zero-padded, as scipy.fft.fft)
 *   d_psd[c, k-1] = float32(|X_k|)^2 / (sampling_freq * n_points),  k = 1 .. n_points/2
 * float32 output [n_chans, ld_psd >= n_points/2]; the reference's `psd[:-1] *= 2` (which
 * doubles all ROWS but the last of a 2-D array) is left to the host wrapper.  Takes the
 * filtered recording where it already is -- on the device -- so the explorer's
 * filter -> spectrum loop never returns the full array to the host.
 * ---------------------------------------------------------------------- */
int parrm_periodogram(const void* d_x, int64_t n_chans, int64_t n_samples, int64_t ld, int dtype,
                      int64_t n_points, double sampling_freq, float* d_psd, int64_t ld_psd,
                      void* stream);

/* Measured FP64 FMA throughput helper for the roofline denominator of the evaluator
 * (bench.py): runs `iters` dependent-chain DFMA batches on every SM; reports flops issued. */
int parrm_fp64_fma_burn(int64_t iters, double* d_sink, double* h_flops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PARRM_B200_H */
