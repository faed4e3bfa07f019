/* vnd_b200.h — C ABI of the B200-native velvet-noise decorrelation hot path.
 *
 * This is the drop-in boundary.  The reference (ckonst/VNDecorrelate) has no FFI; its operator
 * API is Python duck typing (src/vndecorrelate/decorrelation.py:31-59).  Every entry point below
 * names the reference function whose arithmetic it reproduces; INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes.  No exceptions or aborts cross this boundary: every
 *     function returns 0 (VND_OK) or a negative VND_E* code; vnd_status_string() names it and
 *     vnd_last_error() returns a thread-local detail string.
 *   - "_dev" entry points take DEVICE pointers, an explicit cudaStream_t (passed as void*) and a
 *     caller-owned workspace: they never allocate, never synchronise, and are re-entrant on
 *     distinct streams.
 *   - "_host" entry points take HOST pointers and a vnd_ctx that owns a device arena, page-locked
 *     staging (used when the caller's buffers are pageable) and streams; host<->device copies happen
 *     inside the call.
 *   - Signals are addressed as  element(t, c) = base[t * stride_t + c * stride_c]  (strides in
 *     ELEMENTS), so C-order (frames, channels) arrays (stride_t = C, stride_c = 1) and planar
 *     (channels, frames) arrays (stride_t = 1, stride_c = frames) use the same calls.
 *   - Nothing here has a CPU fallback: without a CUDA device every compute call fails with
 *     VND_ECUDA.
 */
#ifndef VND_B200_H
#define VND_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VND_ABI_VERSION 1

enum {
  VND_OK = 0,
  VND_EINVAL = -1,       /* bad argument (null pointer, negative size, bad enum)        */
  VND_ECUDA = -2,        /* CUDA runtime error; see vnd_last_error()                    */
  VND_EUNSUPPORTED = -3, /* valid request this build cannot serve                       */
  VND_ENOMEM = -4,       /* workspace / arena too small or allocation failed            */
  VND_EPROGRAM = -5      /* malformed tap program                                       */
};

/* element types of signal buffers */
enum { VND_F32 = 0, VND_F64 = 1 };

/* Accumulation order of the sparse FIR.
 * VND_ORDER_SEGMENTED : VelvetNoise.convolve (decorrelation.py:393-415) — per segment, subtract
 *                       the negative taps, add the positive taps, multiply by the segment gain,
 *                       add into the output; every step rounded separately (no FMA).
 * VND_ORDER_ASCENDING : convolve_velvet_noise (decorrelation.py:630-660) — ascending tap index,
 *                       y = fl32(y + fl(x * coef)); the product and the sum are float32 when the
 *                       signal and the FIR are both float32, float64 otherwise (numpy promotion).
 * VND_ORDER_ASCENDING_F64 : same, with a float64 FIR (e.g. VelvetNoise.FIR): always float64 steps.
 */
enum { VND_ORDER_SEGMENTED = 0, VND_ORDER_ASCENDING = 1, VND_ORDER_ASCENDING_F64 = 2 };

/* ---------------------------------------------------------------------------------------------
 * Tap program: the per-channel tap table in the layout the kernels read.
 *
 * One int32 array `words` plus `offsets[C + 1]` (channel c owns words[offsets[c] .. offsets[c+1])).
 * An EMPTY range marks an unfiltered channel: the input is copied through
 * (decorrelation.py:399-400).
 *
 * SEGMENTED channel block:   [ S,  (n_neg, n_pos, gain_bits) x S,  tap indices ... ]
 *     tap indices are listed segment by segment, negative list then positive list, each in the
 *     reference's list order (decorrelation.py:247-254, :539-542).  gain_bits is the IEEE-754
 *     bit pattern of float32(segment_envelope[s]).  S may be 0 (filtered channel with no taps:
 *     output is zero).
 * ASCENDING channel block:   [ K,  (index, coef_lo, coef_hi) x K ]
 *     coefficient as a float64 bit pattern split in two words; indices ascending.
 * Taps with index >= frames must be removed by the caller (the reference drops them:
 * decorrelation.py:404-410); `halo` passed to the launchers is 1 + the largest remaining index.
 * -------------------------------------------------------------------------------------------*/
typedef struct vnd_tap_program {
  const int32_t* words;   /* device (for _dev calls) or host (for _host calls) */
  const int32_t* offsets; /* C + 1 entries, same memory space as `words`       */
  int64_t n_words;
  int32_t channels;
  int32_t order;          /* VND_ORDER_*                                       */
  int32_t apply_gain;     /* 0: envelope == (1.0,), the multiply is skipped (decorrelation.py:411) */
  int32_t halo;           /* 1 + max tap index over all channels (0 if no taps) */
  int32_t max_channel_words; /* longest channel block, in words (sizes the shared-memory copy) */
} vnd_tap_program;

/* A strided signal view. */
typedef struct vnd_signal {
  void* data;
  int64_t frames;
  int32_t channels;
  int32_t dtype;     /* VND_F32 or VND_F64 */
  int64_t stride_t;  /* elements */
  int64_t stride_c;  /* elements */
} vnd_signal;

/* Post-FIR stages of VelvetNoise.decorrelate (decorrelation.py:433-440) and the Haas stage of a
 * SignalChain (decorrelation.py:202-230, LR mode), fused into the FIR pass. */
typedef struct vnd_epilogue {
  int32_t ms_encode;      /* 1: encode_signal_to_side_channel (utils/dsp.py:40-63); needs 2 channels */
  int32_t use_width;      /* 1: apply_stereo_width (utils/dsp.py:21-37)                              */
  double width;
  int32_t rms_normalize;  /* 1: rms_normalize DUAL_MONO (utils/dsp.py:87-109), numpy axis-0 order    */
  int32_t haas_delay;     /* >= 0 frames; output has frames + haas_delay frames                      */
  int32_t haas_channel;   /* channel that is delayed                                                 */
} vnd_epilogue;

/* ------------------------------------------------------------------------------ housekeeping */
int vnd_abi_version(void);
const char* vnd_version(void);
const char* vnd_status_string(int status);
const char* vnd_last_error(void);
int vnd_device_count(int* count);

/* ------------------------------------------------------------------------------ device API */

/* Sparse velvet-noise FIR, y[t,c] = sum_k coef_k * x[t + i_k, c], terms past the end dropped.
 * Replaces VelvetNoise.convolve (decorrelation.py:393-415) or convolve_velvet_noise
 * (decorrelation.py:630-660) according to taps->order.  x: F32 or F64; y: F32, same frames,
 * taps->channels channels.  With F64 input every accumulation step is done in float64 and rounded
 * to float32, which is what numpy does for `f32_array -= f64_array`. */
int vnd_sparse_fir_dev(const vnd_signal* x, const vnd_signal* y, const vnd_tap_program* taps, void* stream);

/* Bytes of workspace vnd_vn_decorrelate_dev needs for the given shape/epilogue. */
int vnd_vn_decorrelate_workspace(int64_t frames, int32_t channels, const vnd_epilogue* ep, size_t* bytes);

/* Fused VelvetNoise.decorrelate (+ optional LR Haas delay): FIR -> M/S encode -> width ->
 * RMS gain -> Haas placement.  x: F32 (already cast, decorrelation.py:426); a mono signal is
 * passed with channels = 2 and stride_c = 0 (mono_to_stereo, decorrelation.py:428-429).
 * out: F32 or F64 with frames + ep->haas_delay frames.  Without rms_normalize this is ONE kernel:
 * one read and one write per sample. */
int vnd_vn_decorrelate_dev(const vnd_signal* x, const vnd_signal* out, const vnd_tap_program* taps,
                           const vnd_epilogue* ep, void* workspace, size_t workspace_bytes, void* stream);

/* Batched fused decorrelate: vnd_vn_decorrelate_dev on many stereo clips of any lengths in one call, with a fixed number
 * of launches per batch (1 without rms_normalize, 3 with it) whatever the number of clips.
 *   x               : packed float32 (rows, 2) C-order input (x_dtype must be VND_F32), 8-byte aligned; clip i is rows
 *                     [frame_offsets[i], frame_offsets[i + 1]) - a mono clip is packed with its samples in both columns;
 *   frame_offsets   : n_clips + 1 int64, starting at 0, non-decreasing, ending at rows;
 *   program_of_clip : n_clips int32; clip i runs channels 2 k and 2 k + 1 of `taps` (k = program_of_clip[i]), a SEGMENTED
 *                     program with two channels per distinct filter, each pair packed for that clip's length (taps at or
 *                     beyond the clip's length removed, as vnd_vn_decorrelate_dev expects);
 *   ep              : shared by all clips;
 *   out             : F32 or F64 (rows + n_clips * ep->haas_delay, 2) C-order, clip i from row
 *                     frame_offsets[i] + i * ep->haas_delay, each clip (frames_i + haas_delay) rows.
 * Every clip's output is byte-identical to vnd_vn_decorrelate_dev on that clip with its channel pair.  The _dev call
 * cannot read the device-side offsets: it checks everything else and returns VND_EUNSUPPORTED (before any launch)
 * when the filter's halo does not fit the batched kernel's shared memory, in which case the clips go through
 * vnd_vn_decorrelate_dev one by one (the _host call does that itself).  Workspace:
 * vnd_vn_decorrelate_batch_workspace(rows, n_clips, ep) bytes, 16-byte aligned (0 without rms_normalize). */
int vnd_vn_decorrelate_batch_workspace(int64_t rows, int32_t n_clips, const vnd_epilogue* ep, size_t* bytes);
int vnd_vn_decorrelate_batch_dev(const void* x, int32_t x_dtype, int64_t rows, const int64_t* frame_offsets, int32_t n_clips,
                                 const int32_t* program_of_clip, const vnd_tap_program* taps, const vnd_epilogue* ep, void* out,
                                 int32_t out_dtype, void* workspace, size_t workspace_bytes, void* stream);

/* numpy axis-0 order sum of squares per channel: strict left-to-right float32 running sum of
 * float32-rounded squares (what np.mean(np.square(a), axis=0) does on a C-order array,
 * utils/dsp.py:107-109).  sums: `channels` float32 values on the device. */
int vnd_colsumsq_seq_f32_dev(const vnd_signal* a, float* sums, void* stream);

/* HaasEffect.decorrelate (decorrelation.py:192-230): x F32 (channels = 2; mono passed with
 * stride_c = 0 and mono = 1), out F64 (frames + delay, 2).  mode_ms / width as in the reference. */
int vnd_haas_dev(const vnd_signal* x, const vnd_signal* out, int32_t delay, int32_t delayed_channel,
                 int32_t mode_ms, int32_t mono, int32_t use_width, double width, void* stream);

/* The Haas settings of one clip of vnd_haas_batch_dev: those of vnd_haas_dev.  32 bytes. */
typedef struct vnd_haas_clip {
  int32_t delay;           /* >= 0 frames                                                   */
  int32_t delayed_channel; /* 0 or 1                                                        */
  int32_t mode_ms, mono, use_width, reserved;
  double width;
} vnd_haas_clip;

/* Batched HaasEffect.decorrelate: vnd_haas_dev on many clips of any lengths, each with its own settings, in ONE launch
 * whatever the number of clips (none when out_rows == 0).
 *   x             : packed float32 (rows, 2) C-order input, 8-byte aligned; clip i is rows [frame_offsets[i],
 *                   frame_offsets[i + 1]) - a mono clip is packed with its samples in both columns and mono = 1;
 *   frame_offsets : n_clips + 1 int64, starting at 0, non-decreasing, ending at rows;
 *   clips         : n_clips settings records;
 *   out_offsets   : n_clips int64, out_offsets[i] = frame_offsets[i] + sum_{j < i} clips[j].delay;
 *   out           : float64 (out_rows, 2) C-order, 16-byte aligned, out_rows = rows + sum of the delays; clip i is rows
 *                   [out_offsets[i], out_offsets[i] + frames_i + delay_i).
 * Every clip's output is byte-identical to vnd_haas_dev on that clip with its settings.  The _dev call checks the
 * pointers and sizes it sees; it cannot read the device-side offsets and settings, which must be valid (the _host call
 * checks them). */
int vnd_haas_batch_dev(const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_clips, const vnd_haas_clip* clips,
                       const int64_t* out_offsets, int64_t out_rows, double* out, void* stream);

/* One step of many live signals that arrive block by block: ONE launch for all signals (none when rows == 0 and
 * out_rows == 0; history_out is then not written and history_in stays the current history).
 *   x              : packed float32 (rows, 2) C-order blocks, 8-byte aligned; signal i's block is rows [frame_offsets[i],
 *                    frame_offsets[i + 1]) - a mono block is packed with its samples in both columns;
 *   frame_offsets  : n_signals + 1 int64, starting at 0, non-decreasing, ending at rows;
 *   received       : n_signals int64, the frames signal i received before this step (T0; T1 = T0 + its block's rows);
 *   history_in/out : two float32 (n_signals, history_frames, 2) C-order buffers, 8-byte aligned.  Rows [i H, i H + H) of
 *                    history_in must hold signal i's frames [T0 - H, T0) as the previous step wrote them; the step writes
 *                    its frames [T1 - H, T1) to history_out (those before frame 0 as +0).  The caller swaps the two after
 *                    every step that launched.  A frame the kernel reads before T0 - H or before 0 is +0;
 *   out_offsets    : n_signals + 1 int64, starting at 0, non-decreasing, ending at out_rows: signal i writes out rows
 *                    [out_offsets[i], out_offsets[i + 1]).
 * A final step is the caller's matter: frames at or past T1 read as +0, as past the end of a one-shot signal of T1
 * frames, and the next step of a signal that starts over passes received = 0 (its old history is never read).
 * Neither _dev call can read the device-side tables, which must be valid; both check the pointers and sizes they see.
 *
 * vnd_vn_block_step_dev: VelvetNoise.decorrelate without normaliser.  taps, program_of_signal and ep are those of
 * vnd_vn_decorrelate_batch_dev with every program packed for an unbounded length (all taps kept); ep->rms_normalize
 * and ep->haas_delay must be 0.  emitted[i] = E0 is the number of frames signal i has emitted before; it writes its
 * output frames [E0, E0 + out_offsets[i + 1] - out_offsets[i]) to float32 (out_rows, 2) `out`.  history_frames must be at
 * least taps->halo - 1.  Bit contract: output frame t is byte-identical to frame t of vnd_vn_decorrelate_dev on the
 * signal's first T frames with its channel pair, for any T > t with t + taps->halo - 1 < T1 or T = T1: the frames it reads
 * are the same, and a tap past the end reads +0, which adds nothing, as the one-shot call drops it.  VND_EUNSUPPORTED,
 * checked before anything else after the program and the epilogue, when the filter's halo does not fit the kernel's
 * shared memory (the rule of vnd_vn_decorrelate_batch_dev): a call with n_signals = 0 asks it without a launch.
 *
 * vnd_haas_block_step_dev: HaasEffect.decorrelate with the settings record signals[i] (vnd_haas_batch_dev's; mono as
 * the block is packed), history_frames >= every delay.  Signal i writes its output frames [T0, T0 + out_offsets[i + 1] -
 * out_offsets[i]) to float64 (out_rows, 2) `out`, 16-byte aligned.  Bit contract: output frame m < T1 is byte-identical
 * to frame m of vnd_haas_dev on the signal's first T1 frames (it reads input frames m and m - delay only), and frames
 * [T1, T1 + delay) - a final step's tail - to those of vnd_haas_dev on exactly T1 frames. */
int vnd_vn_block_step_dev(const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_signals, const int64_t* received,
                          const int64_t* emitted, const int32_t* program_of_signal, const vnd_tap_program* taps, const vnd_epilogue* ep,
                          const float* history_in, float* history_out, int32_t history_frames, const int64_t* out_offsets,
                          int64_t out_rows, float* out, void* stream);
int vnd_haas_block_step_dev(const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_signals, const int64_t* received,
                            const vnd_haas_clip* signals, const float* history_in, float* history_out, int32_t history_frames,
                            const int64_t* out_offsets, int64_t out_rows, double* out, void* stream);

/* One VelvetNoise.convolve step of many live multichannel signals: ONE launch for all signals and channels (none when
 * rows == 0 and out_rows == 0).  The step model is vnd_vn_block_step_dev's, with `channels` = C values per row:
 *   x              : packed (rows, C) C-order blocks of `dtype` (VND_F32, or VND_F64 for the float64 arithmetic convolve uses
 *                    on float64 and 32-bit integer input), aligned to the value size;
 *   frame_offsets, received, emitted, out_offsets : as vnd_vn_block_step_dev (n_signals + 1, n, n, n + 1 int64);
 *   taps           : a SEGMENTED program with C channels per filter, filter k = channels [k C, (k + 1) C), each packed for an
 *                    unbounded length (all taps kept); program_of_signal[i] (int32) is signal i's filter;
 *   history_in/out : two (n_signals, history_frames, C) C-order buffers of `dtype`, history_frames >= taps->halo - 1, with
 *                    vnd_vn_block_step_dev's roles (the caller swaps them after every step that launched);
 *   out            : float32 (out_rows, C) C-order, 4-byte aligned; signal i writes its output frames [E0, E0 + out_offsets[i
 *                    + 1] - out_offsets[i]), E0 = emitted[i], to rows [out_offsets[i], out_offsets[i + 1]).
 * Bit contract: output frame t is byte-identical to frame t of vnd_sparse_fir_dev on the signal's first T frames (same
 * dtype), for any T > t with t + taps->halo - 1 < T1 or T = T1.  A tap the one-shot call drops reads +0 here, which in
 * SEGMENTED order cannot change the bits (vnd_fir.cu states why).  Filters of any halo are served: those whose halo does
 * not fit shared memory read their taps from global memory.  Checked before any launch: null or misaligned pointers, one
 * buffer passed as both histories, history_frames < taps->halo - 1, taps->channels not a multiple of channels, a dtype
 * other than VND_F32 / VND_F64, a non-SEGMENTED program, n_signals == 0 with rows. */
int vnd_fir_block_step_dev(const void* x, int32_t dtype, int64_t rows, int32_t channels, const int64_t* frame_offsets, int32_t n_signals,
                           const int64_t* received, const int64_t* emitted, const int32_t* program_of_signal, const vnd_tap_program* taps,
                           const void* history_in, void* history_out, int32_t history_frames, const int64_t* out_offsets, int64_t out_rows,
                           float* out, void* stream);

/* In-place stereo helpers on a (frames, 2) signal, F32 or F64 (utils/dsp.py:21-63, :124-167).
 * op: 0 LR_to_MS, 1 MS_to_LR, 2 apply_stereo_width(width), 3 encode_signal_to_side_channel(x, y)
 * (x = `dry`, y = `a`), 4 rms_normalize(dry, a) DUAL_MONO.  Op 4 sums each signal in the order numpy uses for its
 * layout: frame by frame for a C-order (frames, 2) signal, pairwise per column for a planar / Fortran-ordered one; workspace:
 * 64 bytes, plus 8 * (frames / 64 + 8) when a signal is planar. */
int vnd_stereo_op_dev(const vnd_signal* a, const vnd_signal* dry, int32_t op, double width,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Normalisers and polar form beyond what VelvetNoise itself uses (utils/dsp.py:71-109, :374-422).  Signals are
 * contiguous 1-D (ndim = 1) or C-order (frames, channels) arrays (ndim = 2), F32 or F64.
 *   rms_normalize: STEREO mode and 1-D signals (both statistics with axis=None: numpy's pairwise summation order is
 *       reproduced bit for bit); 2-D DUAL_MONO keeps using vnd_stereo_op op 4 (numpy's axis-0 order).
 *   peak_normalize: every mode.
 *   polar_coordinates: radii, folded (or full) angles and amplitude weights of a stereo pair; weights may be NULL.
 *       Radii and weights are bit-exact, angles within 2 ulp of numpy's arctan2.
 * Workspace: vnd_dsp_workspace(largest element count) bytes. */
int vnd_dsp_workspace(int64_t elems, size_t* bytes);
int vnd_rms_normalize_dev(const vnd_signal* x, int32_t x_ndim, const vnd_signal* y, int32_t y_ndim, int32_t stereo_mode, double epsilon,
                          void* workspace, size_t workspace_bytes, void* stream);
int vnd_peak_normalize_dev(const vnd_signal* y, int32_t ndim, int32_t stereo_mode, double epsilon, void* workspace, size_t workspace_bytes,
                           void* stream);
int vnd_polar_dev(const void* left, const void* right, int64_t n, int32_t dtype, int32_t mode_ms, int32_t semicircular, int32_t normalize,
                  void* radii, void* thetas, void* weights, void* workspace, size_t workspace_bytes, void* stream);

/* Batched stereo-image objective for velvet-noise candidates (optimization.py:46-105 evaluated as
 * optimization.py:108-117 does, for the candidates optimization.py:260-272 builds: channel 0
 * filtered, channel 1 passed through, LR, no normaliser).
 *   clips       : n_clips planar stereo clips, element(clip, c, t) = clips[clip*clip_stride + c*chan_stride + t]
 *   cand        : SEGMENTED tap program with one "channel" per candidate (channels = n_cand)
 *   partials    : n_clips * n_cand * 12 float64 on the device:
 *                 [sum r, sum r*th, sum r*th^2, sum r*th^3, sum L*R, sum L*L,
 *                  |d|, |s| of the frame with the largest |d|/|s| among frames with s >= 0,
 *                  |d|, |s| of the same among frames with s < 0,  frames, 0]
 *                 with d = L - R, s = L + R, th = atan(d / s) (the folded angle, |err| <= 1e-7);
 *                 max|theta| is evaluated by the host from the two tracked frames (rounding is
 *                 monotone, so they are where the reference's float32 maximum is attained).
 * The host combines the partials with the reference's dtype chain (SURVEY.md A.5). */
int vnd_objective_workspace(int64_t frames, int32_t n_clips, int32_t n_cand, size_t* bytes);
int vnd_vn_objective_batch_dev(const float* clips, int64_t frames, int32_t n_clips, int64_t clip_stride,
                               int64_t chan_stride, const vnd_tap_program* cand, double* partials,
                               void* workspace, size_t workspace_bytes, void* stream);

/* Haas candidates (optimization.py:183-203): LR mode, channel 0 delayed by delays[k] frames,
 * float64 arithmetic, frames + delays[k] output frames.  clips may be F32 or F64 (clip_dtype);
 * with delays = {0} this is the objective of an arbitrary stereo signal.  8 float64 per pair:
 *   [sum r, sum r*th, sum r*th^2, sum r*th^3, max|th|, sum L*R, sum L*L, frames] */
int vnd_haas_objective_batch_dev(const void* clips, int32_t clip_dtype, int64_t frames, int32_t n_clips, int64_t clip_stride,
                                 int64_t chan_stride, const int32_t* delays, int32_t n_cand, double* partials,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* The Haas objective above over a flat list of (clip, delay) pairs on ragged clips: one launch, one CTA per pair,
 * whatever the number of clips and their lengths.
 *   x             : float32, the clips packed channel-planar: element (t, c) of clip i is
 *                   x[c * chan_stride + frame_offsets[i] + t], c = 0, 1 (chan_stride >= rows);
 *   frame_offsets : n_clips + 1 int64, starting at 0, non-decreasing, ending at rows (as for vnd_vn_decorrelate_batch_dev);
 *   pair_clip, pair_delay : n_pairs int32 each; pair p is clip pair_clip[p] with channel 0 delayed by pair_delay[p] >= 0
 *                   frames (LR, frames_i + pair_delay[p] output frames).  Any order; listing a clip's delays together keeps
 *                   the clips that CTAs running at the same time read in L2;
 *   partials      : n_pairs * 8 float64, the slots of vnd_haas_objective_batch_dev:
 *                   [sum r, sum r*th, sum r*th^2, sum r*th^3, max|th|, sum L*R, sum L*L, frames].
 * The 8 partials of pair p equal, bit for bit, those vnd_haas_objective_batch_dev returns for clip pair_clip[p] alone
 * (float32, planar) with delays = {pair_delay[p]}: both launch the same kernel body (same per-thread striding from frame
 * 0 of the clip, same accumulation, same warp and block reductions).  The _dev call checks the sizes, the stride and
 * the pointers; it cannot read the device-side offsets and indices, which must be valid (the _host call checks them).
 * n_pairs == 0 launches nothing. */
int vnd_haas_objective_pairs_dev(const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets, int32_t n_clips,
                                 const int32_t* pair_clip, const int32_t* pair_delay, int32_t n_pairs, double* partials, void* stream);

/* The velvet-noise objective above over a list of RUNS on ragged clips: one objective launch and one combine launch,
 * whatever the number of clips, runs and their lengths.
 *   x             : float32, the clips packed channel-planar: element (t, c) of clip i is
 *                   x[c * chan_stride + frame_offsets[i] + t], c = 0, 1 (chan_stride >= rows);
 *   frame_offsets : n_clips + 1 int64, starting at 0, non-decreasing, ending at rows;
 *   cand          : SEGMENTED tap program (device words and offsets), one channel per candidate;
 *   run r         : clip run_clip[r] scored on the run_count[r] >= 0 consecutive channels of `cand` that start at
 *                   run_cand[r]; candidate j's 12 partials go to row run_out[r] + j of `partials` (n_partial_rows x 12
 *                   float64 on the device, the slots of vnd_vn_objective_batch_dev).  Rows no run names are not written.
 *                   The channels a run uses must be packed for its clip's length (taps at or beyond it removed).
 * Unlike the other _dev calls, frame_offsets and the four run arrays (n_runs int32 each) are HOST arrays: the launch
 * geometry depends on every clip's length and every run's size.  The call checks them (offsets as above, chan_stride
 * >= rows, every run's clip in range and not empty - VND_EINVAL "objective of an empty signal" -, its channels inside
 * the program and its rows inside n_partial_rows) before it touches the device, plans the launch, and writes the
 * derived work-item table into the front of the workspace with one cudaMemcpyAsync on `stream` (the host table may be
 * freed on return).  Workspace: vnd_vn_objective_runs_workspace bytes for the same offsets and runs, 256-byte aligned.
 * A filter whose halo (clamped to the longest clip of the runs) does not fit in shared memory returns VND_EUNSUPPORTED
 * before any launch.  n_runs == 0 launches nothing.
 * Bit contract: the 12 partials of (run r, candidate j) equal, bit for bit, row j of what vnd_vn_objective_batch_dev
 * returns for clip run_clip[r] alone (planar) with the one channel run_cand[r] + j as its program: tiles are counted
 * from frame 0 of each clip, staging reads nothing past the clip's last frame, and the chunk partials are added in tile
 * order. */
int vnd_vn_objective_runs_workspace(const int64_t* frame_offsets, int32_t n_clips, const int32_t* run_clip, const int32_t* run_count,
                                    int32_t n_runs, size_t* bytes);
int vnd_vn_objective_runs_dev(const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets, int32_t n_clips,
                              const vnd_tap_program* cand, const int32_t* run_clip, const int32_t* run_cand, const int32_t* run_count,
                              const int32_t* run_out, int32_t n_runs, double* partials, int64_t n_partial_rows, void* workspace,
                              size_t workspace_bytes, void* stream);

/* Settings of one candidate of vnd_vn_stereo_objective_dev: the epilogue of vnd_vn_decorrelate_dev without normaliser
 * or Haas stage.  16 bytes. */
typedef struct vnd_vn_stereo_cand {
  int32_t ms_encode;  /* 1: M/S side-channel encode (mode 'MS')                                      */
  int32_t use_width;  /* 1: apply the stereo width                                                   */
  float w_mid;        /* float32(1 - width), the rounding vnd_vn_decorrelate_dev applies to ep->width */
  float w_side;       /* float32(width)                                                              */
} vnd_vn_stereo_cand;

/* The objective of many VelvetNoise candidates with two outputs and no normaliser - any filtered channels, LR or MS,
 * any width - on one clip, in one objective launch and one combine launch.
 *   x        : float32 channel-planar clip, element (t, c) = x[c * chan_stride + t], c = 0, 1 (chan_stride >= frames >= 1);
 *   taps     : SEGMENTED program (device words and offsets) with 2 n_cand channels: candidate j's filter is channels
 *              2 j (left) and 2 j + 1 (right), each packed for `frames` (vnd_vn_decorrelate_dev's program for that
 *              candidate; an unfiltered channel has no words and is copied through).  One apply_gain for all;
 *   cands    : n_cand settings records (device);
 *   partials : n_cand * 12 float64 on the device, the slots of vnd_vn_objective_batch_dev.
 * Bit contract: candidate j's 12 partials equal, bit for bit, those of vnd_vn_objective_batch_dev on the float32 output
 * of vnd_vn_decorrelate_dev for that candidate (planar, with the one-tap identity program).  The
 * output is never stored: the kernel builds it in registers with the same tap loop and epilogue and feeds the moments
 * with the same frame-to-lane mapping, tiles and chunks.  Checked before any launch: the program (SEGMENTED, 2 n_cand
 * channels), the sizes and the pointers.  VND_EUNSUPPORTED (no launch) when the program's halo does not fit shared
 * memory: the caller then scores candidate by candidate.
 * Workspace: vnd_vn_stereo_objective_workspace bytes, 256-byte aligned. */
int vnd_vn_stereo_objective_workspace(int64_t frames, int32_t n_cand, size_t* bytes);
int vnd_vn_stereo_objective_dev(const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps, const vnd_vn_stereo_cand* cands,
                                int32_t n_cand, double* partials, void* workspace, size_t workspace_bytes, void* stream);

/* The objective of many VelvetNoise candidates with two outputs and the default normaliser rms_normalize (DUAL_MONO) -
 * any filtered channels, LR or MS, any width - on one clip, in three launches on `stream` for any number of candidates:
 * vn_rms_sums_kernel (the sums of squares of x and of every candidate's un-normalised output, then its gains),
 * vn_stereo_objective_kernel on the scaled outputs, and the combine.  No host synchronisation between them.
 *   x, taps, cands, partials: as vnd_vn_stereo_objective_dev (the candidates' records hold no normaliser flag: the
 *              normaliser is what this call adds);
 *   gains    : 2 n_cand float32 on the device, written: candidate j's channel-0 and channel-1 gains at 2 j, 2 j + 1.
 * Bit contract: gains[2 j + c] is the gain vnd_vn_decorrelate_dev with rms_normalize = 1 applies to channel c of
 * candidate j's output when its input is C-order (frames, 2) or mono (x's sums of squares are strict left-to-right
 * float32 running sums, numpy's order for such an input), and candidate j's 12 partials equal, bit for bit, those of
 * vnd_vn_objective_batch_dev on that scaled output (planar, with the one-tap identity program).  Checked before any
 * launch: the program (SEGMENTED, 2 n_cand channels), the sizes and the pointers, gains included.  VND_EUNSUPPORTED (no
 * launch) when the program's halo does not fit either kernel's shared memory.
 * Workspace: vnd_vn_stereo_rms_objective_workspace bytes, 256-byte aligned. */
int vnd_vn_stereo_rms_objective_workspace(int64_t frames, int32_t n_cand, size_t* bytes);
int vnd_vn_stereo_rms_objective_dev(const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps,
                                    const vnd_vn_stereo_cand* cands, int32_t n_cand, float* gains, double* partials, void* workspace,
                                    size_t workspace_bytes, void* stream);

/* The objective of many HaasEffect candidates - any delayed channel, LR or MS, any width - on one clip: one launch, one
 * CTA per candidate.
 *   x        : float32 channel-planar clip as above (a mono clip with its samples in both channels and mono = 1 in every
 *              record);
 *   cands    : n_cand vnd_haas_clip records (device, 16-byte aligned): delay >= 0, delayed_channel 0 or 1;
 *   partials : n_cand * 8 float64 on the device, the slots of vnd_haas_objective_batch_dev.
 * Bit contract: candidate j's 8 partials equal, bit for bit, those of vnd_haas_objective_batch_dev with delays = {0} on
 * the float64 output of vnd_haas_dev for that candidate: every output frame comes from the same per-frame function and
 * enters the sums in the same thread and order.  The _dev call checks the sizes and pointers; it cannot read the
 * device-side records, which must be valid (the _host call checks them). */
int vnd_haas_effect_objective_dev(const float* x, int64_t frames, int64_t chan_stride, const vnd_haas_clip* cands, int32_t n_cand,
                                  double* partials, void* stream);

/* ------------------------------------------------------------------------------ host API */
typedef struct vnd_ctx vnd_ctx;

int vnd_ctx_create(int device, vnd_ctx** ctx);
int vnd_ctx_destroy(vnd_ctx* ctx);
/* Page-locked host memory for callers that want zero-staging transfers: buffers from these calls (or registered
 * with cudaHostRegister) are copied by DMA directly; any other host buffer is staged through the context's own
 * page-locked ring.  vnd_host_alloc allocates on the calling thread's current device, vnd_ctx_host_alloc on the
 * context's device (it never touches another GPU). */
int vnd_host_alloc(size_t bytes, void** ptr);
int vnd_ctx_host_alloc(vnd_ctx* ctx, size_t bytes, void** ptr);
int vnd_host_free(void* ptr);

/* Host-buffer versions of the calls above (all pointers, including taps->words/offsets, are HOST
 * pointers).  Each call takes the context's lock, runs the argument checks of its _dev twin and then those that read
 * its host tables (offsets, indices, records), all before any copy, then uploads the inputs, runs the _dev call on
 * them and downloads; on return the result is in `y`/`out`.
 * vnd_sparse_fir_host overlaps the three for float32 slabs of 8 MB and more: planar (channels, frames) slabs are
 * cut into channel groups, C-order (frames, channels) slabs - the reference's layout - into runs of frames
 * uploaded with the filter's halo (wide ones are transposed to planar on the device around the kernel), and
 * consecutive chunks flow through a three-deep device ring on three streams. */
int vnd_sparse_fir_host(vnd_ctx* ctx, const vnd_signal* x, const vnd_signal* y, const vnd_tap_program* taps);
int vnd_vn_decorrelate_host(vnd_ctx* ctx, const vnd_signal* x, const vnd_signal* out,
                            const vnd_tap_program* taps, const vnd_epilogue* ep);
/* vnd_vn_decorrelate_batch_dev with host buffers (offsets, program indices and tap program on the host too).  Inputs
 * of 8 MB and more flow through the overlapped pipeline in chunks of whole clips (about VND_PIPE_CHUNK_MB each);
 * filters whose halo does not fit the batched kernel run clip by clip through vnd_vn_decorrelate_host. */
int vnd_vn_decorrelate_batch_host(vnd_ctx* ctx, const void* x, int32_t x_dtype, int64_t rows, const int64_t* frame_offsets,
                                  int32_t n_clips, const int32_t* program_of_clip, const vnd_tap_program* taps, const vnd_epilogue* ep,
                                  void* out, int32_t out_dtype);
int vnd_haas_host(vnd_ctx* ctx, const vnd_signal* x, const vnd_signal* out, int32_t delay,
                  int32_t delayed_channel, int32_t mode_ms, int32_t mono, int32_t use_width, double width);
/* vnd_haas_batch_dev with host buffers (x, offsets, settings and out on the host).  Derives the out offsets itself (out
 * holds rows + sum of the delays rows).  Inputs of 8 MB and more flow through the overlapped pipeline in chunks of whole
 * clips (about VND_PIPE_CHUNK_MB each). */
int vnd_haas_batch_host(vnd_ctx* ctx, const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_clips,
                        const vnd_haas_clip* clips, double* out);
int vnd_stereo_op_host(vnd_ctx* ctx, const vnd_signal* a, const vnd_signal* dry, int32_t op, double width);
int vnd_rms_normalize_host(vnd_ctx* ctx, const vnd_signal* x, int32_t x_ndim, const vnd_signal* y, int32_t y_ndim, int32_t stereo_mode,
                           double epsilon);
int vnd_peak_normalize_host(vnd_ctx* ctx, const vnd_signal* y, int32_t ndim, int32_t stereo_mode, double epsilon);
int vnd_polar_host(vnd_ctx* ctx, const void* left, const void* right, int64_t n, int32_t dtype, int32_t mode_ms, int32_t semicircular,
                   int32_t normalize, void* radii, void* thetas, void* weights);
int vnd_vn_objective_batch_host(vnd_ctx* ctx, const float* clips, int64_t frames, int32_t n_clips,
                                int64_t clip_stride, int64_t chan_stride, const vnd_tap_program* cand,
                                double* partials);
int vnd_haas_objective_batch_host(vnd_ctx* ctx, const void* clips, int32_t clip_dtype, int64_t frames, int32_t n_clips,
                                  int64_t clip_stride, int64_t chan_stride, const int32_t* delays,
                                  int32_t n_cand, double* partials);
/* vnd_haas_objective_pairs_dev with host buffers.  No pair may put delay 0 on an empty clip (an empty signal has no
 * objective: optimization.py:41-43). */
int vnd_haas_objective_pairs_host(vnd_ctx* ctx, const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets,
                                  int32_t n_clips, const int32_t* pair_clip, const int32_t* pair_delay, int32_t n_pairs, double* partials);

/* vnd_vn_stereo_objective_dev and vnd_haas_effect_objective_dev with host buffers (x, program, records and partials). */
int vnd_vn_stereo_objective_host(vnd_ctx* ctx, const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps,
                                 const vnd_vn_stereo_cand* cands, int32_t n_cand, double* partials);
int vnd_haas_effect_objective_host(vnd_ctx* ctx, const float* x, int64_t frames, int64_t chan_stride, const vnd_haas_clip* cands, int32_t n_cand,
                                   double* partials);

/* vnd_vn_stereo_rms_objective_dev with host buffers (x, program, records, gains and partials): the same checks, then
 * staging, the device call and the download of partials and gains. */
int vnd_vn_stereo_rms_objective_host(vnd_ctx* ctx, const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps,
                                     const vnd_vn_stereo_cand* cands, int32_t n_cand, float* gains, double* partials);

/* vnd_vn_objective_runs_dev with host buffers (x, program, tables and partials).  Rows no run names come back as
 * zeros. */
int vnd_vn_objective_runs_host(vnd_ctx* ctx, const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets, int32_t n_clips,
                               const vnd_tap_program* cand, const int32_t* run_clip, const int32_t* run_cand, const int32_t* run_count,
                               const int32_t* run_out, int32_t n_runs, double* partials, int64_t n_partial_rows);

/* The overlapped path of vnd_sparse_fir_host with an explicit stage size: x and y are HOST planar
 * (channels, frames) float32 slabs; channels are cut into groups of `channels_per_chunk`, and
 * upload / kernel / download of consecutive groups overlap on three streams.  Page-locked buffers
 * (vnd_host_alloc) are copied directly; pageable ones go through the context's page-locked staging ring,
 * filled and drained by two helper threads. */
int vnd_sparse_fir_stream_host(vnd_ctx* ctx, const float* x, float* y, int64_t frames, int32_t channels,
                               const vnd_tap_program* taps, int32_t channels_per_chunk);

/* Number of kernels this library has launched in the calling process (all threads); bench.py
 * reports the difference across its timed region as `gpu_launches`. */
int64_t vnd_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* VND_B200_H */
